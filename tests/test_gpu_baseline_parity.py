"""BaselineDecoder (models/baseline.py) against the fp64 oracle (oracle.decoders.baseline_decoder_forward / baseline_loss),
step by step and row by row, on both recurrence paths of the bf16 tier: the persistent kernel (K8) and the per-step
launch chain that shapes outside the persistent kernel's rules take (B > 512, H % 16 == 8, H / 4 > 148).

Per-step rule (stated before measuring; the tier bounds of the suite applied to each step instead of the whole tensor):
  * logits: for every step t, |out[:, t] - ref[:, t]| / |ref[:, t]| (norm over rows and vocabulary) <= LOGIT[tier];
    every row b: |out[b] - ref[b]| / |ref[b]| <= LOGIT[tier], and no row more than ROW_K times the median row;
  * loss: relative error <= LOGIT[tier];
  * gradients: every parameter gradient norm-wise, d img_features row by row, d embedding norm-wise <= GRAD[tier];
  * greedy ids: argmax(out[b, t]) may differ from the fp64 argmax only where the fp64 top-2 margin is below
    2 LOGIT[tier] max_v |ref[b, t, v]| (the largest error a logit of that row can carry under the rule above).
fp32-class tiers (fp32, fp32x3): LOGIT 1e-4, GRAD 1e-3.  bf16: LOGIT 5e-3, GRAD 2e-2.
The oracle runs on the CPU in row chunks (rows are independent; only the parameters are shared).
"""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

import helpers as H

LOGIT = {"fp32": 1e-4, "fp32x3": 1e-4, "bf16": 5e-3}
GRAD = {"fp32": 1e-3, "fp32x3": 1e-3, "bf16": 2e-2}
ROW_K = 50
_TESTS = os.path.dirname(os.path.abspath(__file__))

# name -> dims; "max": the largest hidden size the persistent predicate admits at this B (read from the device)
CASES = {
    "cfg1": dict(B=128, L=25, V=9490, E=512, H=512, glove=False),           # configs[1] at full size, ragged + pads
    "chain_b640": dict(B=640, L=25, V=9490, E=512, H=512, glove=False),     # B > 512: 5 row tiles
    "chain_h40": dict(B=96, L=25, V=1200, E=64, H=40, glove=False),         # H % 16 == 8
    "chain_h608": dict(B=64, L=12, V=1200, E=128, H=608, glove=False),      # H / 4 = 152 > 148
    "max_h": dict(B=128, L=25, V=2000, E=256, H="max", glove=False),
    "glove": dict(B=96, L=20, V=2000, E=300, H=256, glove=True),            # fp64 fine-tuned table, E % 8 != 0
    "l1": dict(B=64, L=1, V=500, E=64, H=64, glove=False),                  # no embedding rows: d embedding == 0
    "l200": dict(B=32, L=200, V=300, E=32, H=48, glove=False),              # long recurrence
}
RUNS = [("cfg1", "fp32"), ("cfg1", "fp32x3"), ("cfg1", "bf16"), ("chain_b640", "bf16"), ("chain_h40", "bf16"),
        ("chain_h608", "bf16"), ("max_h", "bf16"), ("glove", "fp32"), ("glove", "fp32x3"), ("glove", "bf16"),
        ("l1", "fp32"), ("l1", "bf16"), ("l200", "fp32"), ("l200", "bf16")]
PERSISTENT = {"cfg1": True, "chain_b640": False, "chain_h40": False, "chain_h608": False, "max_h": True, "glove": True,
              "l1": True, "l200": True}


def _dims(name):
    c = dict(CASES[name])
    if c["H"] == "max":
        from icd_b200._lib import lib
        c["H"] = max(h for h in range(16, 4 * 148 + 1, 16) if lib().icd_lstm_seq_supported(c["B"], c["L"], h))
    return c


def _module_and_inputs(c):
    import icd_b200.models.baseline as my_base
    from icd_b200 import synthetic
    p = my_base.BaselineDecoderParams()
    p.hidden_size, p.embed_size, p.vocab_size = c["H"], c["E"], c["V"]
    torch.manual_seed(c["B"] + c["H"] + c["L"])
    dec = my_base.BaselineDecoder(p)
    if c["glove"]:
        dec.load_pretrained_embeddins(synthetic.glove_like_table(c["V"], c["E"]))
        dec.fine_tune_embeddings(True)
    g = torch.Generator().manual_seed(c["V"] + c["B"])
    img = torch.randn(c["B"], c["E"], generator=g)
    caps, _ = synthetic.captions(c["B"], c["V"], max_len=c["L"], seed=c["B"] * 7 + c["L"],
                                 lengths=("ragged" if c["L"] > 2 else None))
    return dec, img, caps


def _run(dec, img, caps, precision, cuda):
    """-> dict(out, loss, grads{name}, d_img, launches) of one forward + loss + backward on the device."""
    from icd_b200 import ops
    from icd_b200.losses import baseline_caption_loss
    dec = dec.to(cuda)
    dec.precision = precision
    for p_ in dec.parameters():
        p_.grad = None
    img_d = img.to(cuda).requires_grad_(True)
    caps_d = caps.to(cuda)
    torch.cuda.synchronize()
    n0 = ops.launch_count()
    out = dec(img_d, caps_d)
    loss = baseline_caption_loss(out, caps_d)
    loss.backward()
    torch.cuda.synchronize()
    return dict(out=out.detach(), loss=float(loss.detach()), launches=ops.launch_count() - n0, d_img=img_d.grad.detach(),
                grads={k: v.grad.detach().clone() for k, v in dec.named_parameters() if v.grad is not None})


def _oracle(dec, img, caps, chunk=64):
    """fp64 loss, parameter gradients, d img_features and logits (kept on the CPU in fp32 to compare with), in row chunks."""
    from oracle import decoders as O
    w64 = {k: v.detach().cpu().double().requires_grad_(True) for k, v in dec.state_dict().items()}
    n_tok = int((caps != 0).sum())
    B, L = caps.shape
    loss, d_img, outs = 0.0, torch.empty(B, img.shape[1], dtype=torch.float64), []
    for r0 in range(0, B, chunk):
        r1 = min(B, r0 + chunk)
        i64 = img[r0:r1].double().requires_grad_(True)
        o = O.baseline_decoder_forward(w64, i64, caps[r0:r1])
        l = F.cross_entropy(o.reshape(-1, o.shape[2]), caps[r0:r1].reshape(-1), ignore_index=0, reduction="sum") / n_tok
        l.backward()
        loss += float(l.detach())
        d_img[r0:r1] = i64.grad
        outs.append(o.detach())
    ref = torch.cat(outs, 0)
    # the chunked sum equals the oracle's own mean loss
    if B <= 2 * chunk:
        assert abs(float(O.baseline_loss(ref, caps)) - loss) <= 1e-12 * max(1.0, abs(loss))
    return dict(out=ref, loss=loss, d_img=d_img, grads={k: v.grad for k, v in w64.items() if v.grad is not None})


_ORACLE_CACHE = {}


def _oracle_cached(name, dec, img, caps):
    if name not in _ORACLE_CACHE:
        _ORACLE_CACHE[name] = _oracle(dec, img, caps)
    return _ORACLE_CACHE[name]


def _compare(got, ref, tier, caps):
    """-> (failure messages, measured errors) under the per-step rule of the module docstring."""
    lg, gr = LOGIT[tier], GRAD[tier]
    out = got["out"].cpu().double()
    r = ref["out"]
    fails, m = [], {}
    d2 = (out - r) ** 2
    step = H.step_rel_err(torch.stack([d2.sum(dim=(0, 2)), (r ** 2).sum(dim=(0, 2))], 1))
    row = H.row_rel_err(torch.stack([d2.sum(dim=(1, 2)), (r ** 2).sum(dim=(1, 2))], 1))
    m["logits_step_max"], m["logits_row_max"] = float(step.max()), float(row.max())
    if float(step.max()) > lg:
        fails.append("logits: steps %s over %.0e (worst %.2e)" % ((step > lg).nonzero().flatten().tolist()[:16], lg,
                                                                   float(step.max())))
    fails += ["logits " + s for s in H.row_spread_failures(row, lg, ROW_K)]
    m["loss"] = abs(got["loss"] - ref["loss"]) / abs(ref["loss"])
    if m["loss"] > lg:
        fails.append("loss %.8g vs %.8g" % (got["loss"], ref["loss"]))
    grad_err = {}
    for k, g64 in ref["grads"].items():
        e = H.rel_err(got["grads"][k], g64) if float(g64.norm()) > 0 else float(got["grads"][k].abs().max())
        grad_err[k] = e
        if e > gr:
            fails.append("d %s: %.2e > %.0e" % (k, e, gr))
    m["grad_max"] = max(grad_err.values())
    di = got["d_img"].cpu().double()
    di_rows = H.row_rel_err(torch.stack([((di - ref["d_img"]) ** 2).sum(1), (ref["d_img"] ** 2).sum(1)], 1))
    m["d_img_row_max"] = float(di_rows.max())
    if float(di_rows.max()) > gr:
        fails.append("d img_features: rows %s over %.0e" % ((di_rows > gr).nonzero().flatten().tolist()[:16], gr))
    top2 = r.topk(2, dim=2)
    margin = top2.values[..., 0] - top2.values[..., 1]
    flips = out.argmax(dim=2) != top2.indices[..., 0]
    allowed = margin < 2 * lg * r.abs().amax(dim=2)
    m["greedy_flips"] = int(flips.sum())
    if bool((flips & ~allowed).any()):
        bt = (flips & ~allowed).nonzero().tolist()
        fails.append("greedy ids flip at (row, step) %s with fp64 margins above the bound" % bt[:8])
    return fails, m


@pytest.mark.gpu
@pytest.mark.parametrize("name,tier", RUNS)
def test_baseline_decoder_matches_fp64_per_step(cuda, name, tier):
    """One forward + loss + backward of BaselineDecoder against the fp64 oracle under the per-step rule of the module
    docstring.  Each case asserts which recurrence path it took (the persistent predicate and the number of launches:
    the chain launches at least 4 kernels per step, the persistent path one per direction)."""
    from icd_b200 import ops
    c = _dims(name)
    dec, img, caps = _module_and_inputs(c)
    persistent = ops.lstm_seq_supported(c["B"], c["L"], c["H"])
    assert persistent == PERSISTENT[name], "%s: persistent predicate says %s" % (name, persistent)
    got = _run(dec, img, caps, tier, cuda)
    if tier == "bf16" and c["L"] >= 12:
        assert (got["launches"] < 4 * c["L"]) == persistent, "%s: %d launches" % (name, got["launches"])
    ref = _oracle_cached(name, dec, img, caps)
    fails, m = _compare(got, ref, tier, caps)
    if c["L"] == 1:
        assert torch.all(got["grads"]["embedding.weight"] == 0), "L = 1 reads no embedding row"
    if c["glove"]:
        assert got["grads"]["embedding.weight"].dtype == torch.float64
    print("%s %s H=%d persistent=%s launches=%d %s" % (name, tier, c["H"], persistent, got["launches"],
                                                       " ".join("%s=%.3g" % kv for kv in m.items())))
    assert not fails, "%s %s:\n%s" % (name, tier, "\n".join(fails))


def child_main(out_path):
    """Entry point of the children of test_chain_and_persistent_paths: configs[1] bf16 twice, outputs and gradients saved."""
    cuda = torch.device("cuda:0")
    dec, img, caps = _module_and_inputs(_dims("cfg1"))
    runs = [_run(dec, img, caps, "bf16", cuda) for _ in range(2)]
    from icd_b200 import ops
    torch.save(dict(runs=[{k: (v if k != "out" else v.cpu()) for k, v in r.items()} for r in runs],
                    persistent=ops.lstm_seq_supported(128, 25, 512)), out_path)


def _child(tmp_path, tag, **env_over):
    out_path = str(tmp_path / (tag + ".pt"))
    env = dict(os.environ, **env_over)
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_baseline_parity as m; m.child_main(%r)"
            % (H.ROOT, _TESTS, out_path))
    flags = ["-s"] if sys.flags.no_user_site else []
    proc = subprocess.run([sys.executable] + flags + ["-c", code], env=env, cwd=H.ROOT, capture_output=True, text=True,
                          timeout=1200)
    assert proc.returncode == 0, proc.stderr[-4000:]
    return torch.load(out_path, map_location="cpu")


def _same(a, b):
    return (torch.equal(a["out"].cpu(), b["out"].cpu()) and a["loss"] == b["loss"] and torch.equal(a["d_img"].cpu(), b["d_img"].cpu())
            and all(torch.equal(a["grads"][k].cpu(), b["grads"][k].cpu()) for k in a["grads"]))


@pytest.mark.gpu
def test_chain_and_persistent_paths(cuda, tmp_path):
    """configs[1] bf16 on the launch chain (ICD_LSTM_PERSISTENT=0, child process: read once per process) is within the bf16
    bounds of fp64 and of the persistent run (the two need not be bit-identical).  Both paths repeat bit for bit, and the
    chain with every launch stream-serialised (ICD_PDL_MASK=0) is bit-identical to the default chain: a difference would
    be a read before griddepcontrol.wait of data an earlier kernel of the chain writes."""
    from icd_b200 import ops
    c = _dims("cfg1")
    dec, img, caps = _module_and_inputs(c)
    assert ops.lstm_seq_supported(128, 25, 512)
    pers = [_run(dec, img, caps, "bf16", cuda) for _ in range(2)]
    assert _same(pers[0], pers[1]), "the persistent path is not run-to-run deterministic"
    chain = _child(tmp_path, "chain", ICD_LSTM_PERSISTENT="0")
    assert not chain["persistent"]
    assert chain["runs"][0]["launches"] >= 4 * c["L"]
    assert _same(chain["runs"][0], chain["runs"][1]), "the launch chain is not run-to-run deterministic"
    ser = _child(tmp_path, "chain_serialised", ICD_LSTM_PERSISTENT="0", ICD_PDL_MASK="0")
    assert _same(chain["runs"][0], ser["runs"][0]), "default and stream-serialised launch chains differ"
    ref = _oracle_cached("cfg1", dec, img, caps)
    fails, m = _compare(chain["runs"][0], ref, "bf16", caps)
    print("chain vs fp64:", " ".join("%s=%.3g" % kv for kv in m.items()))
    assert not fails, "\n".join(fails)
    as_ref = dict(out=pers[0]["out"].cpu().double(), loss=pers[0]["loss"], d_img=pers[0]["d_img"].cpu().double(),
                  grads={k: v.cpu().double() for k, v in pers[0]["grads"].items()})
    fails, m = _compare(chain["runs"][0], as_ref, "bf16", caps)
    print("chain vs persistent:", " ".join("%s=%.3g" % kv for kv in m.items()))
    assert not [f for f in fails if not f.startswith("greedy")], "\n".join(fails)
