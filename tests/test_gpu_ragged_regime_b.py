"""GPU tier: parity of the attention train step in length regime B at full size — the workload bench.py times as
`configs[2]_regime_B_ragged_bf16`: B = 512 captions of lengths U{8..25} sorted descending, V = 9490, A = D = E = 512,
embedding frozen, train mode with a shared seeded dropout keep-mask, plus the gradient w.r.t. encoder_out
(--fine_tune_encoder).  batch_size_t per step (models/attention.py:261-265):
    512 x 7, 488, 467, 434, 410, 388, 362, 338, 298, 274, 244, 216, 186, 160, 126, 88, 46, 24
so one step of the bf16 tier runs every launch form of the bf16 attention-step kernels inside one PDL chain: forward with 1, 2
and 4 CTAs per row (2 per row with and without the 128-register instantiation), backward in the full row-balance form, the
minimal form and with every row as a half-row cluster (deep at <= 148 rows) — tests/test_abi_and_host.py checks that this
schedule still visits each of them.  The timed configuration (regime A, tests/test_gpu_timed_config.py) keeps 512 rows at
every step and reaches none of the shared forms.

Everything is compared with the fp64 oracle on the same 512 rows (tests/helpers.oracle_fp64_chunked), and not only norm-wise
over whole tensors: a bug confined to the 24 rows of the last step or to the rows one launch form computes touches ~1 % of
the tokens, which a norm-wise bound on a whole gradient cannot see.  Stated bounds (measured values: profiles/r03_regime_b_parity.md, written as JSON to $ICD_REGIME_B_TABLE when set):
    aggregate   predictions, alphas 5e-3 | loss 1e-3 | gradients and d encoder_out 1e-2, the four attention projections 5e-2
                (bf16 tiers);  1e-4 | 1e-5 | 1e-3, fp32x3 3e-3 on the four (fp32-class tiers);  full_att.bias max abs 1e-4
    per step    predictions[:bt[t], t] and alphas[:bt[t], t] of every step t within the aggregate bound
    per row     d encoder_out[b] of every row b within ROW_BOUND of the tier, and max_b <= ROW_K x median_b.  In the fp32-class
                tiers a few rows exceed ROW_K x the median for a known reason: where att_enc + att_dec lies within rounding of
                0, the relu mask of the kernel and of the oracle can differ, which moves d att_enc[b, p, a] by w[a] d_e[b, t, p]
                and d encoder_out[b, p] by that times enc_att.weight[a] — an error along one row of enc_att.weight at one
                pixel (measured: median row 1.8e-6, worst 2.4e-4 in fp32; 81 of 512 rows beyond ROW_K x the median).  Such a row passes when its error with those
                components removed (_kink_residual) is within KINK_K x the median (measured: 2.37e-4 -> 5.0e-6 = 2.8 x the
                median; what remains is the flip's small effect through d att_dec on the recurrence); the bf16 tiers round att_enc itself, their
                rows are uniform and no such allowance is made.
    inactive    predictions and alphas at t >= decode_length[b] exactly 0
    bf16: bit-identical with bf16_grad_only; parameter gradients bit-identical with encoder_out.requires_grad on and off
    launch forms: one CTA per row everywhere (ICD_ATT_FWD_SPLIT=1, ICD_ATT_BWD_SPLIT=0) gives bit-identical predictions and
                alphas (the forward split is bit-identical by design); gradients and d encoder_out within AB_BOUND of the
                default run (only the pixel-split sums of the backward reorder), and the per-row criterion against the oracle
    PDL: the same step with every launch stream-serialised (ICD_PDL_MASK=0, child process: the mask is read once per process)
                is bit-identical to the default run for every tier that is run-to-run deterministic.
"""
import hashlib
import json
import os
import subprocess
import sys

import pytest
import torch

import helpers as H

pytestmark = pytest.mark.gpu

V, A, D, E, MAXLEN, B = 9490, 512, 512, 512, 25, 512
T = MAXLEN - 1
ILL = ("attention.enc_att.weight", "attention.enc_att.bias", "attention.dec_att.weight", "attention.dec_att.bias")
TIERS = ("bf16+bf16_grad_only", "bf16", "fp32x3", "fp32")
ONE_CTA = "bf16 one CTA per row"
ROW_BOUND = {"bf16": 1e-2, "fp32x3": 1.2e-3, "fp32": 5e-4}       # ~2x the worst row measured on a B200 (1000 W)
ROW_K = 2.5
AB_BOUND = 3e-4
KINK_K = 6.0                         # fp32-class tiers: such a row without its kink components within KINK_K x the median
KINK_ROWS = 128                      # fp32-class tiers: rows beyond ROW_K x the median allowed (measured 72 / 81 of 512)
_TESTS = os.path.dirname(os.path.abspath(__file__))


def _inputs():
    from icd_b200 import synthetic
    enc = synthetic.features(B)                                           # bench.py measure_attention(ragged=True)
    caps, lens = synthetic.captions(B, V, max_len=MAXLEN, lengths="ragged")
    keep = H.seeded_keep_mask(T, B, D, 0.5, seed=4321)
    return enc, caps, lens, keep


def _module(cuda, precision):
    """bench.py's construction: seed 0, embedding frozen, train mode."""
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import synthetic_vocab
    p = my_att.AttentionDecoderParams()
    p.vocab = synthetic_vocab(V)
    torch.manual_seed(0)
    dec = my_att.AttentionDecoder(cuda, p)
    dec.fine_tune_embeddings(False)
    sd = {k: v.detach().clone() for k, v in dec.state_dict().items()}
    dec = dec.to(cuda)
    dec.precision = precision
    dec.train()
    return dec, sd


def _step(cuda, tier, enc_d, caps_d, lens, keep, enc_grad=True):
    """One train step -> dict(preds, alphas on the host, loss, grads on the host, d_enc on the device or None, sd)."""
    from icd_b200.losses import attention_caption_loss
    dec, sd = _module(cuda, tier.split("+")[0])
    dec._dropout_mask_override = keep
    x = enc_d.detach().requires_grad_(enc_grad)
    preds, cs, dl, alphas = dec(x, caps_d, lens)
    loss = attention_caption_loss(preds, cs, dl, alphas, alpha_c=1.0, bf16_grad_only=tier.endswith("grad_only"))
    loss.backward()
    out = dict(preds=preds.detach().cpu(), alphas=alphas.detach().cpu(), loss=float(loss.item()), sd=sd,
               grads={k: p.grad.detach().cpu() for k, p in dec.named_parameters() if p.grad is not None},
               d_enc=(x.grad.reshape(B, -1, x.shape[-1]) if enc_grad else None))
    del dec, preds, alphas, loss, x
    torch.cuda.empty_cache()
    return out


def _same(a, b, what=("preds", "alphas", "grads", "d_enc")):
    """-> names of the outputs that are not bit-identical"""
    diff = []
    for k in what:
        if k == "grads":
            diff += ["grad:" + n for n in a["grads"] if not torch.equal(a["grads"][n], b["grads"][n])]
        elif not torch.equal(a[k], b[k]):
            diff.append(k)
    return diff


def _digests(o):
    """Per-row SHA-256 of predictions, alphas and d encoder_out, and of every parameter gradient: a bit-for-bit fingerprint
    that says which rows differ."""
    def rows(t):
        t = t.detach().cpu().contiguous().reshape(t.shape[0], -1)
        return [hashlib.sha256(t[b].numpy().tobytes()).hexdigest()[:24] for b in range(t.shape[0])]
    return dict(preds=rows(o["preds"]), alphas=rows(o["alphas"]), d_enc=rows(o["d_enc"]), loss=o["loss"],
                grads={k: H.checksum(g) for k, g in o["grads"].items()})


def child_main(out_path, tiers):
    """Entry point of the child process of test_stream_serialised_launches_are_bit_identical (ICD_PDL_MASK=0)."""
    cuda = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    enc, caps, lens, keep = _inputs()
    enc_d, caps_d = enc.to(cuda), caps.to(cuda)
    res = {t: _digests(_step(cuda, t, enc_d, caps_d, lens, keep)) for t in tiers}
    with open(out_path, "w") as f:
        json.dump(res, f)


@pytest.fixture(scope="module")
def regime_b(cuda):
    enc, caps, lens, keep = _inputs()
    dl = [l - 1 for l in lens]
    bt = [sum(l > t for l in dl) for t in range(T)]
    enc_d, caps_d = enc.to(cuda), caps.to(cuda)
    out = {t: _step(cuda, t, enc_d, caps_d, lens, keep) for t in TIERS}
    # the same bf16 step without the encoder gradient: its parameter gradients
    no_enc = _step(cuda, "bf16", enc_d, caps_d, lens, keep, enc_grad=False)["grads"]
    # every step on one CTA per row (forward and backward)
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("ICD_ATT_FWD_SPLIT", "1")
        mp.setenv("ICD_ATT_BWD_SPLIT", "0")
        out[ONE_CTA] = _step(cuda, "bf16", enc_d, caps_d, lens, keep)
    # run-to-run determinism, in process: which tiers the PDL A/B can compare bit for bit
    deterministic = {"bf16": _same(out["bf16"], _step(cuda, "bf16", enc_d, caps_d, lens, keep))}
    for t in ("fp32x3", "fp32"):
        deterministic[t] = _same(out[t], _step(cuda, t, enc_d, caps_d, lens, keep))
    torch.set_num_threads(os.cpu_count() or 1)
    cands = tuple(TIERS) + (ONE_CTA,)
    ref = H.oracle_fp64_chunked(out["fp32"]["sd"], enc, caps, lens, keep_mask=keep, p=0.5, frozen=("embedding.weight",),
                                chunk=64, cuda_preds={t: out[t]["preds"] for t in cands},
                                cuda_alphas={t: out[t]["alphas"] for t in cands}, per_step=True,
                                cuda_d_enc={t: out[t]["d_enc"] for t in cands})
    table = {}
    for tier in cands:
        row = {"predictions": ref["err"][tier]["predictions"], "alphas": ref["err"][tier]["alphas"],
               "loss": abs(out[tier]["loss"] - ref["loss"]) / abs(ref["loss"])}
        for k, g in ref["grads"].items():
            row["grad:" + k] = (float(out[tier]["grads"][k].abs().max()) if k == "attention.full_att.bias"
                                else H.rel_err(out[tier]["grads"][k], g))
        ps, pa = (H.step_rel_err(ref["step_sums"][tier][n]) for n in ("predictions", "alphas"))
        re = H.row_rel_err(ref["row_sums"][tier])
        row.update({"worst_step_predictions": float(ps.max()), "worst_step_predictions_t": int(ps.argmax()),
                    "worst_step_alphas": float(pa.max()), "worst_step_alphas_t": int(pa.argmax()),
                    "d_enc": H.aggregate_rel_err(ref["row_sums"][tier]), "d_enc_worst_row": float(re.max()),
                    "d_enc_worst_row_b": int(re.argmax()), "d_enc_median_row": float(re.median())})
        table[tier] = row
    ab = {"grad:" + k: H.rel_err(out[ONE_CTA]["grads"][k], out["bf16"]["grads"][k]) for k in out["bf16"]["grads"]
          if k != "attention.full_att.bias"}
    ab["d_enc"] = H.rel_err(out[ONE_CTA]["d_enc"], out["bf16"]["d_enc"])
    kink = {}
    for tier in ("fp32x3", "fp32"):
        err = H.row_rel_err(ref["row_sums"][tier])
        rows = (err > ROW_K * float(err.median())).nonzero().flatten().tolist()[:KINK_ROWS + 1]
        kink[tier] = [(i, _kink_residual(out[tier]["sd"], enc, caps, lens, keep, i, out[tier]["d_enc"][i])) for i in rows]
        table[tier]["rows_beyond_%g_median" % ROW_K] = len(rows)
        table[tier]["worst_kink_residual"] = max([v for _, v in kink[tier]], default=0.0)
    path = os.environ.get("ICD_REGIME_B_TABLE")
    if path:
        with open(path, "w") as f:
            json.dump({"config": "configs[2] length regime B: B=512, lengths U{8..25} sorted descending, T=24, V=9490, "
                                 "A=D=E=512, dropout 0.5 (shared keep-mask), embedding frozen, + d encoder_out; fp64 oracle "
                                 "on the same 512 rows", "batch_size_t": bt, "oracle_loss": ref["loss"], "table": table,
                       "launch_form_ab": ab, "run_to_run_differences": deterministic}, f, indent=1)
    print("\nregime B, measured errors vs the fp64 oracle:")
    for tier in cands:
        print(" ", tier, {k: ("%.2e" % v if isinstance(v, float) else v) for k, v in table[tier].items()})
    print("  launch-form A/B:", {k: "%.2e" % v for k, v in ab.items()})
    print("  run-to-run differences:", deterministic)
    return dict(out=out, ref=ref, table=table, ab=ab, no_enc=no_enc, deterministic=deterministic, dl=dl, bt=bt, kink=kink)


def _bounds(tier):
    bf16 = tier.startswith("bf16")
    return dict(out=5e-3 if bf16 else 1e-4, loss=1e-3 if bf16 else 1e-5, grad=1e-2 if bf16 else 1e-3,
                ill=5e-2 if bf16 else (3e-3 if tier == "fp32x3" else 1e-3),
                row=ROW_BOUND["bf16" if bf16 else tier])


def _kink_residual(sd, enc, caps, lens, keep, b, got):
    """Row b's d encoder_out error against the fp64 oracle of that row alone, with each pixel's component along its best-aligned
    row of enc_att.weight removed (a relu-kink flip, see the module docstring) -> relative residual."""
    from oracle import decoders as O
    import torch.nn.functional as F
    dl = [l - 1 for l in lens]
    w64 = {k: v.detach().cpu().double() for k, v in sd.items()}
    e64 = enc[b:b + 1].double().reshape(1, -1, enc.shape[-1]).requires_grad_(True)
    masks = [keep[t, b:b + 1].double() for t in range(dl[b])]
    pr, _, _, al = O.attention_decoder_forward(w64, e64, caps[b:b + 1], [lens[b]], dropout_p=0.5, dropout_masks=masks, hoist=True)
    P = e64.shape[1]
    ce = F.cross_entropy(pr[0, :dl[b]], caps[b, 1:dl[b] + 1], reduction="sum") / sum(dl)
    reg = ((1.0 - al.sum(dim=1)) ** 2).sum() / (B * P)
    (ce + reg).backward()
    ref = e64.grad[0]
    err = got.detach().cpu().double().reshape(P, -1) - ref
    U = w64["attention.enc_att.weight"]
    U = U / U.norm(dim=1, keepdim=True)
    for _ in range(2):                                                    # up to two flips at one pixel
        c = err @ U.t()                                                   # (P, A) components
        a = c.abs().argmax(dim=1)
        err = err - c.gather(1, a[:, None]) * U[a]
    return float(err.norm() / ref.norm())


def _check_against_oracle(r, tier):
    b = _bounds(tier)
    row = r["table"][tier]
    assert row["predictions"] < b["out"] and row["alphas"] < b["out"], row
    assert row["loss"] < b["loss"]
    for k, v in row.items():
        if not k.startswith("grad:"):
            continue
        name = k[5:]
        if name == "attention.full_att.bias":
            assert v < 1e-4, "full_att.bias gradient (true value 0): max abs %.2e" % v
        else:
            assert v < (b["ill"] if name in ILL else b["grad"]), "%s: %.2e" % (name, v)
    assert "grad:embedding.weight" not in row
    assert row["d_enc"] < b["grad"], "d encoder_out: %.2e" % row["d_enc"]
    # per step: the last steps (46 and 24 rows) as much as the first
    for name in ("predictions", "alphas"):
        e = H.step_rel_err(r["ref"]["step_sums"][tier][name])
        bad = [(t, r["bt"][t], "%.2e" % float(e[t])) for t in range(T) if float(e[t]) >= b["out"]]
        assert not bad, "%s: steps (t, batch_size_t, error) over %.0e: %s" % (name, b["out"], bad)
    # per row: d encoder_out of every row, and no row out of line with the rest
    err = H.row_rel_err(r["ref"]["row_sums"][tier])
    if tier.startswith("bf16"):
        fails = H.row_spread_failures(err, b["row"], ROW_K)
    else:
        fails = H.row_spread_failures(err, b["row"], float("inf"))
        med = float(err.median())
        out = (err > ROW_K * med).nonzero().flatten().tolist()
        assert len(out) <= KINK_ROWS, "%d rows beyond %g x the median" % (len(out), ROW_K)
        fails += ["row %d: %.2e, %.2e without its relu-kink components (median %.2e)" % (i, float(err[i]), res, med)
                  for i, res in r["kink"][tier] if res > KINK_K * med]
    assert not fails, "d encoder_out per row: " + "; ".join(fails)


@pytest.mark.parametrize("tier", TIERS)
def test_regime_b_matches_fp64_oracle_per_step_and_per_row(regime_b, tier):
    _check_against_oracle(regime_b, tier)
    # inactive positions (t >= decode_length[b]) are exactly 0 (models/attention.py:253, 257)
    o = regime_b["out"][tier]
    inactive = torch.arange(T)[None, :] >= torch.tensor(regime_b["dl"])[:, None]
    assert int(inactive.sum()) == B * T - 8133
    assert torch.all(o["preds"][inactive] == 0) and torch.all(o["alphas"][inactive] == 0)


def test_regime_b_bf16_bit_identities(regime_b):
    out = regime_b["out"]
    a, b = out["bf16"], out["bf16+bf16_grad_only"]
    assert a["loss"] == b["loss"]
    assert not _same(a, b), "bf16 vs bf16_grad_only"
    # the encoder-gradient path adds work after the time loop; it must not change a parameter gradient
    diff = [k for k in a["grads"] if not torch.equal(a["grads"][k], regime_b["no_enc"][k])]
    assert not diff, "parameter gradients differ with encoder_out.requires_grad on / off: %s" % diff


def test_regime_b_launch_forms_agree(regime_b):
    """Every step on one CTA per row against the default launch forms (all of them, see the module docstring)."""
    one, dflt = regime_b["out"][ONE_CTA], regime_b["out"]["bf16"]
    assert torch.equal(one["preds"], dflt["preds"]) and torch.equal(one["alphas"], dflt["alphas"])
    assert one["loss"] == dflt["loss"]
    worst = max(regime_b["ab"].items(), key=lambda kv: kv[1])
    assert worst[1] < AB_BOUND, "launch forms differ by %.2e in %s" % (worst[1], worst[0])
    _check_against_oracle(regime_b, ONE_CTA)


def test_stream_serialised_launches_are_bit_identical(regime_b, tmp_path):
    """ICD_PDL_MASK=0: no kernel starts before its predecessor has finished.  Any difference from the default run (early
    starts) is a read before griddepcontrol.wait of data an earlier kernel of the chain writes."""
    tiers = [t for t in ("bf16", "fp32x3", "fp32") if not regime_b["deterministic"][t]]
    assert "bf16" in tiers, "the bf16 tier must be run-to-run deterministic: %s" % regime_b["deterministic"]["bf16"]
    out_path = str(tmp_path / "serialised.json")
    env = {k: v for k, v in os.environ.items() if not k.startswith("ICD_ATT_")}
    env["ICD_PDL_MASK"] = "0"
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_ragged_regime_b as m; m.child_main(%r, %r)"
            % (H.ROOT, _TESTS, out_path, tiers))
    flags = ["-s"] if sys.flags.no_user_site else []
    proc = subprocess.run([sys.executable] + flags + ["-c", code], env=env, cwd=H.ROOT, capture_output=True, text=True,
                          timeout=1200)
    assert proc.returncode == 0, proc.stderr[-4000:]
    with open(out_path) as f:
        child = json.load(f)
    for t in tiers:
        mine, ser = _digests(regime_b["out"][t]), child[t]
        assert mine["loss"] == ser["loss"], t
        for k in ("preds", "alphas", "d_enc"):
            rows = [b for b in range(B) if mine[k][b] != ser[k][b]]
            assert not rows, "%s %s: rows differ between default and stream-serialised launches: %s" % (t, k, rows[:32])
        diff = [k for k in mine["grads"] if mine["grads"][k] != ser["grads"][k]]
        assert not diff, "%s: gradients differ between default and stream-serialised launches: %s" % (t, diff)
