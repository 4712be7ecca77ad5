"""CPU tier: the C-ABI library loads without a GPU and exports every symbol include/icd_b200.h declares; host-side
logic of the drop-in modules (constructor contract, state_dict keys, batch_size_t schedule, synthetic inputs)."""
import ctypes
import os
import re

import pytest
import torch

import helpers as H


def test_library_loads_and_exports_every_declared_symbol():
    from icd_b200 import _lib
    L = _lib.lib()
    header = open(_lib.HEADER).read()
    declared = re.findall(r"ICD_API\s+[\w\s\*]+?\b(icd_\w+)\s*\(", header)
    assert len(declared) >= 20 and sorted(declared) == sorted(_lib.FUNCTIONS)
    for name in declared:
        assert hasattr(L, name), "libicd_b200.so does not export " + name
    assert L.icd_version() == _lib.DEFINES["ICD_B200_ABI_VERSION"]
    assert L.icd_sizeof_att_desc() == ctypes.sizeof(_lib.AttDesc)
    assert L.icd_sizeof_base_desc() == ctypes.sizeof(_lib.BaseDesc)
    assert L.icd_sizeof_beam_desc() == ctypes.sizeof(_lib.BeamDesc)


def test_argument_errors_are_reported_without_a_gpu():
    from icd_b200 import _lib
    L = _lib.lib()
    d = _lib.GemmDesc()
    _lib.fill(d, M=4, N=4, K=4, sam=3, sak=2, sbn=4, sbk=1, ldc=4, precision=_lib.PREC_FP32)
    rc = L.icd_gemm(ctypes.byref(d), None)
    assert rc < 0 and b"unit stride" in L.icd_last_error_string()
    d.precision = 77
    assert L.icd_gemm(ctypes.byref(d), None) < 0
    with pytest.raises(_lib.IcdError):
        _lib.check(rc, "icd_gemm")


def test_product_path_refuses_cpu_tensors():
    """No CPU / eager fallback: the modules must fail loudly off-GPU."""
    import icd_b200.models.attention as my_att
    import icd_b200.models.baseline as my_base
    from icd_b200 import _lib
    from icd_b200.vocabulary import synthetic_vocab
    case = H.ATT_CASES["att_small_ragged"]
    dec = H.build_attention_module(case, my_att.AttentionDecoder, my_att.AttentionDecoderParams,
                                   synthetic_vocab(case["V"]))
    enc, caps, lens = H.att_inputs(case)
    with pytest.raises(_lib.IcdError):
        dec(enc, caps, lens)
    bcase = H.BASE_CASES["base_small"]
    bdec = H.build_baseline_module(bcase, my_base.BaselineDecoder, my_base.BaselineDecoderParams)
    img, bcaps, _ = H.base_inputs(bcase)
    with pytest.raises(_lib.IcdError):
        bdec(img, bcaps)


def test_no_product_module_imports_the_oracle():
    pkg = os.path.join(H.ROOT, "image-captioning-with-different-decoders_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f
                assert "/root/reference" not in src, f


def test_constructor_contract_and_state_dict_keys():
    import icd_b200.models.attention as my_att
    import icd_b200.models.baseline as my_base
    from icd_b200.vocabulary import Vocabulary, synthetic_vocab
    from oracle import decoders as O
    p = my_att.AttentionDecoderParams()
    assert (p.attention_dim, p.decoder_dim, p.embed_size, p.dropout, p.use_bert, p.vocab) == (512, 512, 512, 0.5, False, None)
    with pytest.raises(AssertionError):
        my_att.AttentionDecoder(torch.device("cpu"), object())
    with pytest.raises(AssertionError):
        my_att.AttentionDecoder(torch.device("cpu"), p)            # vocab must be a Vocabulary
    p.vocab = synthetic_vocab(50)
    p.attention_dim, p.decoder_dim, p.embed_size = 16, 12, 8
    dec = my_att.AttentionDecoder(torch.device("cpu"), p)
    assert list(dec.state_dict().keys()) == O.ATT_KEYS
    assert dec.vocab_size == 50 and dec.encoder_dim == 2048 and isinstance(dec.vocab, Vocabulary)
    assert dec.decode_step.weight_ih.shape == (48, 8 + 2048)
    assert torch.all(dec.fc.bias == 0) and float(dec.fc.weight.abs().max()) <= 0.1
    assert dec.embedding.weight.requires_grad
    dec.fine_tune_embeddings(False)
    assert not dec.embedding.weight.requires_grad
    tbl = torch.zeros(50, 8, dtype=torch.float64)
    dec.load_pretrained_embeddins(tbl)
    assert dec.embedding.weight.dtype == torch.float64 and dec.embedding.weight.requires_grad
    for attr in ("attention", "embedding", "decode_step", "h_lin", "c_lin", "f_beta", "sigmoid", "fc", "dropout"):
        assert hasattr(dec, attr)
    bp = my_base.BaselineDecoderParams()
    assert (bp.hidden_size, bp.embed_size, bp.vocab_size) == (512, 512, None)
    with pytest.raises(AssertionError):
        my_base.BaselineDecoder(bp)
    bp.vocab_size = 50
    bp.hidden_size = bp.embed_size = 8
    b = my_base.BaselineDecoder(bp)
    assert list(b.state_dict().keys()) == O.BASE_KEYS
    assert (b.embed_size, b.hidden_size) == (8, 8)


def test_vocabulary_layout_and_unknown_fallback():
    from icd_b200.vocabulary import END_TOKEN, PAD_TOKEN, START_TOKEN, UNK_TOKEN, synthetic_vocab
    v = synthetic_vocab(9490)
    assert len(v) == 9490
    assert (v(PAD_TOKEN), v(START_TOKEN), v(END_TOKEN), v(UNK_TOKEN)) == (0, 9487, 9488, 9489)
    assert v("never-seen-word") == v(UNK_TOKEN)
    assert v.i2w[v("w3")] == "w3"


def test_synthetic_inputs_shapes_and_schedule():
    from icd_b200 import synthetic
    enc = synthetic.features(3)
    assert enc.shape == (3, 14, 14, 2048) and float(enc.min()) == 0.0 and 0.3 < float(enc.mean()) < 0.5
    caps, lens = synthetic.captions(6, 100, max_len=12, lengths="ragged")
    assert caps.shape == (6, 12) and lens == sorted(lens, reverse=True) and lens[0] == 12
    for b, l in enumerate(lens):
        assert caps[b, 0] == 97 and caps[b, l - 1] == 98 and torch.all(caps[b, l:] == 0)
        assert torch.all((caps[b, 1:l - 1] >= 1) & (caps[b, 1:l - 1] <= 96))
    # batch_size_t schedule of models/attention.py:261 for unsorted lengths: a COUNT, rows taken positionally
    dl = [l - 1 for l in [5, 8, 3, 8]]
    bt = [sum(l > t for l in dl) for t in range(max(dl))]
    assert bt == [4, 4, 3, 3, 2, 2, 2]
    t = synthetic.glove_like_table(20)
    assert t.dtype == torch.float64 and t.shape == (20, 300)
    # the regime-B workload of bench.py (`configs[2]_regime_B_ragged_bf16`, SURVEY.md 8d): lengths U{8..25} sorted descending at
    # B = 512 -> 8133 decode tokens per step against 12 288 in regime A; batch_size_t falls from 512 to a few dozen rows
    caps, lens = synthetic.captions(512, 9490, max_len=25, lengths="ragged")
    assert lens == sorted(lens, reverse=True) and lens[0] == 25 and min(lens) >= 8
    dl = [l - 1 for l in lens]
    assert sum(dl) == 8133
    bt = [sum(l > t for l in dl) for t in range(max(dl))]
    assert len(bt) == 24 and bt[0] == 512 and bt[6] == 512 and bt[-1] < 48 and bt == sorted(bt, reverse=True)


def test_flat_param_buffer_views_share_storage():
    from icd_b200.parallel import FlatParamBuffer
    m = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 2))
    want = [p.detach().clone() for p in m.parameters()]
    buf = FlatParamBuffer(m)
    assert buf.flat.numel() == sum(p.numel() for p in m.parameters())
    for p, w in zip(m.parameters(), want):
        assert torch.equal(p.data, w)
    buf.flat.zero_()
    assert all(float(p.abs().sum()) == 0 for p in m.parameters())
    m(torch.ones(1, 4)).sum().backward()
    g = buf.gather_grads()
    assert torch.equal(g, torch.cat([p.grad.reshape(-1) for p in m.parameters()]))


def test_constructor_accepts_a_foreign_vocabulary_class_with_the_reference_surface():
    """A maintainer swapping imports (INTEGRATION.md level 1) passes the reference's own ``vocabulary.Vocabulary``."""
    import icd_b200.models.attention as my_att
    from icd_b200.vocabulary import Vocabulary as MyVocab

    class Vocabulary(object):          # same surface as the reference's vocabulary.py:8-35, different class object
        def __init__(self):
            self.w2i, self.i2w = {}, {}

        def add_word(self, w):
            if w not in self.w2i:
                self.i2w[len(self.w2i)] = w
                self.w2i[w] = len(self.w2i)

        def __call__(self, w):
            return self.w2i.get(w, self.w2i["<unk>"])

        def __len__(self):
            return len(self.w2i)

    v = Vocabulary()
    for w in ["<pad>", "a", "b", "<start>", "<end>", "<unk>"]:
        v.add_word(w)
    assert isinstance(v, MyVocab) and not isinstance(object(), MyVocab) and not isinstance({}, MyVocab)
    p = my_att.AttentionDecoderParams()
    p.vocab = v
    p.attention_dim = p.decoder_dim = p.embed_size = 8
    dec = my_att.AttentionDecoder(torch.device("cpu"), p)
    assert dec.vocab_size == 6


def test_contraction_plan_host_logic():
    """Pure host logic of the tensor-core tier (no GPU needed): the split-K workspace the plan asks for.
    * the per-step dh contraction (512 x 512 x 4608) runs as 4 K-slices of 64-wide tiles (cost model refitted in round 2 to the
      fixed issue path, DESIGN.md 5.2);
    * shapes that fill the GPU do not split;
    * d fc.weight (9490 x 512 x 12288): the 18-row last m-tile is split off into an 18-slice contraction, the 74 full
      m-tiles x 2 n-tiles = 148 tiles (one wave) need no workspace."""
    from icd_b200._lib import lib
    L = lib()
    L.icd_gemm_bf16_splitk_ws_floats.restype = ctypes.c_int64
    f = lambda M, N, K: int(L.icd_gemm_bf16_splitk_ws_floats(M, N, K))
    assert f(512, 512, 4608) == 4 * 512 * 512
    assert f(100352, 512, 2048) == 0 and f(12288, 9490, 512) == 0 and f(512, 4608, 512) == 0
    assert f(9490, 512, 12288) == 18 * 18 * 512
    assert f(9472, 512, 12288) == 0


def test_attention_step_launch_forms_host_logic(monkeypatch):
    """Pure host logic of the attention-step launchers (no GPU needed): which form a launch of `rows` rows takes
    (DESIGN.md 5.1).  148 SMs, at most 4 resident CTAs per SM (2 for the 128-register instantiations)."""
    from icd_b200._lib import lib, check
    for v in ("ICD_ATT_FWD_SPLIT", "ICD_ATT_BWD_SPLIT", "ICD_ATT_BWD_SPLIT_ROWS", "ICD_ATT_BWD_DEEP"):
        monkeypatch.delenv(v, raising=False)
    L = lib()

    def plan(direction, rows, P=196, C=2048, A=512):
        out = (ctypes.c_int32 * 4)()
        check(L.icd_attention_step_launch_plan_bf16(direction, rows, P, C, A, out), "launch_plan")
        return tuple(out)          # (CTAs per shared row, shared rows, grid, 128-register instantiation)
    # forward: four CTAs per row up to 48 rows, two up to 222, the deep instantiation while the grid stays within 2 CTAs per SM
    assert plan(0, 24) == (4, 24, 96, 1) and plan(0, 48) == (4, 48, 192, 1)
    assert plan(0, 100) == (2, 100, 200, 1) and plan(0, 148) == (2, 148, 296, 1)
    assert plan(0, 149) == (2, 149, 298, 0) and plan(0, 222) == (2, 222, 444, 0)
    assert plan(0, 223) == (1, 0, 223, 0) and plan(0, 512) == (1, 0, 512, 0)
    # backward: every row as two halves up to 222 rows (deep up to 148); above that the row balance over the 148 SMs
    assert plan(1, 32) == (2, 32, 64, 1) and plan(1, 148) == (2, 148, 296, 1) and plan(1, 200) == (2, 200, 400, 0)
    assert plan(1, 512) == (2, 80, 592, 0)            # full form: 432 whole + 160 halves = 4 CTAs per SM
    assert plan(1, 480) == (2, 112, 592, 0)
    assert plan(1, 320) == (2, 24, 344, 0)            # minimal form: the 24 rows beyond 2 per SM run as halves
    assert plan(1, 468) == (2, 24, 492, 0)
    assert plan(1, 296) == (1, 0, 296, 0) and plan(1, 444) == (1, 0, 444, 0) and plan(1, 592) == (1, 0, 592, 0)
    assert plan(1, 400) == (2, 44, 444, 0)
    assert plan(1, 256) == (2, 40, 296, 0)            # full form: 216 whole + 80 halves = 2 CTAs per SM
    assert plan(1, 230) == (1, 0, 230, 0)             # 82 rows beyond one per SM: neither form applies (66 > 230 / 4, 82 > 74)
    for rows in range(1, 700):                        # whole rows always pair up (2-CTA clusters); never more halves than rows
        per, shared, grid, deep = plan(1, rows)
        assert 0 <= shared <= rows and grid == rows + shared and (shared == 0 or (rows - shared) % 2 == 0)
        assert not deep or grid <= 296
        per, shared, grid, deep = plan(0, rows)
        assert grid == rows * per and (not deep or grid <= 296)
    assert plan(1, 300, P=16) == (1, 0, 300, 0)       # fewer than 32 pixels: rows are never shared
    # environment overrides (test hooks)
    monkeypatch.setenv("ICD_ATT_FWD_SPLIT", "1")
    assert plan(0, 24) == (1, 0, 24, 0)
    monkeypatch.setenv("ICD_ATT_BWD_SPLIT", "0")
    assert plan(1, 32) == (1, 0, 32, 0) and plan(1, 512) == (1, 0, 512, 0)
    monkeypatch.setenv("ICD_ATT_BWD_SPLIT", "2")
    assert plan(1, 512) == (2, 512, 1024, 0)
    monkeypatch.delenv("ICD_ATT_BWD_SPLIT")
    monkeypatch.setenv("ICD_ATT_BWD_DEEP", "0")
    assert plan(1, 32) == (2, 32, 64, 0)


def test_regime_b_schedule_visits_every_attention_step_launch_form(monkeypatch):
    """tests/test_gpu_ragged_regime_b.py checks the launch forms of the bf16 attention-step kernels against the oracle by running
    the regime-B schedule (batch_size_t 512 x 7, 488, ..., 46, 24).  If the plan rules change so that the schedule no longer
    reaches one of them, that test silently stops covering it: this fails instead."""
    from icd_b200 import synthetic
    from icd_b200._lib import lib, check
    for v in ("ICD_ATT_FWD_SPLIT", "ICD_ATT_BWD_SPLIT", "ICD_ATT_BWD_SPLIT_ROWS", "ICD_ATT_BWD_DEEP"):
        monkeypatch.delenv(v, raising=False)
    L = lib()
    _, lens = synthetic.captions(512, 9490, max_len=25, lengths="ragged")
    dl = [l - 1 for l in lens]
    bt = [sum(l > t for l in dl) for t in range(max(dl))]
    assert bt == [512] * 7 + [488, 467, 434, 410, 388, 362, 338, 298, 274, 244, 216, 186, 160, 126, 88, 46, 24]

    def plan(direction, rows):
        out = (ctypes.c_int32 * 4)()
        check(L.icd_attention_step_launch_plan_bf16(direction, rows, 196, 2048, 512, out), "launch_plan")
        return tuple(out)

    def fwd_form(rows):
        per, shared, grid, deep = plan(0, rows)
        return "%d per row%s" % (per, " deep" if deep else "")

    def bwd_form(rows):
        per, shared, grid, deep = plan(1, rows)
        if shared == 0:
            return "whole rows"
        if shared == rows:
            return "all halves" + (" deep" if deep else "")
        return "full balance" if grid % 148 == 0 else "minimal balance"    # full: rows + halves fill every SM equally
    fwd, bwd = {}, {}
    for r in bt:
        fwd.setdefault(fwd_form(r), []).append(r)
        bwd.setdefault(bwd_form(r), []).append(r)
    assert fwd == {"1 per row": [512] * 7 + [488, 467, 434, 410, 388, 362, 338, 298, 274, 244], "2 per row": [216, 186, 160],
                   "2 per row deep": [126, 88], "4 per row deep": [46, 24]}
    assert set(bwd) == {"full balance", "minimal balance", "all halves", "all halves deep"}
    assert bwd["minimal balance"] == [467, 338, 298] and 512 in bwd["full balance"] and 488 in bwd["full balance"]
    assert bwd["all halves"] == [216, 186, 160] and bwd["all halves deep"] == [126, 88, 46, 24]


def test_version_counter_guard_of_the_autograd_functions():
    """The decoders' backward reads weights through raw pointers; `_lib.remember_versions` / `check_versions` stand in for
    autograd's saved-tensor check (pure host logic: CPU tensors suffice)."""
    from icd_b200 import _lib

    class Ctx:
        pass
    ctx = Ctx()
    w, b, other = torch.zeros(3, 3), torch.zeros(3), object()
    _lib.remember_versions(ctx, [("fc.weight", w), ("fc.bias", b), ("not_a_tensor", other), ("absent", None)])
    _lib.check_versions(ctx, "Decoder")                      # untouched: passes
    view = w[0]
    view.add_(1.0)                                           # an in-place update through a VIEW bumps the base's counter too
    with pytest.raises(RuntimeError, match="'fc.weight' needed for the backward was modified by an in-place operation"):
        _lib.check_versions(ctx, "Decoder")
    _lib.check_versions(Ctx(), "Decoder")                    # a ctx that recorded nothing checks nothing


def test_reference_install_is_a_verbatim_copy():
    """baseline/_ref (bench.py's reference arm) holds the UNMODIFIED reference: every installed file hashes like its source
    (when the source tree is present) and like the manifest written at install time."""
    import hashlib
    import json
    import os
    ref = os.path.join(H.ROOT, "baseline", "_ref")
    man_path = os.path.join(ref, "MANIFEST.json")
    if not os.path.exists(man_path):
        pytest.skip("baseline/_ref not installed here")
    man = json.load(open(man_path))
    assert "models/attention.py" in man["files"] and "gen_captions.py" in man["files"]
    for rel, sha in man["files"].items():
        assert hashlib.sha256(open(os.path.join(ref, rel), "rb").read()).hexdigest() == sha, rel
        src = os.path.join("/root/reference", rel)
        if os.path.exists(src):
            assert hashlib.sha256(open(src, "rb").read()).hexdigest() == sha, "installed copy differs from the reference: " + rel
    # nothing of it is tracked by git
    import subprocess
    out = subprocess.run(["git", "ls-files", "baseline/_ref"], cwd=H.ROOT, capture_output=True, text=True).stdout.strip()
    assert out == "", "baseline/_ref must stay out of the repository history"
