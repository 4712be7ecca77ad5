"""CPU tier: the sampling definition (tests/sampling_reference.py) — its generator against Random123's known answers, its
greedy and top-1 limits against the baseline beam search, its draw distribution at a fixed seed — and the sampler's C ABI:
descriptor layout and argument / size-query refusals through the built library (no GPU needed)."""
import ctypes
import math

import numpy as np
import pytest
import torch
from scipy import stats

import baseline_beam_reference as BR
import sampling_reference as SR


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    got = SR.philox4x32_10(*ctr, *key)
    assert tuple(int(x) for x in got) == want


def test_uniforms_are_strictly_inside_the_unit_interval():
    bits = np.array([0, 255, 256, 0xFFFFFFFF, 0xFFFFFF00], dtype=np.uint32)
    u = ((bits >> 8).astype(np.float64) + 0.5) * 2.0 ** -24
    assert (u > 0).all() and (u < 1).all()
    assert np.isfinite(SR.gumbel(bits)).all()


def _small_baseline():
    import icd_b200.models.baseline as my_base
    p = my_base.BaselineDecoderParams()
    p.hidden_size, p.embed_size, p.vocab_size = 32, 24, 131
    torch.manual_seed(0)
    dec = my_base.BaselineDecoder(p)
    V = 131
    with torch.no_grad():
        dec.embedding.weight *= 30.0
        dec.linear.weight[V - 2] *= 15.0
        dec.linear.bias[V - 2] = -8.0
    w = {k: v.detach().double() for k, v in dec.state_dict().items()}
    imgs = torch.randn(6, 24, generator=torch.Generator().manual_seed(5)).double()
    return w, imgs, V


def test_greedy_sample_is_the_k1_beam_search():
    w, imgs, V = _small_baseline()
    for i in range(imgs.shape[0]):
        seq, ended = BR.baseline_beam_search(w, imgs[i], 1, V - 3, V - 2, max_steps=30)
        step, st = SR.baseline_start(w, imgs[i])
        s = SR.sample_image(step, st, 1, V - 3, V - 2, 30, 0.0, 0, 1234, i)[0]
        if ended:
            assert s["ended"] and s["seq"] == seq
        else:
            assert not s["ended"] and s["len"] == 32


def test_top1_equals_greedy():
    w, imgs, V = _small_baseline()
    for i in range(3):
        step, st = SR.baseline_start(w, imgs[i])
        g = SR.sample_image(step, st, 2, V - 3, V - 2, 20, 0.0, 0, 7, i)
        t1 = SR.sample_image(step, st, 2, V - 3, V - 2, 20, 1.3, 1, 7, i)
        for a, b in zip(g, t1):
            assert a["seq"] == b["seq"] and a["score"] == b["score"]


@pytest.mark.parametrize("temperature,top_k", [(1.0, 0), (0.7, 5), (1.5, 12)])
def test_seeded_draws_follow_the_restricted_softmax(temperature, top_k):
    """Deterministic (fixed seed) chi-square of 6000 draws against softmax(l / T) over the top-k; nothing outside it."""
    V = 40
    l = torch.randn(V, generator=torch.Generator().manual_seed(3), dtype=torch.float64) * 2.0
    cand = SR.candidates(l.numpy(), top_k)
    p = torch.softmax(l[torch.as_tensor(cand)] / temperature, dim=0).numpy()
    n = 6000
    counts = np.zeros(V, dtype=np.int64)
    for j in range(n):
        tok, _, _ = SR.select(l, temperature, top_k, seed=0xC0FFEE, step=1, img=0, sample=j)
        counts[tok] += 1
    outside = np.setdiff1d(np.arange(V), cand)
    assert counts[outside].sum() == 0
    obs, exp = counts[cand], p * n
    big = exp >= 5                                          # pool the rare cells so the test is valid
    obs = np.append(obs[big], obs[~big].sum()) if (~big).any() else obs[big]
    exp = np.append(exp[big], exp[~big].sum()) if (~big).any() else exp[big]
    assert stats.chisquare(obs, exp).pvalue > 1e-3


# ------------------------------------------------------------------------------------------------------------ C ABI
def _att_desc(**over):
    from icd_b200 import _lib
    d = _lib.SampleDesc()
    fake = 256                                              # non-null device addresses: no CUDA call happens before validation
    kw = dict(n_img=4, m=5, max_steps=20, P=196, C=2048, A=48, D=32, E=24, V=131, precision=_lib.PREC_FP32X3,
              start_id=128, end_id=129, top_k=0, temperature=1.0, seed=1)
    for name, _ in d._fields_:
        if name.startswith(("enc", "dec_", "full_", "w_", "b_", "h_lin", "c_lin", "f_beta", "fc_", "emb_w", "out_")):
            setattr(d, name, fake)
    kw.update(over)
    return _lib.fill(d, **kw)


def _base_desc(**over):
    from icd_b200 import _lib
    d = _lib.BaseSampleDesc()
    kw = dict(n_img=4, m=5, max_steps=20, E=24, H=32, V=131, precision=_lib.PREC_FP32, start_id=128, end_id=129, top_k=0,
              temperature=1.0, seed=1)
    for name, _ in d._fields_:
        if name.startswith(("img_features", "emb_w", "w_", "b_", "lin_", "out_")):
            setattr(d, name, 256)
    kw.update(over)
    return _lib.fill(d, **kw)


def test_sampler_descriptor_layout():
    from icd_b200 import _lib
    L = _lib.lib()
    assert L.icd_sizeof_sample_desc() == ctypes.sizeof(_lib.SampleDesc)
    assert L.icd_sizeof_base_sample_desc() == ctypes.sizeof(_lib.BaseSampleDesc)
    assert _lib.DEFINES["ICD_B200_ABI_VERSION"] == 18


BAD = [dict(m=0), dict(m=9), dict(temperature=-0.5), dict(temperature=math.nan), dict(temperature=math.inf),
       dict(top_k=132), dict(top_k=-1), dict(n_img=13108, m=5), dict(precision=None)]


@pytest.mark.parametrize("which", ["attention", "baseline"])
@pytest.mark.parametrize("bad", range(len(BAD)))
def test_sampler_refuses_bad_arguments(which, bad):
    from icd_b200 import _lib
    L = _lib.lib()
    over = dict(BAD[bad])
    if "precision" in over:
        over["precision"] = _lib.PREC_BF16
    mk, size, run = ((_att_desc, L.icd_sample_captions_ws_bytes, L.icd_sample_captions) if which == "attention" else
                     (_base_desc, L.icd_baseline_sample_captions_ws_bytes, L.icd_baseline_sample_captions))
    good = mk()
    assert size(ctypes.byref(good)) > 0
    d = mk(**over)
    assert size(ctypes.byref(d)) == -1
    d.ws, d.ws_bytes = 256, 1 << 40
    assert run(ctypes.byref(d), None) < 0
    assert L.icd_last_error_string()


@pytest.mark.parametrize("which", ["attention", "baseline"])
def test_sampler_refuses_a_small_workspace_and_null_results(which):
    from icd_b200 import _lib
    L = _lib.lib()
    mk, size, run = ((_att_desc, L.icd_sample_captions_ws_bytes, L.icd_sample_captions) if which == "attention" else
                     (_base_desc, L.icd_baseline_sample_captions_ws_bytes, L.icd_baseline_sample_captions))
    d = mk()
    need = size(ctypes.byref(d))
    d.ws, d.ws_bytes = 256, need - 1
    assert run(ctypes.byref(d), None) < 0 and b"workspace" in L.icd_last_error_string()
    d = mk(out_score=None)
    d.ws, d.ws_bytes = 256, need
    assert run(ctypes.byref(d), None) < 0 and b"null" in L.icd_last_error_string()


def test_sampler_workspace_does_not_grow_with_the_step_cap():
    """No per-step history: a longer cap adds only the per-step ticket counters (one int per step)."""
    from icd_b200 import _lib
    L = _lib.lib()
    a = L.icd_sample_captions_ws_bytes(ctypes.byref(_att_desc(n_img=1024, m=5, max_steps=24, V=9490, A=512, D=512, E=512)))
    b = L.icd_sample_captions_ws_bytes(ctypes.byref(_att_desc(n_img=1024, m=5, max_steps=50, V=9490, A=512, D=512, E=512)))
    assert 0 < a and b - a <= 256
    bd = _lib.BeamDesc()
    _lib.fill(bd, n_img=1024, k=5, max_steps=50, P=196, C=2048, A=512, D=512, E=512, V=9490, precision=_lib.PREC_FP32X3)
    assert L.icd_beam_search_ws_bytes(ctypes.byref(bd)) - b > 200e6          # the beam search's alpha frames and pointers
    c = L.icd_baseline_sample_captions_ws_bytes(ctypes.byref(_base_desc(max_steps=24)))
    e = L.icd_baseline_sample_captions_ws_bytes(ctypes.byref(_base_desc(max_steps=200)))
    assert c == e
