"""CPU checks of oracle/readout.py: the constructed inputs give exact logits, the prefix scan is the softmax, and an
emulation of the kernels' rounding stays well inside the error bound on every profile, dtype and length the GPU readout
tests use (tests/test_gpu_readout.py)."""
import math

import pytest
import torch

from oracle import readout as ro

F64 = torch.float64


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16, torch.float32])
@pytest.mark.parametrize("D", [48, 64, 80, 128])
def test_constructed_scores_are_exact(dtype, D):
    g = torch.Generator().manual_seed(D)
    n, T = 300, (1, 2, 4)
    scale = D ** -0.5
    for name in ro.PROFILES:
        s = ro.profile(name, n, g, scale, dtype)
        k, v = ro.make_kv(s, ro.classes(n, D, g), D, dtype)
        q, t = ro.make_q(torch.arange(2 * D), D, T, dtype)
        prod = q.to(F64) @ k.to(F64).T                                    # what the MMA sums: one nonzero term per key
        assert torch.equal(prod, t[:, None] * s[None, :]), name
        assert torch.equal(prod.to(torch.float32).to(F64), prod), name   # and exact in fp32
        assert torch.equal(v.to(F64).sum(1), torch.ones(n, dtype=F64))
    cols = (q.to(F64) != 0).to(torch.int64).argmax(1)
    assert set(cols.tolist()) == set(range(D))                           # every Q/K column carries some row's score


def test_big_raw_scores_exceed_fp16_with_moderate_logits():
    g = torch.Generator().manual_seed(1)
    s = ro.profile("bigraw", 500, g, 2.0 ** -16, torch.float16)
    k, _ = ro.make_kv(s, ro.classes(500, 64, g), 64, torch.float16)
    assert torch.isfinite(k.float()).all()
    q, t = ro.make_q(torch.arange(64), 64, (8, 16), torch.float16)
    raw = q.to(F64) @ k.to(F64).T
    assert raw.abs().max() > 65504 and (raw * 2.0 ** -16).abs().max() < 8


def _direct(s, cls, D, a):
    x = a * s
    W, lse = [], []
    for p in range(1, s.numel() + 1):
        w = torch.softmax(x[:p], 0)
        W.append(torch.zeros(D, dtype=F64).index_add_(0, cls[:p], w))
        lse.append(torch.logsumexp(x[:p], 0))
    return torch.stack(W), torch.stack(lse)


@pytest.mark.parametrize("case", ["noise", "ramp1500", "sink", "needle", "tiny"])
def test_prefix_scan_matches_direct_softmax(case):
    g = torch.Generator().manual_seed(7)
    D = 16
    n = {"tiny": 3, "ramp1500": 1000}.get(case, 200)
    if case == "ramp1500":
        s = torch.arange(n, dtype=F64) * 1.5                            # 1500 nats from first to last key
    elif case == "sink":
        s = torch.randn(n, generator=g, dtype=F64)
        s[2] = 500.0
    elif case == "needle":
        s = torch.zeros(n, dtype=F64)
        s[77] = 30.0
    else:
        s = 16 * torch.randn(n, generator=g, dtype=F64)
    cls = ro.classes(n, D, g)
    for a in (1.0, 0.25):
        W, lse, wmax, counts = ro.prefix_reference(s, cls, D, a)
        Wd, lsed = _direct(s, cls, D, a)
        assert ((W - Wd).abs() <= 1e-12 * Wd.abs() + 1e-300).all()
        assert ((lse - lsed).abs() <= 1e-12 * lsed.abs().clamp_min(1)).all()
        assert torch.allclose(W.sum(1), torch.ones(n, dtype=F64), rtol=1e-12, atol=0)
        assert torch.equal(counts[-1].long(), torch.bincount(cls, minlength=D))
        assert abs(float(wmax[0]) - 1.0) <= 1e-12


# what tests/test_gpu_readout.py runs: (input dtype, P dtype, lazy prefill rescale, step keys, lengths, t values, scale)
EMULATED = [
    (torch.bfloat16, torch.bfloat16, True, 64, (17, 300, 513, 1000, 4096), ro.RAMP_T, None),     # tcgen05 prefill
    (torch.float16, torch.float16, True, 64, (17, 300, 513, 1000, 4096), ro.RAMP_T, None),
    (torch.bfloat16, torch.bfloat16, False, 16, (1, 17, 333, 1000, 4096), ro.RAMP_T, None),      # TMA decode
    (torch.float16, torch.float16, False, 16, (1, 17, 333, 1000, 4096), ro.RAMP_T, None),
    (torch.float32, torch.float32, False, 32, (7, 100, 1000), ro.RAMP_T, None),                  # SIMT prefill / decode
    (torch.float16, torch.float16, True, 64, (300, 1000), (8, 16), 2.0 ** -16),                  # big raw scores
]


@pytest.mark.parametrize("dtype,p_dtype,lazy,step,lengths,T,scale", EMULATED)
def test_emulated_kernel_rounding_stays_within_the_bound(dtype, p_dtype, lazy, step, lengths, T, scale):
    """Margin check before any GPU run: the bound must hold with room (ratio <= 0.6) for the arithmetic the kernels do."""
    D = 128 if dtype != torch.float32 else 80
    sc = D ** -0.5 if scale is None else scale
    names = ro.PROFILES if scale is None else ("bigraw",)
    worst = 0.0
    for L in lengths:
        for name in names:
            g = torch.Generator().manual_seed(L)
            s = ro.profile(name, L, g, sc, dtype if dtype != torch.float32 else torch.bfloat16)
            cls = ro.classes(L, D, g)
            t = torch.tensor(T, dtype=F64)
            o, lse = ro.emulate(s, cls, D, t, sc, dtype, p_dtype, step, lazy)
            for i, ti in enumerate(T):
                W, rl, wmax, counts = ro.prefix_reference(s, cls, D, ti * sc)
                bnd = ro.bound(W[-1], wmax[-1], counts[-1], dtype, p_dtype)
                r = ro.ratio((o[i] - W[-1]).abs(), bnd)
                rlse = ro.ratio((lse[i] - rl[-1]).abs().view(1), ro.lse_bound(rl[-1]).view(1))
                assert r <= 0.6 and rlse <= 0.6, (L, name, ti, r, rlse)
                worst = max(worst, r)
    assert worst > 0


def test_bound_rejects_the_defects_it_is_meant_to_catch():
    """At the C3 length, with a needle in the last page: a dropped last key, the last page's V read from another page,
    or one masked key let through breaks the bound by orders of magnitude (the needle sweeps put a needle at every key)."""
    g = torch.Generator().manual_seed(3)
    D, L, a = 128, 4096, 128 ** -0.5
    s = ro.profile("needle", L, g, a, torch.bfloat16, needle_at=L - 1)
    cls = ro.classes(L, D, g)
    W, _, wmax, counts = ro.prefix_reference(s, cls, D, a)
    bnd = ro.bound(W[-1], wmax[-1], counts[-1], torch.bfloat16, torch.bfloat16)
    assert ro.ratio((W[-2] - W[-1]).abs(), bnd) > 100                   # last key dropped
    cls2 = cls.clone()
    cls2[-16:] = (cls[:16] + 1) % D
    W2, _, _, _ = ro.prefix_reference(s, cls2, D, a)
    assert ro.ratio((W2[-1] - W[-1]).abs(), bnd) > 100                  # last page's V from another page
    bnd2 = ro.bound(W[-2], wmax[-2], counts[-2], torch.bfloat16, torch.bfloat16)
    assert ro.ratio((W[-1] - W[-2]).abs(), bnd2) > 100                  # the masked needle leaks into the row before it
    assert ro.ratio(torch.tensor([math.nan]), torch.tensor([1.0])) == math.inf
