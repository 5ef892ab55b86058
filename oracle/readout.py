"""Exact-logit readout probes for the attention kernels.  TEST INFRASTRUCTURE ONLY (the product package never imports it).

Random N(0, 1) inputs make the softmax nearly uniform, so |O| shrinks like 1/sqrt(L) and a fixed max-abs tolerance says
little past a few hundred keys.  The inputs built here make the kernel's output a direct readout of its attention weights
and the fp64 reference exact on the kernel's own (rounded) inputs:

  K[j, c] = beta_c * s_j        beta_c = 2^((c mod 4) - 1), s a logit profile rounded to the input dtype
  Q[r, :] = alpha_r * e_{c_r}   one-hot; alpha_r = t_r / beta_{c_r}, t_r a power of two; c_r = 7 r mod D walks every column
  V[j, :] = e_{class(j)}        class(j) in [0, D) drawn with a fixed seed per sequence

q.k = t_r * s_j exactly (one nonzero product, powers of two), so row r's logits are a_r * s_j with a_r = t_r * scale, and
O[r, d] is the total softmax weight of the visible keys of class d.  A swapped K or Q column changes the row's logit
scale; a key read from the wrong place, dropped, doubled or let through a mask moves weight between classes.

Visible keys are always a prefix [0, lim(r)) of the sequence, so one fp64 prefix scan per sequence and per row factor a
(`prefix_reference`) gives the reference of every row.

Bound (`bound`), per element, with u_P / u_out the unit roundoffs of P and of the output:
  |O - O_ref| <= 4 (u_P + u_out) O_ref + 2^-20 w_max [+ n_d 2^-24 w_max if P is fp16] [+ 2^-25 if the output is fp16]
The kernels round each P = exp2(x - m) once to the P type (RNE) while the row sum adds the unrounded fp32 P, and round
the output once: 2u in the worst case.  The 2^-20 w_max term covers fp32 sums, ex2.approx (relative error ~2^-22) and the
fp32 argument x = S * (scale log2 e) - m (scale log2 e); P <= 2^8 against a lagging maximum (prefill's lazy rescale)
leaves the relative rounding unchanged.  fp16 P below 2^-14 is subnormal: absolute error up to 2^-25 of the row's
reference maximum per key, hence the n_d term; an fp16 output below 2^-14 has absolute error up to 2^-25.  The SIMT
kernels keep P in fp32 (expf), u_P = 2^-16 there.  `emulate` replays that arithmetic on the CPU so that the bound is
checked before any GPU run (tests/test_readout_oracle.py).
LSE: |lse - ref| <= 2e-4 + 2^-20 |ref|.
"""
from __future__ import annotations

import math

import torch

F64 = torch.float64
UNIT = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11, torch.float32: 2.0 ** -24}
SIMT_UNIT_P = 2.0 ** -16
LOG2E = 1.0 / math.log(2.0)
FP16_MAX_K = 16000.0                    # |s| cap so that beta_c * s (beta <= 4) stays inside the fp16 range

# logit profiles, in nats at t = 1 (logit = t * scale * s); ramp slopes give 64-key growth of 7.5 / 4 log2 units at t = 1,
# so t in {1, 2, 4} puts one launch just below, at and well above the prefill kernel's 8-unit lazy-rescale threshold
PROFILES = ("uniform", "noise1", "noise4", "noise16", "ramp7.5", "ramp4", "sink", "needle")
RAMP_T = (1, 2, 4)


def beta(D: int) -> torch.Tensor:
    return 2.0 ** ((torch.arange(D) % 4).to(F64) - 1)


def round_to(x: torch.Tensor, dtype) -> torch.Tensor:
    """x rounded to dtype, returned as float64; fp16 values that beta_c = 0.5 would make subnormal are flushed to 0."""
    r = x.to(dtype).to(F64)
    if dtype == torch.float16:
        r = torch.where(r.abs() < 2.0 ** -12, torch.zeros_like(r), r)
    return r


def profile(name: str, n: int, gen: torch.Generator, scale: float, dtype, needle_at: int | None = None) -> torch.Tensor:
    """s (n,) float64, exactly representable in dtype (also after a beta_c scaling)."""
    nats = torch.zeros(n, dtype=F64)
    if name.startswith("noise"):
        nats = float(name[5:]) * torch.randn(n, generator=gen, dtype=F64)
    elif name.startswith("ramp"):
        nats = torch.arange(n, dtype=F64) * (float(name[4:]) / LOG2E / 64)
    elif name == "sink":
        nats = torch.randn(n, generator=gen, dtype=F64)
        nats[min(2, n - 1)] = 40.0
    elif name == "needle":
        nats[n // 3 if needle_at is None else needle_at] = 30.0
    elif name == "bigraw":            # fp16 raw scores q.k up to ~2.5e5 with scale 2^-16: moderate logits, 16-bit S would overflow
        return round_to((torch.rand(n, generator=gen, dtype=F64) * 2 - 1) * FP16_MAX_K, dtype)
    elif name != "uniform":
        raise ValueError(name)
    s = nats / scale
    if dtype == torch.float16 and s.abs().max() > FP16_MAX_K:
        raise ValueError(f"profile {name} over {n} keys leaves the fp16 range")
    return round_to(s, dtype)


def classes(n: int, D: int, gen: torch.Generator) -> torch.Tensor:
    return torch.randint(0, D, (n,), generator=gen)


def make_kv(s: torch.Tensor, cls: torch.Tensor, D: int, dtype):
    """K, V (n, D) in dtype (CPU) for one (sequence, kv head)."""
    k64 = s[:, None] * beta(D)[None, :]
    k = k64.to(dtype)
    assert torch.equal(k.to(F64), k64), "profile not exact in the input dtype"
    v = torch.nn.functional.one_hot(cls, D).to(dtype)
    return k, v


def make_q(idx: torch.Tensor, D: int, T, dtype):
    """One-hot query rows for flat row indices idx (any shape, on any device): q (..., D) in dtype and t (...) float64."""
    c = (idx * 7) % D
    t = torch.tensor(T, dtype=F64, device=idx.device)[(idx + idx // D) % len(T)]
    alpha = t / beta(D).to(idx.device)[c]
    a16 = alpha.to(dtype)
    assert torch.equal(a16.to(F64), alpha), "alpha not exact in the input dtype"
    q = torch.zeros(*idx.shape, D, dtype=dtype, device=idx.device)
    q.scatter_(-1, c.unsqueeze(-1), a16.unsqueeze(-1))
    return q, t


def prefix_reference(s: torch.Tensor, cls: torch.Tensor, D: int, a: float, block: int = 16):
    """Attention of a one-hot-query row with logits a * s over every prefix of the keys, in fp64.

    Returns W (n, D) with W[p - 1, d] = total softmax weight of class d among keys [0, p), lse (n,), wmax (n,) (the
    largest single weight of the prefix) and counts (n, D) int32 (keys of class d in the prefix).  A blockwise scan with
    a running maximum: exact for logit spreads of thousands of nats as long as one block spans less than 650 nats."""
    n = s.numel()
    x = a * s.to(F64)
    nb = (n + block - 1) // block
    xp = torch.full((nb * block,), -math.inf, dtype=F64)
    xp[:n] = x
    xb = xp.view(nb, block)
    mb = xb.max(1).values
    spread = mb - torch.where(torch.isinf(xb), mb[:, None], xb).min(1).values
    if float(spread.max()) > 650.0:
        raise ValueError(f"a {block}-key block spans more than 650 nats: the in-block scan would underflow")
    e = torch.exp(xb - mb[:, None])
    cp = torch.zeros(nb * block, dtype=torch.long)
    cp[:n] = cls
    E = torch.zeros(nb, block, D, dtype=F64)
    E.scatter_(2, cp.view(nb, block, 1), e.unsqueeze(2))
    C = E.cumsum(1)                                  # in-block prefix sums, reference mb
    Ls = e.cumsum(1)
    tot_o, tot_l = C[:, -1], Ls[:, -1]
    # exclusive scan over blocks: state before block b, reference M_prev[b]
    M_prev = torch.full((nb,), -math.inf, dtype=F64)
    L_prev = torch.zeros(nb, dtype=F64)
    O_prev = torch.zeros(nb, D, dtype=F64)
    m, l, o = -math.inf, 0.0, torch.zeros(D, dtype=F64)
    for b in range(nb):
        M_prev[b], L_prev[b], O_prev[b] = m, l, o
        mn = max(m, float(mb[b]))
        f_old = math.exp(m - mn) if m != -math.inf else 0.0
        f_new = math.exp(float(mb[b]) - mn)
        l = l * f_old + float(tot_l[b]) * f_new
        o = o * f_old + tot_o[b] * f_new
        m = mn
    M = torch.maximum(M_prev, mb)
    f_old = torch.where(torch.isinf(M_prev), torch.zeros_like(M), torch.exp(M_prev - M))
    f_new = torch.exp(mb - M)
    lt = L_prev[:, None] * f_old[:, None] + Ls * f_new[:, None]
    W = (O_prev[:, None, :] * f_old[:, None, None] + C * f_new[:, None, None]) / lt[:, :, None]
    lse = (M[:, None] + torch.log(lt)).reshape(-1)[:n]
    W = W.reshape(-1, D)[:n]
    assert torch.isfinite(W).all() and torch.isfinite(lse).all()
    wmax = torch.exp(torch.cummax(x, 0).values - lse)
    counts = torch.nn.functional.one_hot(cls, D).to(torch.int32).cumsum(0, dtype=torch.int32)
    return W, lse, wmax, counts


def bound(o_ref: torch.Tensor, wmax: torch.Tensor, counts: torch.Tensor, out_dtype, p_dtype) -> torch.Tensor:
    """Per-element bound on |O - O_ref| (see the module docstring); wmax broadcasts against o_ref's last dimension."""
    u_p = UNIT[p_dtype] if p_dtype != torch.float32 else SIMT_UNIT_P
    w = wmax.unsqueeze(-1)
    b = 4 * (u_p + UNIT[out_dtype]) * o_ref + 2.0 ** -20 * w
    if p_dtype == torch.float16:
        b = b + counts.to(F64) * 2.0 ** -24 * w
    if out_dtype == torch.float16:
        b = b + 2.0 ** -25
    return b


def lse_bound(ref: torch.Tensor) -> torch.Tensor:
    return 2e-4 + 2.0 ** -20 * ref.abs()


def ratio(err: torch.Tensor, bnd: torch.Tensor) -> float:
    """Worst err / bound; NaN (a NaN error) counts as a failure of any bound, so it is returned as inf."""
    r = err / bnd
    if torch.isnan(r).any():
        return math.inf
    return float(r.max()) if r.numel() else 0.0


def _f32(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float32).to(F64)


def emulate(s: torch.Tensor, cls: torch.Tensor, D: int, t: torch.Tensor, scale: float, dtype, p_dtype,
            step: int, lazy: bool):
    """The kernels' arithmetic for rows with scale factors t over all n keys: S = t s (exact in fp32), per step of `step`
    keys the row maximum, x = fma(S, c, -m c) in fp32 with c = fp32(scale log2 e), P = exp2(x) in fp32 (0 below 2^-126:
    ex2.approx.ftz), the fp32 row sum of P, P rounded RNE to p_dtype into fp32 class sums, and the output O / d rounded
    to dtype.  lazy=True is prefill's lazy rescale: the reference maximum moves only when it grew by more than 8 log2
    units, so P reaches 2^8.  Returns o (R, D) float64 and lse (R,)."""
    c = float(torch.tensor(scale, dtype=torch.float32) * torch.tensor(LOG2E, dtype=torch.float32))
    S = _f32(t[:, None] * s[None, :])
    R, n = S.shape
    m_ref = torch.full((R,), -math.inf, dtype=F64)
    d = torch.zeros(R, dtype=torch.float32)
    O = torch.zeros(R, D, dtype=torch.float32)
    for k0 in range(0, n, step):
        Sb = S[:, k0:k0 + step]
        m_new = torch.maximum(Sb.max(1).values, m_ref)
        if k0 == 0:
            m_ref = m_new
        else:
            move = (_f32((m_new - m_ref) * c) > 8.0) if lazy else (m_new > m_ref)
            alpha = torch.where(move, _f32(torch.exp2(_f32(m_ref * c) - _f32(m_new * c))), torch.ones_like(m_ref))
            d = (d.to(F64) * alpha).to(torch.float32)
            O = (O.to(F64) * alpha[:, None]).to(torch.float32)
            m_ref = torch.where(move, m_new, m_ref)
        nmc = _f32(-m_ref * c)
        x = _f32(Sb * c + nmc[:, None])
        p = _f32(torch.exp2(x))
        p = torch.where(p < 2.0 ** -126, torch.zeros_like(p), p)
        d = (d.to(F64) + p.sum(1)).to(torch.float32)
        pr = p.to(p_dtype).to(F64) if p_dtype != torch.float32 else p
        add = torch.zeros(R, D, dtype=F64).index_add_(1, cls[k0:k0 + step], pr)
        O = (O.to(F64) + add).to(torch.float32)
    o = (O.to(F64) / d.to(F64)[:, None]).to(torch.float32).to(dtype).to(F64)
    lse = (m_ref * c + torch.log2(d.to(F64))) / LOG2E
    return o, lse
