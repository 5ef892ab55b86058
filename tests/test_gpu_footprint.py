"""Footprint tests: every C-ABI entry point writes exactly its declared outputs and nothing else.

Each pointer argument of a call gets its own uint8 buffer, an *arena*:

    [ front guard | region (the tensor, with the gaps its padded strides leave) | back guard ]

Guards are 256 KiB (more than any TMA box or vector overrun of these kernels) and hold pattern A (0xA5).  The gaps of an
output hold pattern A as well; the gaps of an input hold 0xFF, a NaN in every float type, so a read of a gap changes the
result.  Every element an output declares it writes starts as a sentinel NaN no kernel produces (pattern B).  After the
call and one synchronise, each case asserts
  (a) nothing outside: every guard and gap byte of every argument is bit-identical to before;
  (b) nothing missed: no element of the write set still holds the sentinel;
  (c) inputs untouched: every input arena (data, gaps and guards) is bitwise unchanged;
  (d) same values: the outputs equal, bit for bit, those of the same call on dense tensors, served by the same kernel kind.
A failure names the first offending byte as (argument, front guard / gap / back guard / element index).

`Arg` works on any device: tests/test_footprint_harness.py checks on the CPU that it reports what it should.
"""
import ctypes
import math

import numpy as np
import pytest
import torch

from physics_llm_inference_b200 import _lib

GUARD = 256 * 1024               # bytes on each side of a region
ALIGN = 256                      # region size granule (regions start 256-byte aligned)
PAT_A = 0xA5                     # guards, output gaps, workspace
PAT_IN_GAP = 0xFF                # input gaps: NaN in bf16, f16 and f32
# pattern B: NaNs with a payload no kernel produces (kernels emit 0x7FC0 / 0x7FFF / 0x7FC00000 / 0x7FFFFFFF NaNs);
# bf16 needs 0x7FDA, as 0x7E5A is a finite bf16 number
SENTINEL = {torch.bfloat16: 0x7FDA, torch.float16: 0x7E5A, torch.float32: 0x7FA5A5A5}
INT_OF = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}
CODE = {torch.bfloat16: _lib.PLI_BF16, torch.float16: _lib.PLI_F16, torch.float32: _lib.PLI_F32}
INT32_MAX = 2 ** 31 - 1


def padded_strides(shape, pad=None, order=None):
    """Element strides of `shape` laid out in `order` (dimensions outermost first, default: as given), where pad[d]
    extra elements follow every step along dimension d (0 for the innermost dimension)."""
    n = len(shape)
    pad = pad or [0] * n
    order = list(range(n)) if order is None else list(order)
    st, run = [0] * n, 1
    for d in reversed(order):
        st[d] = run + pad[d]
        run = st[d] * shape[d]
    return st


def _signed(x, bits):
    return x - (1 << bits) if x >= 1 << (bits - 1) else x


class Arg:
    """One pointer argument of a call inside its own arena.

    role: "in"    read-only: the whole arena must come back bit-identical;
          "out"   every element (or `wset` of them) is written: starts as pattern B, nothing else may change;
          "inout" holds data; the elements of `wset` start as pattern B and must be written, nothing else may change;
          "ws"    scratch (a workspace): its elements may change, its gaps and guards may not."""

    def __init__(self, name, shape, dtype, role, device="cuda", pad=None, order=None, strides=None):
        assert role in ("in", "out", "inout", "ws")
        self.name, self.shape, self.dtype, self.role = name, tuple(shape), dtype, role
        self.esz = torch.empty((), dtype=dtype).element_size()
        self.strides = tuple(padded_strides(shape, pad, order) if strides is None else strides)
        span = 1 + sum((n - 1) * s for n, s in zip(self.shape, self.strides)) if all(self.shape) else 0
        self.region = -(-span * self.esz // ALIGN) * ALIGN
        self.buf = torch.full((2 * GUARD + self.region,), PAT_A, dtype=torch.uint8, device=device)
        if role in ("in", "inout"):
            self.buf[GUARD:GUARD + self.region] = PAT_IN_GAP
        self.t = self.buf.view(dtype).as_strided(self.shape, self.strides, GUARD // self.esz)
        self.wset, self.snap = None, None

    @classmethod
    def of(cls, name, src, role="in", **kw):
        """An arena holding a copy of `src`."""
        a = cls(name, src.shape, src.dtype, role, device=src.device, **kw)
        a.t.copy_(src)
        return a

    @property
    def ptr(self):
        return self.t.data_ptr()

    def bits(self):
        return self.t.view(INT_OF[self.esz])

    def arm(self, wset=None):
        """Fill the write set with pattern B and take the snapshot the checks compare against."""
        self.wset = wset
        if self.role in ("out", "inout"):
            s = _signed(SENTINEL[self.dtype], 8 * self.esz)
            if wset is None:
                self.bits().fill_(s)
            else:
                self.bits()[wset] = s
        self.snap = self.buf.clone()
        return self

    def _byte_mask(self, which):
        m = torch.zeros(self.region // self.esz, dtype=INT_OF[self.esz], device=self.buf.device)
        v = m.as_strided(self.shape, self.strides)
        if which is None:
            v.fill_(-1)
        else:
            v[which] = -1
        return m.view(torch.uint8) != 0

    def index_of(self, e):
        """Index of the element stored at storage element e of the region, or None for a gap."""
        m = torch.full((self.region // self.esz,), -1, dtype=torch.int64, device=self.buf.device)
        n = math.prod(self.shape)
        m.as_strided(self.shape, self.strides).copy_(torch.arange(n, device=m.device).view(self.shape))
        flat = int(m[e])
        return None if flat < 0 else tuple(int(i) for i in np.unravel_index(flat, self.shape))

    def where(self, o):
        """Byte offset o of the arena as (argument, front guard / gap / back guard / element index)."""
        if o < GUARD:
            return f"{self.name}: front guard, byte {o - GUARD}"
        r = o - GUARD
        if r >= self.region:
            return f"{self.name}: back guard, byte {r - self.region}"
        idx = self.index_of(r // self.esz)
        if idx is None:
            return f"{self.name}: gap, region byte {r}"
        return f"{self.name}: element {idx}"

    def check(self):
        """Failures of (a), (b) and, for inputs, (c), as text."""
        assert self.snap is not None, f"{self.name}: arm() was not called"
        errs = []
        bad = self.buf != self.snap
        if self.role != "in":
            allowed = self._byte_mask(self.wset if self.role in ("out", "inout") else None)
            bad[GUARD:GUARD + self.region] &= ~allowed
        if bool(bad.any()):
            o = int(torch.nonzero(bad)[0])
            what = "input modified" if self.role == "in" else "store outside the write set"
            errs.append(f"{self.where(o)}: {what} (0x{int(self.snap[o]):02x} -> 0x{int(self.buf[o]):02x}; "
                        f"{int(bad.sum())} bytes in all)")
        if self.role in ("out", "inout"):
            left = self.bits() == _signed(SENTINEL[self.dtype], 8 * self.esz)
            if self.wset is not None:
                left &= self.wset
            if bool(left.any()):
                idx = tuple(int(i) for i in torch.nonzero(left)[0])
                errs.append(f"{self.name}: element {idx} of the write set was never written "
                            f"({int(left.sum())} elements in all)")
        return errs


def verify(*args):
    """(a)-(c) over every argument of a call."""
    if any(a.buf.is_cuda for a in args):
        torch.cuda.synchronize()
    errs = [e for a in args for e in a.check()]
    assert not errs, "\n".join(errs)


def same_bits(a, b, what=""):
    """(d): bit-identical values (NaN-safe)."""
    ia, ib = a.view(INT_OF[a.element_size()]), b.view(INT_OF[b.element_size()])
    if not torch.equal(ia, ib):
        n = int((ia != ib).sum())
        i = tuple(int(x) for x in torch.nonzero(ia != ib)[0])
        raise AssertionError(f"{what}: {n} elements differ from the dense call, first at {i}: {a[i]} vs {b[i]}")


# ---------------------------------------------------------------------------------------------------------------------
# GPU cases
# ---------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _rand(shape, dtype, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(shape, generator=g, device="cuda") * scale).to(dtype)


def _fresh(shape, dtype=torch.float32):
    """A dense output of the reference call, also inside guards (its contents are not checked)."""
    return Arg("dense", shape, dtype, "ws").t


def _ptr(t):
    return None if t is None else t.data_ptr()


def _i64(t, n):
    return _lib.i64(*t.stride()[:n])


# ---- prefill, contiguous K/V ----------------------------------------------------------------------------------------
def _prefill_call(q, k, v, o, lse, Hkv, Nk, scale, causal):
    B, Hq, Nq, D = q.shape
    lib = _lib.load()
    kind = lib.pli_prefill_kernel_kind(D, CODE[q.dtype], _i64(q, 3), _i64(k, 3), _i64(v, 3), _i64(o, 3), q.data_ptr(),
                                       k.data_ptr(), v.data_ptr(), o.data_ptr())
    _lib.check(lib.pli_prefill_fwd(q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr(), _ptr(lse), B, Hq, Hkv, Nq,
                                   Nk, D, _i64(q, 3), _i64(k, 3), _i64(v, 3), _i64(o, 3), scale, int(causal),
                                   CODE[q.dtype], _stream()))
    # pli_prefill_kernel_kind does not see the scale: pli_prefill_fwd serves scale <= 0 with the SIMT kernel
    return kind if scale > 0 else _lib.PLI_KIND_SIMT


def _prefill_case(B, Hq, Hkv, Nq, Nk, D, dtype, causal, o_order, with_lse, pads, scale=None, seed=0, kind=None,
                  kv_strides=None):
    """pads: (q pad, o pad, k/v pad) per dimension of (B, H, N, D).  kv_strides: explicit K/V strides (broadcasts)."""
    scale = D ** -0.5 if scale is None else scale
    q = _rand((B, Hq, Nq, D), dtype, seed)
    k = _rand((B, Hkv, Nk, D), dtype, seed + 1)
    v = _rand((B, Hkv, Nk, D), dtype, seed + 2)
    if kv_strides is not None:                            # one K/V row set read through zero strides
        k, v = k[:1, :1].expand(B, Hkv, Nk, D), v[:1, :1].expand(B, Hkv, Nk, D)
    qp, op, kp = pads
    o_ref = _fresh((B, Hq, Nq, D), dtype)
    lse_ref = _fresh((B, Hq, Nq)) if with_lse else None
    kind_ref = _prefill_call(q, k.contiguous() if kv_strides is None else k, v.contiguous() if kv_strides is None else v,
                             o_ref, lse_ref, Hkv, Nk, scale, causal)
    aq = Arg.of("q", q, pad=qp)
    if kv_strides is None:
        ak, av = Arg.of("k", k, pad=kp), Arg.of("v", v, pad=kp)
    else:
        ak = Arg("k", k.shape, dtype, "in", strides=kv_strides)
        av = Arg("v", v.shape, dtype, "in", strides=kv_strides)
        ak.t[0, 0].copy_(k[0, 0])
        av.t[0, 0].copy_(v[0, 0])
    ao = Arg("o", (B, Hq, Nq, D), dtype, "out", pad=op, order=o_order)
    al = Arg("lse", (B, Hq, Nq), torch.float32, "out") if with_lse else None
    args = [a for a in (aq, ak, av, ao, al) if a is not None]
    for a in args:
        a.arm()
    kind_a = _prefill_call(aq.t, ak.t, av.t, ao.t, al.t if al else None, Hkv, Nk, scale, causal)
    verify(*args)
    assert kind_a == kind_ref, (_lib.KIND_NAMES[kind_a], _lib.KIND_NAMES[kind_ref])
    if kind is not None:
        assert _lib.KIND_NAMES[kind_a] == kind
    same_bits(ao.t, o_ref, "o")
    if with_lse:
        same_bits(al.t, lse_ref, "lse")


BHND, BNHD = (0, 1, 2, 3), (0, 2, 1, 3)
P8 = ([64, 16, 8, 0], [128, 24, 16, 0], [0, 8, 8, 0])      # q / o / kv pads: multiples of 8 keep tcgen05 eligible


@gpu
@pytest.mark.parametrize("B,Hq,Hkv,Nq,Nk,D,dtype,causal,order,lse", [
    (2, 4, 4, 77, 77, 64, torch.bfloat16, True, BHND, True),          # G 1: row-pair items
    (1, 6, 2, 300, 300, 128, torch.float16, False, BNHD, True),       # G 3
    (2, 4, 2, 513, 513, 128, torch.bfloat16, True, BNHD, False),      # G 2: head pairs, no LSE
    (1, 8, 2, 300, 700, 128, torch.bfloat16, True, BHND, True),       # G 4: CTA pairs, pair MMA; Nq < Nk
    (2, 8, 2, 513, 513, 64, torch.float16, True, BNHD, True),         # G 4, D 64
    (1, 8, 1, 1, 33, 64, torch.float16, True, BHND, True),            # G 8, one query row
    (2, 16, 2, 77, 300, 128, torch.float16, False, BHND, False),      # G 8, D 128
    (1, 3, 1, 129, 129, 64, torch.bfloat16, False, BNHD, True),       # G 3, D 64
    (3, 6, 3, 513, 513, 128, torch.bfloat16, True, BHND, True),       # 5 slots in blocks of 4: short last block
    (1, 6, 3, 513, 513, 128, torch.bfloat16, True, BNHD, True),
])
def test_prefill_tcgen05(B, Hq, Hkv, Nq, Nk, D, dtype, causal, order, lse):
    _prefill_case(B, Hq, Hkv, Nq, Nk, D, dtype, causal, order, lse, P8, seed=B + Hq + Nq, kind="tcgen05")


@gpu
def test_prefill_tcgen05_many_items():
    """B16 x 32 q / 8 kv heads x N 2048: more than 16 x 148 items, so the scheduling block doubles and the schedule runs
    several rounds."""
    _prefill_case(16, 32, 8, 2048, 2048, 64, torch.bfloat16, True, BHND, True, P8, seed=5, kind="tcgen05")


@gpu
@pytest.mark.parametrize("D,causal,pads", [
    (48, True, ([3, 1, 1, 0], [5, 3, 1, 0], [0, 1, 3, 0])),
    (80, False, ([0, 0, 3, 0], [1, 1, 3, 0], [7, 3, 1, 0])),
])
def test_prefill_simt_fp32(D, causal, pads):
    _prefill_case(2, 4, 2, 70, 100, D, torch.float32, causal, BHND, True, pads, seed=D, kind="simt")


@gpu
def test_prefill_simt_negative_scale_and_zero_strides():
    _prefill_case(1, 4, 2, 200, 200, 128, torch.bfloat16, True, BNHD, True, ([0, 1, 3, 0], [0, 3, 1, 0], [0, 8, 8, 0]),
                  scale=-(128 ** -0.5), seed=3, kind="simt")
    N, D = 150, 128
    _prefill_case(3, 4, 4, N, N, D, torch.bfloat16, True, BHND, True, ([0, 8, 8, 0], [0, 1, 3, 0], None), seed=4,
                  kind="simt", kv_strides=(0, 0, D + 3, 1))


@gpu
def test_prefill_simt_reads_nothing_past_nk():
    """Poison around the rows a SIMT prefill reads: K/V of Nk + 40 tokens with NaN K / Inf V past Nk, and NaN in the
    head-dim gaps (+3 elements per token).  The result must be bit-identical to dense K/V of Nk tokens."""
    B, Hq, Hkv, Nq, Nk, D = 2, 4, 2, 50, 90, 48
    q = _rand((B, Hq, Nq, D), torch.float32, 7)
    k, v = _rand((B, Hkv, Nk, D), torch.float32, 8), _rand((B, Hkv, Nk, D), torch.float32, 9)
    o_ref, lse_ref = _fresh(q.shape, q.dtype), _fresh((B, Hq, Nq))
    _prefill_call(q, k, v, o_ref, lse_ref, Hkv, Nk, D ** -0.5, True)
    big = (B, Hkv, Nk + 40, D)
    ak, av = Arg("k", big, torch.float32, "in", pad=[0, 0, 3, 0]), Arg("v", big, torch.float32, "in", pad=[0, 0, 3, 0])
    ak.t.fill_(float("nan"))
    av.t.fill_(float("inf"))
    ak.t[:, :, :Nk] = k
    av.t[:, :, :Nk] = v
    aq, ao = Arg.of("q", q), Arg("o", q.shape, torch.float32, "out")
    al = Arg("lse", (B, Hq, Nq), torch.float32, "out")
    for a in (aq, ak, av, ao, al):
        a.arm()
    assert _prefill_call(aq.t, ak.t[:, :, :Nk], av.t[:, :, :Nk], ao.t, al.t, Hkv, Nk, D ** -0.5, True) == \
        _lib.PLI_KIND_SIMT
    verify(aq, ak, av, ao, al)
    same_bits(ao.t, o_ref, "o")
    same_bits(al.t, lse_ref, "lse")


# ---- paged pools ----------------------------------------------------------------------------------------------------
class Pools:
    """Paged K/V pools (P, layers, bs, Hkv, D) with the pages of each sequence in a seeded random order; the table has
    one column more than the longest sequence needs, its padding holds `fill`."""

    def __init__(self, lens, bs, Hkv, D, dtype, seed, layers=2, layer=1, extra_pages=3, fill=0):
        g = torch.Generator().manual_seed(seed)
        self.lens, self.bs, self.layer = list(lens), bs, layer
        self.npg = [max(1, -(-L // bs)) for L in lens]
        self.P = sum(self.npg) + extra_pages
        perm = torch.randperm(self.P, generator=g).to(torch.int32)
        self.table = torch.full((len(lens), max(self.npg) + 1), fill, dtype=torch.int32)
        at = 0
        for b, n in enumerate(self.npg):
            self.table[b, :n] = perm[at:at + n]
            at += n
        self.spare = perm[at:]                                       # pages no sequence uses
        self.table = self.table.cuda()
        self.k = _rand((self.P, layers, bs, Hkv, D), dtype, seed + 11)
        self.v = _rand((self.P, layers, bs, Hkv, D), dtype, seed + 12)
        self.lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")

    def poison_page(self):
        """A spare page of NaN K / Inf V; returns its id."""
        p = int(self.spare[0])
        self.k[p] = float("nan")
        self.v[p] = float("inf")
        return p

    def hostile(self, value):
        """The table with every entry past each sequence's last page set to `value`."""
        t = self.table.clone()
        for b, n in enumerate(self.npg):
            t[b, n:] = value
        return t


def _paged_call(q, kp, vp, table, lens, o, lse, Hkv, max_len, bs, layer, cu=None, max_q=None):
    lib = _lib.load()
    D = q.shape[-1]
    if cu is None:
        B, Hq, Nq, _ = q.shape
        _lib.check(lib.pli_prefill_paged_fwd(q.data_ptr(), kp.data_ptr(), vp.data_ptr(), table.data_ptr(), lens.data_ptr(),
                                             o.data_ptr(), _ptr(lse), B, Hq, Hkv, Nq, D, max_len, bs, table.stride(0),
                                             layer, kp.shape[0], _i64(q, 3), _i64(kp, 4), _i64(o, 3), D ** -0.5,
                                             CODE[q.dtype], _stream()))
    else:
        T, Hq, _ = q.shape
        _lib.check(lib.pli_prefill_varlen_paged_fwd(q.data_ptr(), kp.data_ptr(), vp.data_ptr(), table.data_ptr(),
                                                    lens.data_ptr(), cu.data_ptr(), o.data_ptr(), _ptr(lse), len(lens),
                                                    Hq, Hkv, T, max_q, D, max_len, bs, table.stride(0), layer,
                                                    kp.shape[0], _i64(q, 2), _i64(kp, 4), _i64(o, 2), D ** -0.5,
                                                    CODE[q.dtype], _stream()))


def _paged_prefill_case(bs, D, Hkv, G, Nq, lens, dtype, seed, table=None, pools=None):
    B, Hq = len(lens), Hkv * G
    pl = pools or Pools(lens, bs, Hkv, D, dtype, seed)
    q = _rand((B, Hq, Nq, D), dtype, seed)
    o_ref, lse_ref = _fresh((B, Hq, Nq, D), dtype), _fresh((B, Hq, Nq))
    _paged_call(q, pl.k, pl.v, pl.table, pl.lens_t, o_ref, lse_ref, Hkv, max(lens), bs, pl.layer)
    aq, ak, av = Arg.of("q", q, pad=[32, 8, 8, 0]), Arg.of("k_pool", pl.k), Arg.of("v_pool", pl.v)
    at = Arg.of("block_table", pl.table if table is None else table)
    asl = Arg.of("seq_lens", pl.lens_t)
    ao = Arg("o", q.shape, dtype, "out", pad=[40, 16, 8, 0])
    al = Arg("lse", (B, Hq, Nq), torch.float32, "out")
    args = (aq, ak, av, at, asl, ao, al)
    for a in args:
        a.arm()
    _paged_call(aq.t, ak.t, av.t, at.t, asl.t, ao.t, al.t, Hkv, max(lens), bs, pl.layer)
    verify(*args)
    same_bits(ao.t, o_ref, "o")
    same_bits(al.t, lse_ref, "lse")
    for b, L in enumerate(lens):                              # rows that see no key: O = 0, LSE = -inf
        if L < Nq:
            assert torch.count_nonzero(ao.t[b, :, :Nq - L].float()) == 0
            assert bool(torch.isneginf(al.t[b, :, :Nq - L]).all())


@gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("bs,D,Hkv,G,Nq,lens", [
    (16, 128, 2, 4, 77, [300, 77, 129]),          # CTA pairs
    (32, 128, 1, 2, 100, [333, 100]),             # head pairs
    (64, 64, 2, 1, 96, [1000, 97]),               # row pairs
    (128, 128, 1, 3, 50, [130, 20]),              # G 3; sequence 1 has 30 rows that see no key
    (16, 64, 1, 8, 33, [33, 500]),
])
def test_paged_prefill(bs, D, Hkv, G, Nq, lens, dtype):
    _paged_prefill_case(bs, D, Hkv, G, Nq, lens, dtype, seed=bs + D + G)


def _varlen_case(bs, D, Hkv, G, q_lens, lens, dtype, seed, table=None, pools=None):
    B, Hq, T = len(lens), Hkv * G, sum(q_lens)
    pl = pools or Pools(lens, bs, Hkv, D, dtype, seed)
    q = _rand((T, Hq, D), dtype, seed)
    cu = torch.tensor([0] + q_lens, dtype=torch.int32).cumsum(0, dtype=torch.int32).cuda()
    o_ref, lse_ref = _fresh((T, Hq, D), dtype), _fresh((Hq, T))
    _paged_call(q, pl.k, pl.v, pl.table, pl.lens_t, o_ref, lse_ref, Hkv, max(lens), bs, pl.layer, cu, max(q_lens))
    aq, ak, av = Arg.of("q", q, pad=[16, 8, 0]), Arg.of("k_pool", pl.k), Arg.of("v_pool", pl.v)
    at, asl, acu = Arg.of("block_table", pl.table if table is None else table), Arg.of("seq_lens", pl.lens_t), \
        Arg.of("cu_seqlens_q", cu)
    ao = Arg("o", q.shape, dtype, "out", pad=[24, 8, 0])
    al = Arg("lse", (Hq, T), torch.float32, "out")
    args = (aq, ak, av, at, asl, acu, ao, al)
    for a in args:
        a.arm()
    _paged_call(aq.t, ak.t, av.t, at.t, asl.t, ao.t, al.t, Hkv, max(lens), bs, pl.layer, acu.t, max(q_lens))
    verify(*args)
    same_bits(ao.t, o_ref, "o")
    same_bits(al.t, lse_ref, "lse")


@gpu
@pytest.mark.parametrize("bs,D,Hkv,G,q_lens,lens", [
    (16, 128, 2, 4, [130, 0, 1, 77], [300, 5, 1, 77]),       # an empty sequence between two non-empty ones
    (64, 64, 1, 2, [1, 200, 0, 129], [64, 200, 10, 500]),
    (32, 128, 1, 3, [37, 1], [37, 300]),
    (128, 128, 2, 1, [255, 3], [255, 1000]),
])
def test_varlen_paged_prefill(bs, D, Hkv, G, q_lens, lens):
    _varlen_case(bs, D, Hkv, G, q_lens, lens, torch.bfloat16, seed=bs + G)


# ---- decode ---------------------------------------------------------------------------------------------------------
def _decode_call(q, k, v, table, lens, o, lse, Hkv, max_len, bs, layer, ws, splits, scale=None, q_len=1):
    """pli_decode_fwd (q (B, Hq, D)) or pli_decode_fwd_multi (q (B, Hq, q_len, D)); returns the decode kernel kind."""
    lib = _lib.load()
    D = q.shape[-1]
    B, Hq = q.shape[:2]
    scale = D ** -0.5 if scale is None else scale
    paged = table is not None
    kvs = k.stride()[:4] if paged else (k.stride(0), 0, k.stride(1), k.stride(2))
    common = (k.data_ptr(), v.data_ptr(), _ptr(table), lens.data_ptr(), o.data_ptr(), _ptr(lse))
    tail = (bs if paged else 0, table.stride(0) if paged else 0, layer, k.shape[0])
    wsb = ws.shape[0]
    if q_len == 1:
        _lib.check(lib.pli_decode_fwd(q.data_ptr(), *common, B, Hq, Hkv, D, max_len, *tail, _i64(q, 2), _lib.i64(*kvs),
                                      _i64(o, 2), scale, CODE[q.dtype], splits, ws.data_ptr(), wsb, _stream()))
    else:
        _lib.check(lib.pli_decode_fwd_multi(q.data_ptr(), *common, B, Hq, Hkv, q_len, D, max_len, *tail, _i64(q, 3),
                                            _lib.i64(*kvs), _i64(o, 3), scale, CODE[q.dtype], splits, ws.data_ptr(),
                                            wsb, _stream()))
    return lib.pli_decode_kernel_kind(D, CODE[q.dtype], bs if paged else 0, _lib.i64(*kvs), k.data_ptr(), v.data_ptr())


def _ws_bytes(B, Hv, D, splits):
    return int(_lib.load().pli_decode_workspace_bytes(B, Hv, D, splits))


class DecodeInputs:
    """q, K/V storage (paged pools, or the contiguous (B, cap, Hkv, D) cache when bs == 0), lengths."""

    def __init__(self, dtype, D, bs, G, Hkv, lens, seed, q_len=1):
        self.B, self.Hq, self.Hkv, self.D, self.bs, self.lens = len(lens), Hkv * G, Hkv, D, bs, list(lens)
        self.q_len, self.dtype = q_len, dtype
        shape = (self.B, self.Hq, q_len, D) if q_len > 1 else (self.B, self.Hq, D)
        self.q = _rand(shape, dtype, seed)
        self.lens_t = torch.tensor(lens, dtype=torch.int32, device="cuda")
        if bs:
            self.pools = Pools(lens, bs, Hkv, D, dtype, seed)
            self.k, self.v, self.table, self.layer = self.pools.k, self.pools.v, self.pools.table, self.pools.layer
        else:
            self.pools, self.table, self.layer = None, None, 0
            cap = max(lens) + 5
            self.k, self.v = _rand((self.B, cap, Hkv, D), dtype, seed + 1), _rand((self.B, cap, Hkv, D), dtype, seed + 2)
        self.max_len = max(max(lens), 1)

    def out_shape(self):
        return self.q.shape

    def lse_shape(self):
        return self.q.shape[:-1]

    def dense(self, splits, k=None, v=None, table=None):
        o, lse = _fresh(self.q.shape, self.dtype), _fresh(self.lse_shape())
        ws = _fresh((_ws_bytes(self.B, self.Hq * self.q_len, self.D, splits),), torch.uint8)
        kind = _decode_call(self.q, self.k if k is None else k, self.v if v is None else v,
                            self.table if table is None else table, self.lens_t, o, lse, self.Hkv, self.max_len, self.bs,
                            self.layer, ws, splits, q_len=self.q_len)
        return o, lse, kind


def _o_pads(di, odd):
    """Padded output strides: {batch, head} for one token; {batch, token} for q_len > 1 (head stride = q_len x token)."""
    if di.q_len > 1:
        return [24, 0, 1 if odd else 8, 0]
    return [3, 1, 0] if odd else [40, 8, 0]


def _decode_case(di, splits, odd=False, hostile=None):
    o_ref, lse_ref, kind_ref = di.dense(splits)
    table = di.table
    if hostile is not None:
        table = di.pools.hostile(di.pools.poison_page() if hostile == "poison" else INT32_MAX)
        di.k, di.v = di.pools.k, di.pools.v                       # (the poisoned spare page is read by no sequence)
    aq = Arg.of("q", di.q, pad=([1, 3, 0] if di.q_len == 1 else [1, 3, 1, 0]) if odd else
                ([16, 8, 0] if di.q_len == 1 else [16, 8, 8, 0]))
    ak, av, asl = Arg.of("k", di.k), Arg.of("v", di.v), Arg.of("seq_lens", di.lens_t)
    at = Arg.of("block_table", table) if table is not None else None
    if di.q_len > 1:
        st = padded_strides(di.out_shape(), _o_pads(di, odd))
        st[1] = di.q_len * st[2]
        ao = Arg("o", di.out_shape(), di.dtype, "out", strides=st)
    else:
        ao = Arg("o", di.out_shape(), di.dtype, "out", pad=_o_pads(di, odd))
    al = Arg("lse", di.lse_shape(), torch.float32, "out")
    aw = Arg("workspace", (_ws_bytes(di.B, di.Hq * di.q_len, di.D, splits),), torch.uint8, "ws")
    args = [a for a in (aq, ak, av, at, asl, ao, al, aw) if a is not None]
    for a in args:
        a.arm()
    kind = _decode_call(aq.t, ak.t, av.t, at.t if at else None, asl.t, ao.t, al.t, di.Hkv, di.max_len, di.bs, di.layer,
                        aw.t, splits, q_len=di.q_len)
    verify(*args)
    assert kind == kind_ref
    same_bits(ao.t, o_ref, "o")
    same_bits(al.t, lse_ref, "lse")
    for b, L in enumerate(di.lens):
        if L == 0:                                                  # zero-length sequence: O = 0, LSE = -inf
            assert torch.count_nonzero(ao.t[b].float()) == 0
            assert bool(torch.isneginf(al.t[b]).all())
    return kind


DECODE_CASES = [
    # dtype, D, bs, G, Hkv, lens, splits
    (torch.bfloat16, 128, 16, 4, 2, [300, 0, 17], 1),             # one split: direct store
    (torch.bfloat16, 128, 16, 1, 4, [2000, 0, 700], 3),           # fused merge; G 1 puts the last counter pair last
    (torch.float16, 64, 32, 3, 2, [1500, 3000], 2),               # one cluster of 2 per unit
    (torch.bfloat16, 128, 16, 5, 1, [3000, 100], 4),              # cluster of 4
    (torch.bfloat16, 64, 64, 8, 2, [4000, 0, 700], 8),            # cluster of 8
    (torch.bfloat16, 128, 16, 16, 1, [9000, 50], 24),             # clusters, then partials
    (torch.float16, 128, 16, 32, 1, [9000, 1], 40),               # two 16-row chunks
    (torch.bfloat16, 128, 16, 1, 2, [9000, 0, 4000], 24),
    (torch.bfloat16, 128, 0, 3, 2, [700, 0, 257], 3),             # contiguous cache
    (torch.bfloat16, 64, 0, 5, 1, [64, 1000], 1),
]


@gpu
@pytest.mark.parametrize("dtype,D,bs,G,Hkv,lens,splits", DECODE_CASES)
def test_decode_tma(dtype, D, bs, G, Hkv, lens, splits):
    kind = _decode_case(DecodeInputs(dtype, D, bs, G, Hkv, lens, seed=G + splits + bs), splits)
    assert _lib.KIND_NAMES[kind] == "mma_tma"


@gpu
@pytest.mark.parametrize("bs,lens,splits,odd", [
    (7, [300, 1, 0, 77], 3, True),               # SIMT + combine: f32, D 48, 7-token pages
    (7, [300, 0, 77], 1, False),
    (0, [300, 0, 77], 3, True),                  # contiguous
])
def test_decode_simt(bs, lens, splits, odd):
    kind = _decode_case(DecodeInputs(torch.float32, 48, bs, 3, 2, lens, seed=bs + splits), splits, odd=odd)
    assert _lib.KIND_NAMES[kind] == "simt"


@gpu
@pytest.mark.parametrize("G,q_len,bs,splits,dtype", [
    (3, 6, 16, 0, torch.bfloat16),               # 18 rows per KV head: a 16-row chunk straddles q heads
    (5, 7, 0, 3, torch.bfloat16),                # contiguous cache
    (2, 5, 32, 1, torch.float16),
    (8, 3, 16, 24, torch.bfloat16),
    (3, 4, 24, 3, torch.float32),                # SIMT
])
def test_decode_multi(G, q_len, bs, splits, dtype):
    D = 48 if dtype == torch.float32 else 128
    lens = [q_len, 300 + 7 * q_len, 1000]
    di = DecodeInputs(dtype, D, bs, G, 2, lens, seed=G * q_len, q_len=q_len)
    if splits == 0:
        splits = int(_lib.load().pli_decode_num_splits_multi(di.B, di.Hq, di.Hkv, q_len, di.max_len))
    _decode_case(di, splits, odd=dtype == torch.float32)


def _splitkv(di, q, k, v, table, lens, ws, splits):
    _lib.check(_lib.load().pli_decode_splitkv(q.data_ptr(), k.data_ptr(), v.data_ptr(), table.data_ptr(),
                                              lens.data_ptr(), di.B, di.Hq, di.Hkv, di.D, di.max_len, di.bs,
                                              table.stride(0), di.layer, k.shape[0], _i64(q, 2), _i64(k, 4),
                                              di.D ** -0.5, CODE[q.dtype], splits, ws.data_ptr(), ws.shape[0],
                                              _stream()))


def _combine(di, ws, o, lse, splits):
    _lib.check(_lib.load().pli_decode_combine(ws.data_ptr(), o.data_ptr(), lse.data_ptr(), di.B, di.Hq, di.D, splits,
                                              _i64(o, 2), CODE[o.dtype], _stream()))


@gpu
@pytest.mark.parametrize("splits", [3, 16])
def test_decode_two_pass(splits):
    """pli_decode_splitkv writes only inside the workspace; pli_decode_combine writes only o / lse.  (The reference is
    the same two launches on dense tensors: the one-launch merge of 16 splits goes through clusters and may differ in
    the last bit.)"""
    di = DecodeInputs(torch.bfloat16, 128, 16, 4, 2, [2000, 0, 65], seed=splits)
    o_ref, lse_ref = _fresh(di.out_shape(), di.dtype), _fresh(di.lse_shape())
    ws_ref = _fresh((_ws_bytes(di.B, di.Hq, di.D, splits),), torch.uint8)
    _splitkv(di, di.q, di.k, di.v, di.table, di.lens_t, ws_ref, splits)
    _combine(di, ws_ref, o_ref, lse_ref, splits)
    aq, ak, av = Arg.of("q", di.q, pad=[16, 8, 0]), Arg.of("k", di.k), Arg.of("v", di.v)
    at, asl = Arg.of("block_table", di.table), Arg.of("seq_lens", di.lens_t)
    aw = Arg("workspace", (_ws_bytes(di.B, di.Hq, di.D, splits),), torch.uint8, "ws")
    ins = (aq, ak, av, at, asl)
    for a in ins + (aw,):
        a.arm()
    _splitkv(di, aq.t, ak.t, av.t, at.t, asl.t, aw.t, splits)
    verify(*ins, aw)
    aw.role = "in"                                              # combine only reads the workspace
    ao = Arg("o", di.out_shape(), di.dtype, "out", pad=[40, 8, 0])
    al = Arg("lse", di.lse_shape(), torch.float32, "out")
    for a in (aw, ao, al):
        a.arm()
    _combine(di, aw.t, ao.t, al.t, splits)
    verify(aw, ao, al)
    same_bits(ao.t, o_ref, "o")
    same_bits(al.t, lse_ref, "lse")


@gpu
def test_decode_python_wrappers_with_out():
    """flash_decode(out=...) and DecodePlan(out=...): the same footprint through the Python layer."""
    import physics_llm_inference_b200 as pli
    for q_len in (1, 4):
        di = DecodeInputs(torch.bfloat16, 128, 16, 4, 2, [700, 0, 65], seed=20 + q_len, q_len=q_len)
        splits = 3
        o_ref, lse_ref, _ = di.dense(splits)
        if q_len > 1:
            st = padded_strides(di.out_shape(), [40, 0, 8, 0])
            st[1] = q_len * st[2]
            ao = Arg("o", di.out_shape(), di.dtype, "out", strides=st)
        else:
            ao = Arg("o", di.out_shape(), di.dtype, "out", pad=[40, 8, 0])
        aw = Arg("workspace", (_ws_bytes(di.B, di.Hq * q_len, di.D, splits),), torch.uint8, "ws")
        for call in ("flash_decode", "DecodePlan"):
            for a in (ao, aw):
                a.arm()
            kw = dict(block_tables=di.table, layer=di.layer, num_splits=splits, max_seq_len=di.max_len,
                      workspace=aw.t, out=ao.t, return_lse=True)
            if call == "flash_decode":
                o, lse = pli.flash_decode(di.q, di.k, di.v, di.lens_t, **kw)
            else:
                o, lse = pli.DecodePlan(di.q, di.k, di.v, di.lens_t, **kw)()
            verify(ao, aw)
            assert o.data_ptr() == ao.ptr
            same_bits(ao.t, o_ref, call)
            same_bits(lse, lse_ref, call + " lse")


# ---- read side: poison the storage a kernel must not read ------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype,q_len", [(torch.bfloat16, 1), (torch.bfloat16, 4), (torch.float32, 1),
                                         (torch.float32, 3)])
def test_decode_contiguous_cache_poisoned_past_seq_len(dtype, q_len):
    """NaN K and Inf V past seq_lens[b] in the contiguous cache: not a bit of the result may change."""
    D = 128 if dtype == torch.bfloat16 else 48
    di = DecodeInputs(dtype, D, 0, 4, 2, [700, 64 + q_len, 3 + q_len], seed=30 + q_len, q_len=q_len)
    splits = 3
    o_ref, lse_ref, kind_ref = di.dense(splits)
    for b, L in enumerate(di.lens):
        di.k[b, L:] = float("nan")
        di.v[b, L:] = float("inf")
    kind = _decode_case(di, splits)
    assert kind == kind_ref
    o2, lse2, _ = di.dense(splits)
    same_bits(o2, o_ref, "o over the poisoned cache")
    same_bits(lse2, lse_ref, "lse over the poisoned cache")


@gpu
@pytest.mark.parametrize("hostile", ["int32_max", "poison"])
@pytest.mark.parametrize("dtype,D,bs,q_len", [(torch.bfloat16, 128, 16, 1), (torch.float32, 48, 7, 1),
                                              (torch.bfloat16, 64, 32, 5)])
def test_decode_hostile_table_padding(hostile, dtype, D, bs, q_len):
    """Block-table entries past each sequence's last page hold INT32_MAX, or the id of a NaN / Inf page: the header
    requires only the entries in use to be valid."""
    di = DecodeInputs(dtype, D, bs, 4, 2, [700, 5 + q_len, 1000], seed=40 + bs, q_len=q_len)
    di.pools.table = di.table = torch.cat([di.table, torch.zeros_like(di.table)], 1)   # wider than any sequence needs
    _decode_case(di, 3, hostile=hostile)


@gpu
@pytest.mark.parametrize("hostile", ["int32_max", "poison"])
def test_prefill_hostile_table_padding(hostile):
    pl = Pools([300, 77, 129], 16, 2, 128, torch.bfloat16, seed=50)
    pl.table = torch.cat([pl.table, torch.zeros_like(pl.table)], 1)
    table = pl.hostile(pl.poison_page() if hostile == "poison" else INT32_MAX)
    _paged_prefill_case(16, 128, 2, 4, 77, [300, 77, 129], torch.bfloat16, 50, table=table, pools=pl)
    pv = Pools([300, 5, 1, 77], 16, 2, 128, torch.bfloat16, seed=51)
    table = pv.hostile(pv.poison_page() if hostile == "poison" else INT32_MAX)
    _varlen_case(16, 128, 2, 4, [130, 0, 1, 77], [300, 5, 1, 77], torch.bfloat16, 51, table=table, pools=pv)


# ---- KV append, page gather -----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype,D,paged,tok_pad", [
    (torch.bfloat16, 128, True, 0),              # 16-byte vectors
    (torch.float16, 36, True, 0),                # D 36: scalar path
    (torch.float32, 128, False, 0),              # contiguous cache
    (torch.bfloat16, 128, True, 1),              # odd new-token stride: scalar path
    (torch.float16, 128, False, 3),
])
def test_kv_append(dtype, D, paged, tok_pad):
    """n_new = 40 tokens over 16-token pages from ragged start positions; k_new / v_new are views of one fused
    projection buffer.  Declared write set: exactly the n_new x Hkv x D elements per pool; every other byte of both pools
    (other slots, other layers, page tails, free pages) must not change."""
    B, Hkv, Hq, n, bs, layers, layer = 3, 2, 4, 40, 16, 3, 1
    start = [5, 30, 0]
    ends = [s + n for s in start]
    if paged:
        npg = [-(-e // bs) for e in ends]
        P = sum(npg) + 2
        table = torch.zeros(B, max(npg) + 1, dtype=torch.int32)
        ids = list(range(P - 1, -1, -1))          # the last sequence's last token goes to the end of the pool
        at = 0
        for b in range(B - 1, -1, -1):
            table[b, :npg[b]] = torch.tensor(ids[at:at + npg[b]][::-1], dtype=torch.int32)
            at += npg[b]
        table = table.cuda()
        shape = (P, layers, bs, Hkv, D)
    else:
        table = None
        shape = (B, max(ends), Hkv, D)            # the last sequence fills its cache to the end
    fused = _rand((B, n, Hq + 2 * Hkv, D), dtype, 60 + D)
    kp0, vp0 = _rand(shape, dtype, 61), _rand(shape, dtype, 62)
    wset = torch.zeros(shape, dtype=torch.bool, device="cuda")
    exp_k, exp_v = kp0.clone(), vp0.clone()
    for b in range(B):
        for i in range(n):
            t = start[b] + i
            idx = (int(table[b, t // bs]), layer, t % bs) if paged else (b, t)
            wset[idx] = True
            exp_k[idx] = fused[b, i, Hq:Hq + Hkv]
            exp_v[idx] = fused[b, i, Hq + Hkv:]
    af = Arg.of("kv_new", fused, pad=[0, tok_pad, 0, 0])
    ak, av = Arg.of("k_store", kp0, role="inout"), Arg.of("v_store", vp0, role="inout")
    asp = Arg.of("start_pos", torch.tensor(start, dtype=torch.int32, device="cuda"))
    atb = Arg.of("block_table", table) if paged else None
    args = [a for a in (af, ak, av, asp, atb) if a is not None]
    for a in args:
        a.arm(wset if a in (ak, av) else None)
    kn, vn = af.t[:, :, Hq:Hq + Hkv], af.t[:, :, Hq + Hkv:]
    kvs = ak.t.stride()[:4] if paged else (ak.t.stride(0), 0, ak.t.stride(1), ak.t.stride(2))
    _lib.check(_lib.load().pli_kv_append(kn.data_ptr(), vn.data_ptr(), ak.ptr, av.ptr, _ptr(atb.t if atb else None),
                                         asp.ptr, B, n, Hkv, D, bs if paged else 0, table.stride(0) if paged else 0,
                                         layer if paged else 0, _i64(kn, 3), _lib.i64(*kvs), CODE[dtype], _stream()))
    verify(*args)
    same_bits(ak.t, exp_k, "k_store")
    same_bits(av.t, exp_v, "v_store")


@gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_paged_gather(dtype):
    lens, bs, Hkv, D, max_len = [100, 0, 33], 16, 2, 40, 120
    pl = Pools(lens, bs, Hkv, D, dtype, seed=70)
    B = len(lens)
    ast, atb, asl = Arg.of("store", pl.k), Arg.of("block_table", pl.table), Arg.of("seq_lens", pl.lens_t)
    ao = Arg("out", (B, max_len, Hkv, D), dtype, "out")
    for a in (ast, atb, asl, ao):
        a.arm()
    _lib.check(_lib.load().pli_paged_gather(ast.ptr, ao.ptr, atb.ptr, asl.ptr, B, max_len, Hkv, D, bs, pl.table.stride(0),
                                            pl.layer, _i64(pl.k, 4), CODE[dtype], _stream()))
    verify(ast, atb, asl, ao)
    exp = torch.zeros(B, max_len, Hkv, D, dtype=dtype, device="cuda")
    for b, L in enumerate(lens):
        for t in range(L):
            exp[b, t] = pl.k[int(pl.table[b, t // bs]), pl.layer, t % bs]
    same_bits(ao.t, exp, "out")                                  # rows at or past seq_len come out as 0


# ---- online softmax -------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype,pad", [(torch.float32, 3), (torch.bfloat16, 1), (torch.float16, 8)])
def test_online_softmax(dtype, pad):
    rows, n = 37, 300
    x = _rand((rows, n), dtype, 80, scale=3.0)
    ref = _fresh(x.shape, dtype)
    lib = _lib.load()
    _lib.check(lib.pli_online_softmax(x.data_ptr(), ref.data_ptr(), rows, n, n, n, CODE[dtype], _stream()))
    ax = Arg.of("x", x, pad=[pad, 0])                          # NaN in the gaps of every input row
    ao = Arg("out", (rows, n), dtype, "out", pad=[pad + 2, 0])
    for a in (ax, ao):
        a.arm()
    _lib.check(lib.pli_online_softmax(ax.ptr, ao.ptr, rows, n, ax.t.stride(0), ao.t.stride(0), CODE[dtype], _stream()))
    verify(ax, ao)
    same_bits(ao.t, ref, "out")
    torch.testing.assert_close(ao.t.float(), torch.softmax(x.float(), -1), atol=1e-2, rtol=1e-2)


@gpu
@pytest.mark.parametrize("dv", [1, 130, 256])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_online_softmax_with_output(dv, dtype):
    rows, n = 21, 77
    x, v = _rand((rows, n), dtype, 81, scale=2.0), _rand((rows, n, dv), dtype, 82)
    lib = _lib.load()
    o_ref, d_ref = _fresh((rows, dv), dtype), _fresh((rows,))
    _lib.check(lib.pli_online_softmax_with_output(x.data_ptr(), v.data_ptr(), o_ref.data_ptr(), d_ref.data_ptr(), rows, n,
                                                  dv, n, n * dv, dv, dv, CODE[dtype], _stream()))
    ax, av = Arg.of("x", x, pad=[5, 0]), Arg.of("v", v, pad=[3, 1, 0])
    ao, ad = Arg("o", (rows, dv), dtype, "out", pad=[3, 0]), Arg("d", (rows,), torch.float32, "out")
    for a in (ax, av, ao, ad):
        a.arm()
    _lib.check(lib.pli_online_softmax_with_output(ax.ptr, av.ptr, ao.ptr, ad.ptr, rows, n, dv, ax.t.stride(0),
                                                  av.t.stride(0), av.t.stride(1), ao.t.stride(0), CODE[dtype],
                                                  _stream()))
    verify(ax, av, ao, ad)
    same_bits(ao.t, o_ref, "o")
    same_bits(ad.t, d_ref, "d")
    p = torch.softmax(x.float(), -1)
    torch.testing.assert_close(ao.t.float(), torch.einsum("rn,rnd->rd", p, v.float()), atol=2e-2, rtol=2e-2)


# ---- peer output, world of one --------------------------------------------------------------------------------------
def _peer(header, out_arg):
    """pli_peer_scatter for rank 0 of 1: output buffers in `out_arg` (dim 0 = buffer), words in `header`."""
    ps = _lib.PeerScatter()
    ps.n_peers, ps.rank = 1, 0
    ps.peer_o[0] = out_arg.t[0].data_ptr()
    base = header.ptr
    ps.peer_flags[0], ps.peer_ready[0], ps.epoch, ps.cta_counter = base, base + 64, base + 256, base + 260
    ps.buffer_stride = out_arg.t.stride(0) if out_arg.shape[0] == 2 else 0
    return ps


def _header():
    h = Arg("peer_words", (512,), torch.uint8, "ws")
    h.t.zero_()
    return h


def _epoch(h):
    return int(h.t[256:260].view(torch.int32)[0])


@gpu
@pytest.mark.parametrize("dtype,D", [(torch.float32, 48), (torch.bfloat16, 128)])
def test_decode_peer_output_single_rank(dtype, D):
    """Scatter mode (f32 / SIMT): step e writes buffer e & 1 and nothing else, the other buffer stays bit-identical.
    Gather mode (bf16 / TMA): one buffer, nothing outside it changes.  The copy to a fixed destination writes exactly
    nbytes."""
    di = DecodeInputs(dtype, D, 16, 4, 2, [700, 0, 65], seed=90)
    splits = 3
    o_ref, lse_ref, kind = di.dense(splits)
    scatter = _lib.KIND_NAMES[kind] == "simt"
    lib = _lib.load()
    nbuf = 2 if scatter else 1
    ao = Arg("peer_o", (nbuf,) + tuple(di.out_shape()), dtype, "out", pad=[64, 0, 0, 0])
    h = _header()
    aq, ak, av, at, asl = (Arg.of("q", di.q), Arg.of("k", di.k), Arg.of("v", di.v), Arg.of("block_table", di.table),
                           Arg.of("seq_lens", di.lens_t))
    al = Arg("lse", di.lse_shape(), torch.float32, "out")
    aw = Arg("workspace", (_ws_bytes(di.B, di.Hq, D, splits),), torch.uint8, "ws")
    ps = _peer(h, ao)
    wset = torch.zeros(ao.shape, dtype=torch.bool, device="cuda")
    for step in range(1, 4):
        buf = step & 1 if scatter else 0
        wset.zero_()
        wset[buf] = True
        for a in (aq, ak, av, at, asl, al, aw, h):
            a.arm()
        ao.arm(wset)
        fwd = lib.pli_decode_fwd_scatter if scatter else lib.pli_decode_fwd_gather
        _lib.check(fwd(aq.ptr, ak.ptr, av.ptr, at.ptr, asl.ptr, al.ptr, di.B, di.Hq, di.Hkv, D, di.max_len, di.bs,
                       at.t.stride(0), di.layer, di.k.shape[0], _i64(aq.t, 2), _i64(ak.t, 4),
                       _lib.i64(ao.t.stride(1), ao.t.stride(2)), D ** -0.5, CODE[dtype], splits, aw.ptr, aw.shape[0],
                       ctypes.byref(ps), _stream()))
        if scatter:
            _lib.check(lib.pli_peer_publish_wait(ctypes.byref(ps), _stream()))
        verify(aq, ak, av, at, asl, al, aw, h, ao)
        _lib.raise_on_device_fault()
        assert _epoch(h) == step
        same_bits(ao.t[buf], o_ref, f"step {step}")
        same_bits(al.t, lse_ref, f"lse step {step}")
        if scatter:                                               # select-copy the finished step's buffer
            nbytes = o_ref.numel() * o_ref.element_size()
            ad = Arg("dst", (nbytes // o_ref.element_size(),), dtype, "out")
            ao.role = "in"
            for a in (ad, ao, h):
                a.arm()
            _lib.check(lib.pli_peer_select_copy(ctypes.byref(ps), ad.ptr, nbytes, o_ref.element_size(), _stream()))
            verify(ad, ao, h)
            ao.role = "out"
            same_bits(ad.t.view(o_ref.shape), o_ref, "select_copy")


@gpu
def test_prefill_peer_output_single_rank():
    """pli_prefill_fwd_scatter, world of one: step e writes buffer e & 1, the other buffer stays bit-identical."""
    B, Hq, Hkv, N, D, dtype = 2, 8, 2, 300, 128, torch.bfloat16
    q, k, v = _rand((B, Hq, N, D), dtype, 95), _rand((B, Hkv, N, D), dtype, 96), _rand((B, Hkv, N, D), dtype, 97)
    o_ref, lse_ref = _fresh(q.shape, dtype), _fresh((B, Hq, N))
    _prefill_call(q, k, v, o_ref, lse_ref, Hkv, N, D ** -0.5, True)
    lib = _lib.load()
    ao = Arg("peer_o", (2, B, Hq, N, D), dtype, "out", pad=[512, 0, 0, 0, 0])
    h = _header()
    aq, ak, av = Arg.of("q", q), Arg.of("k", k), Arg.of("v", v)
    al = Arg("lse", (B, Hq, N), torch.float32, "out")
    ps = _peer(h, ao)
    wset = torch.zeros(ao.shape, dtype=torch.bool, device="cuda")
    for step in range(1, 4):
        buf = step & 1
        wset.zero_()
        wset[buf] = True
        for a in (aq, ak, av, al, h):
            a.arm()
        ao.arm(wset)
        _lib.check(lib.pli_prefill_fwd_scatter(aq.ptr, ak.ptr, av.ptr, al.ptr, B, Hq, Hkv, N, N, D, _i64(q, 3),
                                               _i64(k, 3), _i64(v, 3), _lib.i64(*ao.t.stride()[1:4]), D ** -0.5, 1,
                                               _lib.PLI_BF16, B, Hq, 0, 0, ctypes.byref(ps), _stream()))
        _lib.check(lib.pli_peer_publish_wait(ctypes.byref(ps), _stream()))
        verify(aq, ak, av, al, h, ao)
        _lib.raise_on_device_fault()
        assert _epoch(h) == step
        same_bits(ao.t[buf], o_ref, f"step {step}")
        same_bits(al.t, lse_ref, f"lse step {step}")
