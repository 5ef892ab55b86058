"""Exact-logit readout tests of every attention kernel (oracle/readout.py): one-hot Q, K = beta_c * s_j, one-hot V, so
O is the kernel's attention weights read back per V class and the fp64 prefix-scan reference is exact on the kernel's
inputs.  Every row of every case is compared against a bound derived from the rounding the kernels do; each case
records its worst err / bound ratio, which must be in (0, 1]."""
import math

import pytest
import torch

import physics_llm_inference_b200 as pli
from oracle import readout as ro
from physics_llm_inference_b200 import _lib

pytestmark = pytest.mark.gpu
F64 = torch.float64
CHUNK = 32768                     # rows compared at a time
WORST = {}                        # path -> worst (O ratio, LSE ratio) over the module


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nreadout worst err/bound ratio per path (O, LSE):")
    for path in sorted(WORST):
        print(f"  {path:32s} {WORST[path][0]:.4f} {WORST[path][1]:.4f}")


def _note(path, r_o, r_l):
    assert r_o <= 1.0 and r_l <= 1.0, (path, r_o, r_l)
    assert r_o > 0, f"{path}: nothing was compared"
    w = WORST.get(path, (0.0, 0.0))
    WORST[path] = (max(w[0], r_o), max(w[1], r_l))


class Batch:
    """B sequences x Hkv kv heads of readout K / V (lens[b] keys each), with the reference of each (sequence, head)."""

    def __init__(self, seed, B, Hkv, lens, D, dtype, profs, scale, needles=None):
        self.B, self.Hkv, self.lens, self.D, self.dtype, self.scale = B, Hkv, list(lens), D, dtype, scale
        self.seqs, self._refs = {}, {}
        for b in range(B):
            for hk in range(Hkv):
                u = b * Hkv + hk
                g = torch.Generator().manual_seed(seed * 7919 + u)
                L = self.lens[b]
                if L == 0:
                    self.seqs[b, hk] = None
                    continue
                nd = None if needles is None else needles[u] % L
                name = "needle" if nd is not None else profs[(u + seed) % len(profs)]
                s = ro.profile(name, L, g, scale, dtype, needle_at=nd)
                cls = ro.classes(L, D, g)
                self.seqs[b, hk] = (s, cls) + ro.make_kv(s, cls, D, dtype)

    def _garbage(self, *shape, seed=0):
        return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)).to(self.dtype)

    def contiguous(self, Nk):
        """K, V (B, Hkv, Nk, D)."""
        K = self._garbage(self.B, self.Hkv, Nk, self.D, seed=1)
        V = self._garbage(self.B, self.Hkv, Nk, self.D, seed=2)
        for (b, hk), sq in self.seqs.items():
            if sq is not None:
                K[b, hk, :self.lens[b]], V[b, hk, :self.lens[b]] = sq[2], sq[3]
        return K.cuda(), V.cuda()

    def cache(self, cap):
        """ch02 cache layout (B, cap, Hkv, D); slots past seq_len hold garbage."""
        K = self._garbage(self.B, cap, self.Hkv, self.D, seed=3)
        V = self._garbage(self.B, cap, self.Hkv, self.D, seed=4)
        for (b, hk), sq in self.seqs.items():
            if sq is not None:
                K[b, :self.lens[b], hk], V[b, :self.lens[b], hk] = sq[2], sq[3]
        return K.cuda(), V.cuda()

    def pools(self, bs, layers=1, layer=0, seed=5):
        """ch07 pools (P, layers, bs, Hkv, D) in a random page order; unused slots hold garbage."""
        npg = [max(1, (L + bs - 1) // bs) for L in self.lens]
        P = sum(npg) + 3
        perm = torch.randperm(P, generator=torch.Generator().manual_seed(seed)).to(torch.int32)
        table = torch.zeros(self.B, max(npg), dtype=torch.int32)
        at = 0
        for b, n in enumerate(npg):
            table[b, :n] = perm[at:at + n]
            at += n
        kp = self._garbage(P, layers, bs, self.Hkv, self.D, seed=6)
        vp = self._garbage(P, layers, bs, self.Hkv, self.D, seed=7)
        for (b, hk), sq in self.seqs.items():
            if sq is None:
                continue
            pages = table[b, :npg[b]].long()
            for pool, x in ((kp, sq[2]), (vp, sq[3])):
                blk = pool[pages, layer, :, hk].reshape(-1, self.D)
                blk[:self.lens[b]] = x
                pool[pages, layer, :, hk] = blk.view(npg[b], bs, self.D)
        return kp.cuda(), vp.cuda(), table.cuda()

    def ref(self, b, hk, t):
        key = (b, hk, t)
        if key not in self._refs:
            s, cls = self.seqs[b, hk][:2]
            self._refs[key] = ro.prefix_reference(s, cls, self.D, t * self.scale)
        return self._refs[key]

    def check(self, b, hk, o, lse, t, lim, p_dtype=None):
        """o (R, D) on the GPU, lse (R,) or None, t (R,) float64, lim (R,) visible-prefix lengths: (O ratio, LSE ratio)."""
        p_dtype = self.dtype if p_dtype is None else p_dtype
        t, lim = t.cpu(), lim.cpu().long()
        r_o = r_l = 0.0
        dead = lim <= 0
        if bool(dead.any()):                              # no visible key: O = 0, LSE = -inf, no NaN
            od = o[dead.to(o.device)].float()
            assert not torch.isnan(od).any() and torch.count_nonzero(od) == 0
            if lse is not None:
                ld = lse[dead.to(lse.device)]
                assert bool(torch.isinf(ld).all()) and bool((ld < 0).all())
        for tv in torch.unique(t).tolist():
            rows = torch.nonzero((t == tv) & ~dead).flatten()
            if not rows.numel():
                continue
            W, rl, wmax, counts = self.ref(b, hk, tv)
            for c0 in range(0, rows.numel(), CHUNK):
                rr = rows[c0:c0 + CHUNK]
                p = lim[rr] - 1
                og = o[rr.to(o.device)].to(F64).cpu()
                bnd = ro.bound(W[p], wmax[p], counts[p], self.dtype, p_dtype)
                r_o = max(r_o, ro.ratio((og - W[p]).abs(), bnd))
                if lse is not None:
                    lg = lse[rr.to(lse.device)].to(F64).cpu()
                    r_l = max(r_l, ro.ratio((lg - rl[p]).abs(), ro.lse_bound(rl[p])))
        return r_o, r_l


def _q(shape, D, T, dtype, device="cuda"):
    n = math.prod(shape)
    return ro.make_q(torch.arange(n, device=device).view(*shape), D, T, dtype)


def _worst(*pairs):
    return max(p[0] for p in pairs), max(p[1] for p in pairs)


# ---------------------------------------------------------------------------------------------------------------------
# prefill, contiguous
# ---------------------------------------------------------------------------------------------------------------------
def _prefill(path, seed, B, Hq, Hkv, Nq, Nk, D, dtype, causal, profs, T=ro.RAMP_T, scale=None, p_dtype=None,
             kind=None):
    sc = D ** -0.5 if scale is None else scale
    bt = Batch(seed, B, Hkv, [Nk] * B, D, dtype, profs, sc)
    K, V = bt.contiguous(Nk)
    q, t = _q((B, Hq, Nq), D, T, dtype)
    if kind is not None:
        assert pli.prefill_kernel_kind(q, K, V) == kind
    o, lse = pli.flash_attention_forward(q, K, V, scale, causal=causal, return_lse=True)
    torch.cuda.synchronize()
    G = Hq // Hkv
    i = torch.arange(Nq)
    lim_i = i + 1 + Nk - Nq if causal else torch.full((Nq,), Nk)
    res = []
    for b in range(B):
        for hk in range(Hkv):
            hs = slice(hk * G, (hk + 1) * G)
            res.append(bt.check(b, hk, o[b, hs].reshape(-1, D), lse[b, hs].reshape(-1), t[b, hs].reshape(-1),
                                lim_i.repeat(G), p_dtype))
    r = _worst(*res)
    _note(path, *r)
    return o, lse


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("shape", [
    (1, 8, 8, 512, 512, 64),         # G 1
    (1, 4, 1, 256, 256, 128),        # G 4, two Q tiles
    (2, 8, 1, 300, 300, 128),        # G 8, ragged tiles
    (3, 6, 3, 513, 513, 128),
    (1, 4, 2, 77, 333, 64),          # Nq < Nk
    (1, 8, 2, 129, 1000, 128),
    (1, 2, 2, 1, 17, 128),
])
def test_prefill_tcgen05(shape, causal, dtype):
    B, Hq, Hkv, Nq, Nk, D = shape
    _prefill("prefill_tcgen05", B + Hq + Nq + Nk + D + causal, B, Hq, Hkv, Nq, Nk, D, dtype, causal, ro.PROFILES,
             kind="tcgen05")


def test_prefill_fp16_large_raw_scores():
    """q.k up to ~2.5e5 (outside fp16) with scale 2^-16: S must stay fp32 on its way to the exponentials."""
    _prefill("prefill_tcgen05_bigraw", 11, 1, 4, 2, 300, 300, 128, torch.float16, True, ("bigraw",), T=(8, 16),
             scale=2.0 ** -16, kind="tcgen05")


def test_prefill_c2_every_row():
    """BASELINE C2 (B4, 32 q / 8 kv heads, N 8192, D 128, causal, bf16): every row of every head."""
    _prefill("prefill_c2", 12, 4, 32, 8, 8192, 8192, 128, torch.bfloat16, True,
             ("ramp7.5", "noise4", "ramp4", "sink", "noise16", "uniform", "noise1", "needle"), kind="tcgen05")


def test_prefill_c4_shard_every_row():
    """The C4 rank shard (B1, 4 q / 1 kv head, N 65 536, causal, bf16): every row."""
    _prefill("prefill_c4_shard", 13, 1, 4, 1, 65536, 65536, 128, torch.bfloat16, True, ("noise4",), T=(1, 2),
             kind="tcgen05")


@pytest.mark.parametrize("D", [48, 80])
@pytest.mark.parametrize("causal", [False, True])
def test_prefill_simt_fp32(D, causal):
    _prefill("prefill_simt", 14 + D, 2, 4, 2, 70, 100, D, torch.float32, causal, ro.PROFILES, kind="simt")


def test_prefill_simt_negative_scale_and_zero_strides():
    """scale <= 0 goes to the SIMT kernel (P in fp32); broadcast K / V through the C ABI reach it too."""
    _prefill("prefill_simt_neg_scale", 15, 1, 4, 2, 200, 200, 128, torch.bfloat16, True, ("noise4", "ramp4"),
             scale=-(128 ** -0.5), p_dtype=torch.float32)
    D, N, B, Hq = 128, 150, 3, 4
    bt = Batch(16, 1, 1, [N], D, torch.bfloat16, ("noise4",), D ** -0.5)
    K, V = bt.contiguous(N)
    ke, ve = K.expand(B, Hq, -1, -1), V.expand(B, Hq, -1, -1)          # batch and head stride 0
    q, t = _q((B, Hq, N), D, ro.RAMP_T, torch.bfloat16)
    o = torch.empty_like(q)
    lse = torch.empty(B, Hq, N, device="cuda")
    lib = _lib.load()
    _lib.check(lib.pli_prefill_fwd(q.data_ptr(), ke.data_ptr(), ve.data_ptr(), o.data_ptr(), lse.data_ptr(), B, Hq, Hq,
                                   N, N, D, _lib.i64(*q.stride()[:3]), _lib.i64(*ke.stride()[:3]),
                                   _lib.i64(*ve.stride()[:3]), _lib.i64(*o.stride()[:3]), D ** -0.5, 1, _lib.PLI_BF16,
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    lim = torch.arange(N) + 1
    res = [bt.check(0, 0, o[b].reshape(-1, D), lse[b].reshape(-1), t[b].reshape(-1), lim.repeat(Hq), torch.float32)
           for b in range(B)]
    _note("prefill_simt_zero_stride", *_worst(*res))


# ---------------------------------------------------------------------------------------------------------------------
# prefill over the paged pools: flash_attention_paged, flash_attention_varlen_paged, mixed_batch_attention
# ---------------------------------------------------------------------------------------------------------------------
def _paged_prefill(path, seed, bs, D, Hkv, G, Nq, lens, dtype, profs, needles=None):
    B, Hq = len(lens), Hkv * G
    bt = Batch(seed, B, Hkv, lens, D, dtype, profs, D ** -0.5, needles=needles)
    kp, vp, table = bt.pools(bs, layers=2, layer=1)
    q, t = _q((B, Hq, Nq), D, ro.RAMP_T, dtype)
    lens_t = torch.tensor(lens, dtype=torch.int32).cuda()
    o, lse = pli.flash_attention_paged(q, kp, vp, table, lens_t, layer=1, return_lse=True, max_seq_len=max(lens))
    torch.cuda.synchronize()
    res = []
    for b in range(B):
        lim = torch.arange(Nq) + 1 + lens[b] - Nq
        for hk in range(Hkv):
            hs = slice(hk * G, (hk + 1) * G)
            res.append(bt.check(b, hk, o[b, hs].reshape(-1, D), lse[b, hs].reshape(-1), t[b, hs].reshape(-1),
                                lim.repeat(G)))
    r = _worst(*res)
    _note(path, *r)
    return r


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("bs,D,Hkv,G,Nq,lens", [
    (16, 128, 2, 4, 128, [512, 300, 128]),          # CTA pairs
    (16, 128, 1, 2, 200, [777, 200]),               # head pairs
    (64, 64, 2, 1, 96, [1000, 97, 640]),            # MHA row pairs, D 64
    (128, 128, 2, 8, 256, [1500, 256]),
    (32, 128, 1, 4, 1, [33, 1, 64]),
])
def test_paged_prefill(bs, D, Hkv, G, Nq, lens, dtype):
    _paged_prefill("prefill_paged", bs + D + G, bs, D, Hkv, G, Nq, lens, dtype, ro.PROFILES)


def _varlen(path, seed, bs, D, Hkv, G, q_lens, lens, dtype, profs, needles=None):
    B, Hq, T = len(lens), Hkv * G, sum(q_lens)
    bt = Batch(seed, B, Hkv, lens, D, dtype, profs, D ** -0.5, needles=needles)
    kp, vp, table = bt.pools(bs, layers=2, layer=1)
    q, t = _q((T, Hq), D, ro.RAMP_T, dtype)
    cu = torch.tensor([0] + q_lens, dtype=torch.int32).cumsum(0, dtype=torch.int32)
    o, lse = pli.flash_attention_varlen_paged(q, kp, vp, table, torch.tensor(lens, dtype=torch.int32).cuda(),
                                              cu.cuda(), max(q_lens), layer=1, return_lse=True, max_seq_len=max(lens))
    torch.cuda.synchronize()
    res = []
    for b in range(B):
        a, e = int(cu[b]), int(cu[b + 1])
        lim = torch.arange(e - a) + 1 + lens[b] - (e - a)
        for hk in range(Hkv):
            hs = slice(hk * G, (hk + 1) * G)
            res.append(bt.check(b, hk, o[a:e, hs].transpose(0, 1).reshape(-1, D), lse[hs, a:e].reshape(-1),
                                t[a:e, hs].transpose(0, 1).reshape(-1), lim.repeat(G)))
    r = _worst(*res)
    _note(path, *r)
    return r


@pytest.mark.parametrize("bs,D,Hkv,G,q_lens,lens", [
    (16, 128, 2, 4, [128, 37, 300, 1], [512, 300, 300, 77]),
    (16, 128, 1, 2, [200, 129, 5], [777, 129, 900]),
    (64, 64, 2, 1, [96, 260, 31], [1000, 260, 640]),
    (32, 128, 1, 3, [64, 257], [64, 300]),
])
def test_varlen_paged_prefill(bs, D, Hkv, G, q_lens, lens):
    _varlen("prefill_varlen", bs + G, bs, D, Hkv, G, q_lens, lens, torch.bfloat16, ro.PROFILES)


def test_mixed_batch_attention():
    """Two prompts prefilled while three requests decode, over a PagedKVCache."""
    Hq, Hkv, D, bs, dtype = 8, 2, 128, 16, torch.bfloat16
    G = Hq // Hkv
    prefill_ids, prefill_lens, decode_ids = [10, 11], [333, 90], [3, 4, 5]
    lens = [333, 90 + 50, 500, 77, 1300]                            # cached lengths incl. this step's tokens
    rids = prefill_ids + decode_ids
    bt = Batch(17, len(rids), Hkv, lens, D, dtype, ro.PROFILES, D ** -0.5)
    cache = pli.PagedKVCache(num_blocks=256, block_size=bs, num_layers=1, num_heads=Hkv, head_dim=D, dtype=dtype,
                             device="cuda")
    for i, rid in enumerate(rids):
        k = torch.stack([bt.seqs[i, hk][2] for hk in range(Hkv)], 1).unsqueeze(0).cuda()
        v = torch.stack([bt.seqs[i, hk][3] for hk in range(Hkv)], 1).unsqueeze(0).cuda()
        cache.append([rid], k, v)
    n_rows = prefill_lens + [1] * len(decode_ids)
    q, t = _q((sum(n_rows), Hq), D, ro.RAMP_T, dtype)
    o = pli.mixed_batch_attention(q, cache, prefill_ids, prefill_lens, decode_ids)
    torch.cuda.synchronize()
    res, at = [], 0
    for i, n in enumerate(n_rows):
        lim = torch.arange(n) + 1 + lens[i] - n
        for hk in range(Hkv):
            hs = slice(hk * G, (hk + 1) * G)
            res.append(bt.check(i, hk, o[at:at + n, hs].transpose(0, 1).reshape(-1, D), None,
                                t[at:at + n, hs].transpose(0, 1).reshape(-1), lim.repeat(G)))
        at += n
    _note("mixed_batch", *_worst(*res))


# ---------------------------------------------------------------------------------------------------------------------
# decode: one token (TMA, SIMT, contiguous, every split merge, the two-pass C-ABI path), several tokens
# ---------------------------------------------------------------------------------------------------------------------
def _decode(path, bt, q, t, o, lse, Nq):
    """o (B, Hq, D) or (B, Hq, Nq, D); row i of a sequence of length L sees keys [0, i + 1 + L - Nq)."""
    B, Hq, D, Hkv = q.shape[0], q.shape[1], q.shape[-1], bt.Hkv
    G = Hq // Hkv
    res = []
    for b in range(B):
        lim = torch.arange(Nq) + 1 + bt.lens[b] - Nq if bt.lens[b] else torch.zeros(Nq, dtype=torch.long)
        for hk in range(Hkv):
            if bt.seqs[b, hk] is None:
                assert torch.count_nonzero(o[b, hk * G:(hk + 1) * G]) == 0
                assert bool(torch.isneginf(lse[b, hk * G:(hk + 1) * G]).all())
                continue
            hs = slice(hk * G, (hk + 1) * G)
            res.append(bt.check(b, hk, o[b, hs].reshape(-1, D), lse[b, hs].reshape(-1), t[b, hs].reshape(-1),
                                lim.repeat(G)))
    r = _worst(*res)
    _note(path, *r)
    return r


def _paged_decode(path, seed, bs, D, Hkv, G, lens, dtype, splits, profs=ro.PROFILES, Nq=1, needles=None, p_dtype=None):
    B, Hq = len(lens), Hkv * G
    bt = Batch(seed, B, Hkv, lens, D, dtype, profs, D ** -0.5, needles=needles)
    kp, vp, table = bt.pools(bs, layers=2, layer=1)
    q, t = _q((B, Hq, Nq) if Nq > 1 else (B, Hq), D, ro.RAMP_T, dtype)
    lens_t = torch.tensor(lens, dtype=torch.int32).cuda()
    o, lse = pli.flash_decode(q, kp, vp, lens_t, block_tables=table, layer=1, return_lse=True, num_splits=splits,
                              max_seq_len=max(lens))
    torch.cuda.synchronize()
    assert pli.decode_kernel_kind(kp, table) == ("simt" if p_dtype == torch.float32 else "mma_tma")
    return _decode(path, bt, q, t, o, lse, Nq)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("splits", [None, 1, 2, 3, 8, 16, 37, 64])
@pytest.mark.parametrize("bs,D,G,lens", [
    (16, 128, 4, [4096, 100, 1, 17, 2048]),      # G <= 8
    (64, 64, 8, [3000, 513, 65]),
    (128, 128, 16, [2500, 128, 129]),            # 16 rows
    (16, 128, 32, [2000, 555, 16]),              # G > 16: two 16-row chunks
])
def test_decode_tma_one_token(bs, D, G, lens, splits, dtype):
    _paged_decode("decode_tma", bs + D + G + (splits or 0), bs, D, 2, G, lens, dtype, splits)


@pytest.mark.parametrize("splits", [None, 3])
def test_decode_simt_and_contiguous(splits):
    """SIMT (fp32, D 48, 7-token pages) and the contiguous ch02 cache on both kernels."""
    _paged_decode("decode_simt", 30, 7, 48, 2, 3, [300, 1, 77], torch.float32, splits, p_dtype=torch.float32)
    for dtype in (torch.bfloat16, torch.float32):
        lens = [700, 3, 257, 64]
        bt = Batch(31, len(lens), 2, lens, 128, dtype, ro.PROFILES, 128 ** -0.5)
        kc, vc = bt.cache(705)
        q, t = _q((len(lens), 8), 128, ro.RAMP_T, dtype)
        o, lse = pli.flash_decode(q, kc, vc, torch.tensor(lens, dtype=torch.int32).cuda(), return_lse=True,
                                  num_splits=splits)
        torch.cuda.synchronize()
        assert pli.decode_kernel_kind(kc) == ("mma_tma" if dtype == torch.bfloat16 else "simt")
        _decode("decode_contiguous_" + pli.decode_kernel_kind(kc), bt, q, t, o, lse, 1)


@pytest.mark.parametrize("splits", [3, 16])
def test_decode_two_pass_c_abi(splits):
    """pli_decode_splitkv + pli_decode_combine."""
    B, Hkv, G, D, bs = 3, 2, 4, 128, 16
    lens = [2000, 700, 65]
    Hq = Hkv * G
    bt = Batch(32, B, Hkv, lens, D, torch.bfloat16, ro.PROFILES, D ** -0.5)
    kp, vp, table = bt.pools(bs)
    q, t = _q((B, Hq), D, ro.RAMP_T, torch.bfloat16)
    lens_t = torch.tensor(lens, dtype=torch.int32).cuda()
    lib = _lib.load()
    ws = torch.empty(int(lib.pli_decode_workspace_bytes(B, Hq, D, splits)) // 4, dtype=torch.float32, device="cuda")
    o = torch.empty(B, Hq, D, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, Hq, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pli_decode_splitkv(q.data_ptr(), kp.data_ptr(), vp.data_ptr(), table.data_ptr(), lens_t.data_ptr(),
                                      B, Hq, Hkv, D, max(lens), bs, table.stride(0), 0, kp.shape[0],
                                      _lib.i64(q.stride(0), q.stride(1)), _lib.i64(*kp.stride()[:4]), D ** -0.5,
                                      _lib.dtype_code(q.dtype), splits, ws.data_ptr(), ws.numel() * 4, stream))
    _lib.check(lib.pli_decode_combine(ws.data_ptr(), o.data_ptr(), lse.data_ptr(), B, Hq, D, splits,
                                      _lib.i64(o.stride(0), o.stride(1)), _lib.dtype_code(q.dtype), stream))
    torch.cuda.synchronize()
    _decode("decode_two_pass", bt, q, t, o, lse, 1)


def test_decode_c3_every_sequence_and_head():
    """BASELINE C3 (B64, ctx 4096, 32 q / 8 kv heads, D 128, 16-token pages, bf16): every sequence and head."""
    lens = [4096] * 64
    lens[17] = 4091
    _paged_decode("decode_c3", 33, 16, 128, 8, 4, lens, torch.bfloat16, None,
                  profs=("noise4", "ramp7.5", "sink", "noise16", "uniform", "needle", "noise1", "ramp4"))


@pytest.mark.parametrize("Nq,G,splits,bs", [(2, 4, None, 16), (3, 8, 3, 64), (5, 2, 8, 0), (8, 4, 37, 16),
                                            (16, 1, 2, 128), (6, 3, None, 16), (7, 5, 3, 32), (16, 4, 1, 0)])
def test_decode_multi_token(Nq, G, splits, bs):
    """Nq new tokens per sequence; G = 3 with Nq = 6 and G = 5 with Nq = 7 put 16-row chunks across q heads."""
    dtype, D, Hkv = torch.bfloat16, 128, 2
    lens = [Nq, 300 + 7 * Nq, 64 + Nq - 1, 1000]
    bt = Batch(40 + Nq + G, len(lens), Hkv, lens, D, dtype, ro.PROFILES, D ** -0.5)
    q, t = _q((len(lens), Hkv * G, Nq), D, ro.RAMP_T, dtype)
    lens_t = torch.tensor(lens, dtype=torch.int32).cuda()
    if bs:
        kp, vp, table = bt.pools(bs)
        o, lse = pli.flash_decode(q, kp, vp, lens_t, block_tables=table, return_lse=True, num_splits=splits,
                                  max_seq_len=max(lens))
    else:
        kc, vc = bt.cache(max(lens) + 3)
        o, lse = pli.flash_decode(q, kc, vc, lens_t, return_lse=True, num_splits=splits)
    torch.cuda.synchronize()
    _decode("decode_multi", bt, q, t, o, lse, Nq)


def test_decode_multi_token_simt():
    _paged_decode("decode_multi_simt", 50, 24, 64, 2, 4, [4, 77, 130, 300], torch.float32, 3, Nq=4,
                  p_dtype=torch.float32)


# ---------------------------------------------------------------------------------------------------------------------
# needle sweeps: one needle per (sequence, kv head) per launch, launches until every key index has held one
# ---------------------------------------------------------------------------------------------------------------------
def _sweep(L, n_units, run):
    worst = (0.0, 0.0)
    for r in range((L + n_units - 1) // n_units):
        needles = [(r * n_units + u) % L for u in range(n_units)]
        worst = _worst(worst, run(needles))
    return worst


def test_needle_sweep_paged_decode():
    """bs 16, L = 1000 (not a multiple of 16), 3 splits, 8 x 4 = 32 (sequence, head) units per launch."""
    L = 1000
    _sweep(L, 32, lambda nd: _paged_decode("needle_decode", 60, 16, 128, 4, 4, [L] * 8, torch.bfloat16, 3,
                                           needles=nd))


def test_needle_sweep_paged_decode_five_tokens():
    L = 1000
    _sweep(L, 32, lambda nd: _paged_decode("needle_decode_multi", 61, 16, 128, 4, 4, [L] * 8, torch.bfloat16, 3,
                                           Nq=5, needles=nd))


def test_needle_sweep_contiguous_decode():
    L, B, Hkv, G, D = 1000, 8, 4, 4, 128

    def run(nd):
        bt = Batch(62, B, Hkv, [L] * B, D, torch.bfloat16, (), D ** -0.5, needles=nd)
        kc, vc = bt.cache(L + 8)
        q, t = _q((B, Hkv * G), D, ro.RAMP_T, torch.bfloat16)
        o, lse = pli.flash_decode(q, kc, vc, L, return_lse=True)
        torch.cuda.synchronize()
        return _decode("needle_decode_contiguous", bt, q, t, o, lse, 1)
    _sweep(L, B * Hkv, run)


def test_needle_sweep_causal_prefill():
    """77 queries over 333 keys, bf16: rows before the needle must not see it."""
    def run(nd):
        B, Hkv, G, Nq, Nk, D = 8, 4, 2, 77, 333, 64
        bt = Batch(63, B, Hkv, [Nk] * B, D, torch.bfloat16, (), D ** -0.5, needles=nd)
        K, V = bt.contiguous(Nk)
        q, t = _q((B, Hkv * G, Nq), D, ro.RAMP_T, torch.bfloat16)
        o, lse = pli.flash_attention_forward(q, K, V, causal=True, return_lse=True)
        torch.cuda.synchronize()
        lim = torch.arange(Nq) + 1 + Nk - Nq
        res = [bt.check(b, hk, o[b, hk * G:(hk + 1) * G].reshape(-1, D), lse[b, hk * G:(hk + 1) * G].reshape(-1),
                        t[b, hk * G:(hk + 1) * G].reshape(-1), lim.repeat(G)) for b in range(B) for hk in range(Hkv)]
        r = _worst(*res)
        _note("needle_prefill_causal", *r)
        return r
    _sweep(333, 32, run)


def test_needle_sweep_paged_prefill():
    """CTA-pair shape (G 4), 16-token pages, 128 new tokens over 300 cached keys."""
    _sweep(300, 32, lambda nd: _paged_prefill("needle_prefill_paged", 64, 16, 128, 4, 4, 128, [300] * 8,
                                              torch.bfloat16, (), needles=nd))


def test_needle_sweep_varlen():
    q_lens, lens = [128, 37, 200, 1, 64, 5, 99, 150], [300, 300, 300, 300, 300, 300, 300, 300]
    _sweep(300, 32, lambda nd: _varlen("needle_prefill_varlen", 65, 16, 128, 4, 2, q_lens, lens, torch.bfloat16, (),
                                       needles=nd))


# ---------------------------------------------------------------------------------------------------------------------
# zero-length sequences in a one-token decode batch
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,splits,G,lens", [
    (torch.bfloat16, 1, 4, [300, 0, 17]),                    # TMA, direct output
    (torch.bfloat16, 3, 4, [2000, 0, 700, 0]),               # fused merge
    (torch.bfloat16, 4, 4, [3000, 0, 1500]),                 # one cluster per unit
    (torch.bfloat16, 32, 4, [9000, 0, 4000]),                # clusters, then partials
    (torch.float32, 3, 2, [300, 0, 77]),                     # SIMT + combine
])
def test_zero_length_decode_sequence(dtype, splits, G, lens):
    p = torch.float32 if dtype == torch.float32 else None
    _paged_decode("decode_zero_length", 70 + splits, 16, 128 if dtype != torch.float32 else 64, 2, G, lens, dtype,
                  splits, p_dtype=p)


def test_zero_length_decode_sequence_two_pass():
    B, Hkv, G, D, bs, splits = 3, 2, 4, 128, 16, 3
    lens = [1000, 0, 64]
    Hq = Hkv * G
    bt = Batch(75, B, Hkv, lens, D, torch.bfloat16, ro.PROFILES, D ** -0.5)
    kp, vp, table = bt.pools(bs)
    q, t = _q((B, Hq), D, ro.RAMP_T, torch.bfloat16)
    lens_t = torch.tensor(lens, dtype=torch.int32).cuda()
    lib = _lib.load()
    ws = torch.empty(int(lib.pli_decode_workspace_bytes(B, Hq, D, splits)) // 4, dtype=torch.float32, device="cuda")
    o = torch.full((B, Hq, D), float("nan"), device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(B, Hq, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pli_decode_splitkv(q.data_ptr(), kp.data_ptr(), vp.data_ptr(), table.data_ptr(), lens_t.data_ptr(),
                                      B, Hq, Hkv, D, max(lens), bs, table.stride(0), 0, kp.shape[0],
                                      _lib.i64(q.stride(0), q.stride(1)), _lib.i64(*kp.stride()[:4]), D ** -0.5,
                                      _lib.dtype_code(q.dtype), splits, ws.data_ptr(), ws.numel() * 4, stream))
    _lib.check(lib.pli_decode_combine(ws.data_ptr(), o.data_ptr(), lse.data_ptr(), B, Hq, D, splits,
                                      _lib.i64(o.stride(0), o.stride(1)), _lib.dtype_code(q.dtype), stream))
    torch.cuda.synchronize()
    _decode("decode_zero_length_two_pass", bt, q, t, o, lse, 1)
