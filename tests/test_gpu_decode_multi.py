"""GPU tests of decode with 2-16 query tokens per sequence in one split-KV launch (pli_decode_fwd_multi): parity with the
CPU oracle's offset causal mask (ch02/cached_generation.py:85-91), the per-row mask at split / warp-step boundaries,
the SIMT path, dirty storage and workspace, CUDA graphs and the unchanged one-token path."""
import pytest
import torch

import physics_llm_inference_b200 as pli
from physics_llm_inference_b200 import _lib
from oracle import attention_oracle as orc

pytestmark = pytest.mark.gpu
TOL = {torch.float32: 1e-3, torch.bfloat16: 2e-2, torch.float16: 2e-2}
LSE_TOL = 1e-3


def _q(seed, B, Hq, Nq, D):
    return torch.randn(B, Hq, Nq, D, generator=torch.Generator().manual_seed(seed))


def _paged(seed, B, Hq, Hkv, Nq, D, bs, lens, dtype, n_layers=1):
    _, kp, vp, table, lens_t = orc.seeded_paged(seed, B, Hq, Hkv, D, bs, lens, num_layers=n_layers)
    return _q(seed + 1, B, Hq, Nq, D).to(dtype).cuda(), kp.to(dtype).cuda(), vp.to(dtype).cuda(), table, lens_t


def _contiguous(seed, B, Hq, Hkv, Nq, D, lens, dtype):
    g = torch.Generator().manual_seed(seed)
    L = max(lens) + 5
    kc = torch.randn(B, L, Hkv, D, generator=g).to(dtype).cuda()
    vc = torch.randn(B, L, Hkv, D, generator=g).to(dtype).cuda()
    return _q(seed + 1, B, Hq, Nq, D).to(dtype).cuda(), kc, vc, torch.tensor(lens, dtype=torch.int32)


def _check(o, lse, ro, rlse, dtype):
    assert not torch.isnan(o).any() and not torch.isnan(lse).any()
    eo = (o.float().cpu() - ro).abs().max().item()
    el = (lse.cpu() - rlse).abs().max().item()
    assert eo <= TOL[dtype] and el <= LSE_TOL, (eo, el)


def _run(q, kc, vc, table, lens_t, bs, dtype, layer=0, splits=None):
    """flash_decode + the oracle over paged pools (bs > 0) or the contiguous cache (bs == 0)."""
    if bs:
        o, lse = pli.flash_decode(q, kc, vc, lens_t.cuda(), block_tables=table.cuda(), layer=layer, return_lse=True,
                                  num_splits=splits, max_seq_len=int(lens_t.max()))
        ro, rlse = orc.paged_decode_oracle(q, kc, vc, table, lens_t, layer=layer)
    else:
        o, lse = pli.flash_decode(q, kc, vc, lens_t.cuda(), return_lse=True, num_splits=splits)
        ro, rlse = orc.cached_attention_oracle(q, kc, vc, lens_t)
    assert o.shape == q.shape and o.dtype == dtype and lse.shape == q.shape[:3]
    return o, lse, ro, rlse


STORAGE = [16, 32, 64, 128, 0]            # page sizes; 0 = the contiguous cache
SPLITS = [None, 1, 2, 3, 8, 37]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("D", [64, 128])
@pytest.mark.parametrize("G", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("Nq", [2, 3, 4, 5, 8, 16])
def test_multi_token_parity(Nq, G, D, dtype):
    """Every (dtype, D, G, Nq); storage and forced split count rotate over the cases so that each (G, Nq) pair meets
    several of them.  Ragged lengths include seq_lens[b] == Nq."""
    i = [2, 3, 4, 5, 8, 16].index(Nq) + 6 * [1, 2, 4, 8, 16].index(G) + 30 * (D == 128) + 60 * (dtype == torch.float16)
    bs, splits = STORAGE[i % 5], SPLITS[(i // 5 + i) % 6]
    Hkv = 2
    lens = [Nq, 300 + 7 * Nq, 64 + Nq - 1, 1000]
    if bs:
        q, kc, vc, table, lens_t = _paged(40 + i, len(lens), G * Hkv, Hkv, Nq, D, bs, lens, dtype, n_layers=2)
        assert pli.decode_kernel_kind(kc, table) == "mma_tma"
        o, lse, ro, rlse = _run(q, kc, vc, table, lens_t, bs, dtype, layer=1, splits=splits)
    else:
        q, kc, vc, lens_t = _contiguous(40 + i, len(lens), G * Hkv, Hkv, Nq, D, lens, dtype)
        o, lse, ro, rlse = _run(q, kc, vc, None, lens_t, 0, dtype, splits=splits)
    _check(o, lse, ro, rlse, dtype)


@pytest.mark.parametrize("bs", [16, 64, 0])
@pytest.mark.parametrize("Nq,splits", [(8, 2), (16, 2), (8, 3), (16, 8), (5, 37), (16, 1)])
def test_mask_at_split_and_warp_boundaries(Nq, splits, bs):
    """Lengths whose split boundaries (multiples of 64 tokens) and 16-token warp steps fall inside the last Nq - 1 keys:
    rows that see no key of a warp step, or of a whole split, must not produce NaN."""
    dtype, D, G, Hkv = torch.bfloat16, 128, 4, 2
    # split s covers [s * c, (s + 1) * c) with c = ceil(L / S) rounded up to 64: for L = 129, S = 2 the second split is
    # the single key 128, which rows i < Nq - 1 of the last split do not see
    lens = [129, 130, 136, 145, 64 * splits + 3, 16 * 9 + Nq // 2, Nq]
    if bs:
        q, kc, vc, table, lens_t = _paged(60 + Nq + splits, len(lens), G * Hkv, Hkv, Nq, D, bs, lens, dtype)
        o, lse, ro, rlse = _run(q, kc, vc, table, lens_t, bs, dtype, splits=splits)
    else:
        q, kc, vc, lens_t = _contiguous(60 + Nq + splits, len(lens), G * Hkv, Hkv, Nq, D, lens, dtype)
        o, lse, ro, rlse = _run(q, kc, vc, None, lens_t, 0, dtype, splits=splits)
    assert torch.isfinite(o.float()).all() and torch.isfinite(lse).all()
    _check(o, lse, ro, rlse, dtype)


@pytest.mark.parametrize("dtype,D,bs,splits", [(torch.float32, 128, 16, None), (torch.float32, 64, 32, 3),
                                               (torch.bfloat16, 48, 16, 2), (torch.float16, 128, 7, None),
                                               (torch.bfloat16, 64, 24, 37)])
def test_multi_token_simt_path(dtype, D, bs, splits):
    """f32 storage, a head dim other than 64 / 128, non-power-of-two pages: the SIMT kernel over virtual heads."""
    Nq, G, Hkv = 4, 4, 2
    lens = [Nq, 77, 130, 300]
    q, kc, vc, table, lens_t = _paged(80 + D + bs, len(lens), G * Hkv, Hkv, Nq, D, bs, lens, dtype, n_layers=2)
    assert pli.decode_kernel_kind(kc, table) == "simt"
    o, lse, ro, rlse = _run(q, kc, vc, table, lens_t, bs, dtype, layer=1, splits=splits)
    _check(o, lse, ro, rlse, dtype)
    qc, kcc, vcc, lc = _contiguous(81 + D, len(lens), G * Hkv, Hkv, Nq, D, lens, dtype)
    if D % 64 or dtype == torch.float32:
        o, lse, ro, rlse = _run(qc, kcc, vcc, None, lc, 0, dtype, splits=splits)
        _check(o, lse, ro, rlse, dtype)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_dirty_storage_past_seq_len(dtype):
    """NaN / Inf in every slot past seq_lens[b] changes no bit of O or LSE."""
    Nq, G, Hkv, D, bs = 4, 4, 2, 128, 16
    lens = [100, 37, Nq, 64]
    q, kd, vd, table, lens_t = _paged(90, len(lens), G * Hkv, Hkv, Nq, D, bs, lens, dtype)
    for splits in (None, 2, 3):
        o0, l0 = pli.flash_decode(q, kd, vd, lens_t.cuda(), block_tables=table.cuda(), return_lse=True, num_splits=splits)
        used = torch.zeros(kd.shape[0], bs, dtype=torch.bool)
        for b, L in enumerate(lens):
            for t in range(L):
                used[int(table[b, t // bs]), t % bs] = True
        k2, v2 = kd.clone(), vd.clone()
        k2[:, 0][~used.cuda()] = float("nan")
        v2[:, 0][~used.cuda()] = float("inf")
        o1, l1 = pli.flash_decode(q, k2, v2, lens_t.cuda(), block_tables=table.cuda(), return_lse=True, num_splits=splits)
        assert torch.equal(o0, o1) and torch.equal(l0, l1)


@pytest.mark.parametrize("splits", [3, 8, 16])
def test_dirty_workspace_fused_combine(splits):
    """A 0xFF-filled or reused workspace gives the bits of a fresh one (fused combine: unclustered, one cluster, two
    clusters per unit)."""
    Nq, G, Hkv, D, bs = 4, 4, 2, 128, 16
    lens = [2000, 1500, 700, Nq]
    q, kd, vd, table, lens_t = _paged(95, len(lens), G * Hkv, Hkv, Nq, D, bs, lens, torch.bfloat16)
    B, Hq = len(lens), G * Hkv
    kw = dict(block_tables=table.cuda(), return_lse=True, num_splits=splits)
    o0, l0 = pli.flash_decode(q, kd, vd, lens_t.cuda(), workspace=pli.decode_workspace(B, Hq * Nq, D, splits, "cuda"), **kw)
    ws = pli.decode_workspace(B, Hq * Nq, D, splits, "cuda")
    ws.view(torch.int32).fill_(-1)
    for _ in range(3):
        o1, l1 = pli.flash_decode(q, kd, vd, lens_t.cuda(), workspace=ws, **kw)
        assert torch.equal(o0, o1) and torch.equal(l0, l1)
    ro, rlse = orc.paged_decode_oracle(q, kd, vd, table, lens_t)
    _check(o0, l0, ro, rlse, torch.bfloat16)


def test_plan_in_cuda_graph_is_bit_identical():
    Nq, G, Hkv, D, bs = 4, 4, 8, 128, 16
    lens = [4096, 333, 1000, Nq]
    q, kd, vd, table, lens_t = _paged(100, len(lens), G * Hkv, Hkv, Nq, D, bs, lens, torch.bfloat16)
    out = torch.empty_like(q)
    for splits in (None, 3):
        plan = pli.DecodePlan(q, kd, vd, lens_t.cuda(), block_tables=table.cuda(), out=out, num_splits=splits,
                              max_seq_len=4096)
        o_eager = plan().clone()
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            plan()
            torch.cuda.synchronize()
            with torch.cuda.graph(g):
                plan()
        torch.cuda.current_stream().wait_stream(side)
        out.zero_()
        g.replay()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, o_eager)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_plan_reads_a_transposed_q_view_in_place(dtype):
    """q as the projection's (B, Nq, Hq, D).transpose(1, 2) view (head stride D, token stride Hq * D): a DecodePlan reads
    the caller's tensor at every call and graph replay, so writing new queries into it in place is seen."""
    Nq, G, Hkv, D, bs = 4, 4, 2, 128, 16
    Hq = G * Hkv
    lens = [300, 77, Nq]
    _, kd, vd, table, lens_t = _paged(120, len(lens), Hq, Hkv, Nq, D, bs, lens, dtype)
    x = torch.randn(len(lens), Nq, Hq, D, generator=torch.Generator().manual_seed(121)).to(dtype).cuda()
    q = x.transpose(1, 2)
    assert q.stride(1) == D and q.stride(2) == Hq * D
    plan = pli.DecodePlan(q, kd, vd, lens_t.cuda(), block_tables=table.cuda(), max_seq_len=max(lens))
    kinds = {pli.decode_kernel_kind(kd, table)}
    assert kinds == {"mma_tma" if dtype == torch.bfloat16 else "simt"}
    o = plan().clone()
    assert torch.equal(o, pli.flash_decode(q.contiguous(), kd, vd, lens_t.cuda(), block_tables=table.cuda(),
                                           max_seq_len=max(lens)))
    ro, _ = orc.paged_decode_oracle(q, kd, vd, table, lens_t)
    assert (o.float().cpu() - ro).abs().max().item() <= TOL[dtype]
    x.copy_(torch.randn(x.shape, generator=torch.Generator().manual_seed(122)).to(dtype))      # new queries, in place
    ref = pli.flash_decode(q.contiguous(), kd, vd, lens_t.cuda(), block_tables=table.cuda(), max_seq_len=max(lens))
    assert torch.equal(plan(), ref)
    out = plan._prep.out
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        plan()
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            plan()
    torch.cuda.current_stream().wait_stream(side)
    x.copy_(torch.randn(x.shape, generator=torch.Generator().manual_seed(123)).to(dtype))
    g.replay()
    torch.cuda.synchronize()
    ref = pli.flash_decode(q.contiguous(), kd, vd, lens_t.cuda(), block_tables=table.cuda(), max_seq_len=max(lens))
    assert torch.equal(out, ref)


@pytest.mark.parametrize("paged", [True, False])
def test_graph_runner_verify_step(paged):
    """DecodeGraphRunner(tokens_per_step=4): append 4 tokens per sequence and attend them in one captured launch,
    against the same eager kv_append + flash_decode."""
    k, B, Hq, Hkv, D = 4, 3, 16, 4, 128
    g = torch.Generator().manual_seed(105)
    start = torch.tensor([50, 200, 0], dtype=torch.int32)
    if paged:
        bs, P, pages = 16, 64, 16
        k_cache = torch.randn(P, 1, bs, Hkv, D, generator=g).bfloat16().cuda()
        table = torch.randperm(P, generator=g)[:B * pages].view(B, pages).to(torch.int32).cuda()
    else:
        k_cache = torch.randn(B, 256, Hkv, D, generator=g).bfloat16().cuda()
        table = None
    v_cache = torch.randn(k_cache.shape, generator=g).bfloat16().cuda()
    k_ref, v_ref = k_cache.clone(), v_cache.clone()
    runner = pli.DecodeGraphRunner(k_cache, v_cache, Hq, block_tables=table, tokens_per_step=k)
    assert runner.capture(start.cuda())
    lens = start.clone()
    for step in range(3):
        q = torch.randn(B, Hq, k, D, generator=g).bfloat16().cuda()
        kn = torch.randn(B, k, Hkv, D, generator=g).bfloat16().cuda()
        vn = torch.randn(B, k, Hkv, D, generator=g).bfloat16().cuda()
        o = runner.run(q, kn, vn)
        pli.kv_append(k_ref, v_ref, kn, vn, lens.cuda(), block_tables=table)
        lens += k
        ref = pli.flash_decode(q, k_ref, v_ref, lens.cuda(), block_tables=table, num_splits=runner.num_splits,
                               max_seq_len=runner.capacity)
        assert o.shape == (B, Hq, k, D)
        assert torch.equal(o, ref), step
        runner.seq_lens.copy_(lens.cuda())
        if paged:
            ro, _ = orc.paged_decode_oracle(q, k_ref, v_ref, table.cpu(), lens)
        else:
            ro, _ = orc.cached_attention_oracle(q, k_ref, v_ref, lens)
        assert (o.float().cpu() - ro).abs().max().item() <= 2e-2


def test_one_token_4d_matches_3d_and_rejections_launch_nothing():
    G, Hkv, D, bs = 4, 2, 128, 16
    lens = [300, 17, 1]
    q, kd, vd, table, lens_t = _paged(110, len(lens), G * Hkv, Hkv, 1, D, bs, lens, torch.bfloat16)
    kw = dict(block_tables=table.cuda(), return_lse=True)
    o4, l4 = pli.flash_decode(q, kd, vd, lens_t.cuda(), **kw)
    o3, l3 = pli.flash_decode(q[:, :, 0], kd, vd, lens_t.cuda(), **kw)
    assert o4.shape == q.shape and l4.shape == (len(lens), G * Hkv)
    assert torch.equal(o4[:, :, 0], o3) and torch.equal(l4, l3)

    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    q17 = torch.zeros(3, G * Hkv, 17, D, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError, match="flash_attention_paged"):
        pli.flash_decode(q17, kd, vd, lens_t.cuda(), block_tables=table.cuda())
    q4 = torch.zeros(3, G * Hkv, 4, D, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError, match="peer_out"):
        pli.flash_decode(q4, kd, vd, lens_t.cuda(), block_tables=table.cuda(), peer_out=object())
    with pytest.raises(ValueError):                       # seq_lens[2] = 1 < Nq = 4
        pli.flash_decode(q4, kd, vd, lens_t.cuda(), block_tables=table.cuda(), validate=True)
    kc = torch.zeros(3, 64, Hkv, D, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        pli.flash_decode(q4, kc, kc, 3)
    with pytest.raises(ValueError):
        pli.flash_decode(q4, kc, kc, torch.tensor([5, 3, 9], dtype=torch.int32, device="cuda"), validate=True)
    with pytest.raises(RuntimeError, match="out must be"):
        pli.flash_decode(q4, kc, kc, 8, out=torch.empty(3, G * Hkv, 4, D, device="cuda", dtype=torch.bfloat16)[:, :, :2])
    assert _lib.launch_count() == n0


def test_c3_shape_four_tokens_at_size():
    """C3 (B64, ctx 4096, 32q/8kv, D128, 16-token pages) with Nq = 4: sampled sequences against the oracle."""
    B, Hq, Hkv, D, bs, L, Nq = 64, 32, 8, 128, 16, 4096, 4
    pages_per = L // bs
    P = B * pages_per + 5
    g = torch.Generator(device="cuda").manual_seed(115)
    kp = torch.randn(P, 1, bs, Hkv, D, device="cuda", generator=g).bfloat16()
    vp = torch.randn(P, 1, bs, Hkv, D, device="cuda", generator=g).bfloat16()
    q = torch.randn(B, Hq, Nq, D, device="cuda", generator=g).bfloat16()
    table = torch.randperm(P, generator=torch.Generator().manual_seed(116))[:B * pages_per].to(torch.int32)
    table = table.view(B, pages_per).cuda()
    lens = torch.full((B,), L, dtype=torch.int32, device="cuda")
    lens[17] = L - 5
    o, lse = pli.flash_decode(q, kp, vp, lens, block_tables=table, return_lse=True, max_seq_len=L)
    kc, vc = kp.cpu(), vp.cpu()
    for b in (0, 17, 63):
        ro, rlse = orc.paged_decode_oracle(q[b:b + 1], kc, vc, table[b:b + 1].cpu(), [int(lens[b])])
        _check(o[b:b + 1], lse[b:b + 1], ro, rlse, torch.bfloat16)
