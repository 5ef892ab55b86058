"""Decode-time attention over the ch02 contiguous cache or the ch07 paged pools.

The reference computes this inside `CachedGQA.forward` (ch02/cached_generation.py:72-94: slice the
cache to seq_len, transpose, repeat_interleave K/V G times, QK^T/sqrt(D), no mask when one new
token, softmax, PV).  `flash_decode` is that attention block for one query token per sequence as a
split-KV kernel + log-sum-exp combine, reading K/V in place:

  contiguous  k_cache, v_cache (B, max_seq_len, Hkv, D)            ch02/kv_cache.py:25-34
  paged       k_cache, v_cache (P, num_layers, bs, Hkv, D) pools   ch07/paged_memory.py:38-48
              + block_tables (B, max_pages) int32: token t of sequence b is at
                page block_tables[b, t // bs], slot t % bs          ch07/paged_memory.py:54,84-86
"""
from __future__ import annotations

import torch

from . import _lib
from .kv_cache import KVCache, LayerKVCache
from .paged_memory import PagedKVCache


def decode_num_splits(B: int, Hkv: int, max_seq_len: int, *, group: int = 1, q_len: int = 1) -> int:
    """The library's split count; with q_len > 1 tokens per sequence (group = Hq / Hkv) the one pli_decode_fwd_multi
    picks (pli_decode_num_splits_multi)."""
    if q_len > 1:
        return int(_lib.load().pli_decode_num_splits_multi(B, group * Hkv, Hkv, q_len, max_seq_len))
    return int(_lib.load().pli_decode_num_splits(B, Hkv, max_seq_len))


def decode_workspace(B: int, Hq: int, D: int, num_splits: int, device) -> torch.Tensor:
    nbytes = int(_lib.load().pli_decode_workspace_bytes(B, Hq, D, num_splits))
    return torch.empty(nbytes // 4, dtype=torch.float32, device=device)


def _storage(q_dtype, B, Hq, D, k_cache, v_cache, seq_lens, block_tables, layer, max_seq_len, validate, scale,
             q_len: int = 1):
    """Checks and marshalling of the KV storage, lengths and scale shared by the one- and multi-token calls."""
    lo = q_len if q_len > 1 else 0         # smallest length validate=True accepts
    if not (q_dtype == k_cache.dtype == v_cache.dtype):
        raise RuntimeError(f"q and the KV storage must share a dtype; got {q_dtype}, {k_cache.dtype}, {v_cache.dtype}")
    if k_cache.shape != v_cache.shape or k_cache.stride() != v_cache.stride():
        raise RuntimeError("k and v storage must have the same shape and strides")
    if k_cache.stride(-1) != 1:
        raise RuntimeError("KV storage must have a unit head_dim stride")
    paged = block_tables is not None
    if paged:
        if k_cache.dim() != 5:
            raise RuntimeError(f"paged pools must be (P, layers, bs, Hkv, D); got {tuple(k_cache.shape)}")
        P, n_layers, bs, Hkv, Dk = k_cache.shape
        if not 0 <= layer < n_layers:
            raise IndexError(f"layer {layer} out of range for {n_layers} layers")
        if block_tables.dtype != torch.int32 or not block_tables.is_cuda or block_tables.dim() != 2:
            raise RuntimeError("block_tables must be a 2-D CUDA int32 tensor")
        if block_tables.shape[0] != B:
            raise RuntimeError(f"block_tables has {block_tables.shape[0]} rows for batch {B}")
        if block_tables.stride(-1) != 1:
            block_tables = block_tables.contiguous()
        kv_strides = k_cache.stride()[:4]
        kv_extent, cap = P, block_tables.shape[1] * bs
        table_ptr, tstride = block_tables.data_ptr(), block_tables.stride(0)
    else:
        if k_cache.dim() != 4:
            raise RuntimeError(f"contiguous cache must be (B, max_seq_len, Hkv, D); got {tuple(k_cache.shape)}")
        Bk, cap, Hkv, Dk = k_cache.shape
        if Bk != B:
            raise RuntimeError(f"cache batch {Bk} does not match q batch {B}")
        bs = 0
        kv_strides = (k_cache.stride(0), 0, k_cache.stride(1), k_cache.stride(2))
        kv_extent = B
        table_ptr, tstride = None, 0
    if Dk != D:
        raise RuntimeError(f"head_dim mismatch: q {D}, cache {Dk}")
    if Hq % Hkv != 0:
        raise RuntimeError(f"num_heads ({Hq}) must be a multiple of num_kv_heads ({Hkv})")

    if isinstance(seq_lens, int):
        if not 0 < seq_lens <= cap or seq_lens < q_len:
            raise ValueError(f"seq_len {seq_lens} outside ({lo}, {cap}]" if q_len == 1 else
                             f"seq_len {seq_lens} outside [{q_len}, {cap}]: it counts the {q_len} new tokens")
        lens = torch.full((B,), seq_lens, dtype=torch.int32, device=k_cache.device)
        if max_seq_len is None:
            max_seq_len = seq_lens
    else:
        lens = seq_lens
        if lens.dtype != torch.int32 or not lens.is_cuda or lens.shape != (B,):
            raise RuntimeError("seq_lens must be an int or a (B,) CUDA int32 tensor")
        if not lens.is_contiguous():
            lens = lens.contiguous()
        if max_seq_len is None:
            max_seq_len = cap
    max_seq_len = min(int(max_seq_len), cap)
    if validate:        # opt-in, one synchronising copy: the device-side preconditions (see validate_paged_args)
        from .flash_attention import validate_paged_args
        if paged:
            validate_paged_args(lens, block_tables, bs, P, q_lens=q_len if q_len > 1 else None, min_len=0,
                                max_seq_len=max_seq_len)
        elif int(lens.max()) > max_seq_len or int(lens.min()) < lo:
            raise ValueError(f"seq_lens outside [{lo}, {max_seq_len}]")
    if scale is None:
        scale = D ** -0.5
    return Hkv, lens, block_tables, bs, kv_strides, kv_extent, table_ptr, tstride, max_seq_len, scale


def _prepare_decode(
    q: torch.Tensor,
    k_cache: torch.Tensor,
    v_cache: torch.Tensor,
    seq_lens,
    *,
    block_tables: torch.Tensor | None = None,
    layer: int = 0,
    scale: float | None = None,
    return_lse: bool = False,
    num_splits: int | None = None,
    max_seq_len: int | None = None,
    workspace: torch.Tensor | None = None,
    out: torch.Tensor | None = None,
    peer_out=None,
    validate: bool = False,
):
    """Attention of the newest query token(s) of each sequence over cached K/V.

    q         (B, Hq, 1, D) or (B, Hq, D); or (B, Hq, Nq, D) with 2 <= Nq <= 16 new tokens per sequence (the verify
              step of speculative decoding), attended in ONE launch: query i sees key j iff j <= i + seq_lens[b] - Nq
              (ch02/cached_generation.py:85-91), so seq_lens counts the Nq new tokens and must be >= Nq
    seq_lens  int (one length for the whole batch, like the reference's caches) or (B,) int32 CUDA
              tensor (ragged batch; no host sync is made to read it)
    max_seq_len  host upper bound of seq_lens, used to pick the split count; defaults to the int
              seq_lens, else the cache length (contiguous) / table width * page size (paged)
    validate  opt-in host check (one sync) of seq_lens / block-table ranges; off by default (no host sync)
    peer_out  a `sharding.PeerOutput` (one query token only): q / caches are this rank's head shard; the kernel stores
              the shard's output into EVERY rank's full (B_total, Hq_total, D) buffer over NVLink and the call returns
              that full tensor once all ranks' slices have landed (fused all-gather, no NCCL call).
    Returns o shaped like q (and lse (B, Hq) float32 when return_lse; (B, Hq, Nq) for Nq > 1).
    """
    if not (q.is_cuda and k_cache.is_cuda and v_cache.is_cuda):
        raise RuntimeError("flash_decode runs on CUDA tensors only: there is no CPU fallback for the decode path")
    if q.dim() == 4 and q.shape[2] != 1:
        if not 2 <= q.shape[2] <= 16:
            raise RuntimeError(f"decode takes 1 to 16 query tokens per sequence; got q {tuple(q.shape)} "
                               "(use flash_attention_forward(..., causal=True) or flash_attention_paged for chunks)")
        if peer_out is not None:
            raise RuntimeError("peer_out takes one query token per sequence")
        return _prepare_decode_multi(q, k_cache, v_cache, seq_lens, block_tables=block_tables, layer=layer, scale=scale,
                                     return_lse=return_lse, num_splits=num_splits, max_seq_len=max_seq_len,
                                     workspace=workspace, out=out, validate=validate)
    if q.dim() == 4:
        q3 = q[:, :, 0, :]
    elif q.dim() == 3:
        q3 = q
    else:
        raise RuntimeError(f"q must be (B, Hq, 1, D) or (B, Hq, D); got {tuple(q.shape)}")
    if q3.stride(-1) != 1:
        q3 = q3.contiguous()
    B, Hq, D = q3.shape
    dev = q.device
    st = _storage(q.dtype, B, Hq, D, k_cache, v_cache, seq_lens, block_tables, layer, max_seq_len, validate, scale)
    Hkv, lens, block_tables, bs, kv_strides, kv_extent, table_ptr, tstride, max_seq_len, scale = st

    lib = _lib.load()
    if num_splits is None:
        num_splits = int(lib.pli_decode_num_splits(B, Hkv, max_seq_len))
    need = int(lib.pli_decode_workspace_bytes(B, Hq, D, num_splits))
    if workspace is None:
        workspace = torch.empty(need // 4, dtype=torch.float32, device=dev)
    elif workspace.numel() * workspace.element_size() < need or not workspace.is_cuda:
        raise RuntimeError(f"workspace too small: need {need} bytes")
    lse = torch.empty((B, Hq), dtype=torch.float32, device=dev) if return_lse else None
    lse_ptr = lse.data_ptr() if lse is not None else None
    ws_bytes = workspace.numel() * workspace.element_size()
    keep = (q3, k_cache, v_cache, block_tables, lens, workspace, lse)       # the launch only holds raw pointers
    if peer_out is not None:
        import ctypes
        sh = peer_out.shard
        Bt, Ht, Dt = peer_out.shape
        if (B, Hq, D) != (sh.b_end - sh.b_start, sh.q_end - sh.q_start, Dt) or peer_out.dtype != q3.dtype:
            raise RuntimeError(f"local decode shape {(B, Hq, D)} / dtype does not match the PeerOutput shard")
        ps = _lib.PeerScatter()
        ps.n_peers, ps.rank = sh.world_size, sh.rank
        for r in range(sh.world_size):
            ps.peer_o[r] = peer_out.output_ptrs[r]
            ps.peer_flags[r] = peer_out.flag_ptrs[r]
        ps.epoch = peer_out.epoch_ptr
        ps.slice_offset = peer_out.slice_offset
        # one launch and one buffer when the TMA kernel serves the call (pli_decode_fwd_gather), else two of each
        st_i64 = _lib.i64(*kv_strides)
        gather = scale > 0 and q3.stride(0) % 2 == 0 and q3.stride(1) % 2 == 0 and q3.data_ptr() % 4 == 0 and \
            lib.pli_decode_kernel_kind(D, _lib.dtype_code(q3.dtype), bs, st_i64, k_cache.data_ptr(),
                                       v_cache.data_ptr()) == _lib.PLI_KIND_MMA_TMA
        peer_out.use_mode("gather" if gather else "scatter")
        ps.buffer_stride = 0 if gather else peer_out.buffer_stride
        for r in range(sh.world_size):
            ps.peer_ready[r] = peer_out.ready_ptrs[r]
        ps.cta_counter = peer_out.cta_counter_ptr
        ps_ref = ctypes.byref(ps)
        args = (q3.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), table_ptr, lens.data_ptr(), lse_ptr, B, Hq, Hkv, D,
                max_seq_len, bs, tstride, layer, kv_extent, _lib.i64(q3.stride(0), q3.stride(1)), _lib.i64(*kv_strides),
                _lib.i64(Ht * Dt, Dt), float(scale), _lib.dtype_code(q3.dtype), num_splits, workspace.data_ptr(), ws_bytes,
                ps_ref)
        return _Prepared(dev, "gather" if gather else "scatter", args, keep + (ps,), None, lse, peer_out, ps, q.dim() == 4)
    if out is None:
        out = torch.empty((B, Hq, D), dtype=q.dtype, device=dev)
    elif out.shape != (B, Hq, D) or out.dtype != q.dtype or out.stride(-1) != 1:
        raise RuntimeError("out must be (B, Hq, D), q's dtype, unit inner stride")
    args = (q3.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), table_ptr, lens.data_ptr(), out.data_ptr(), lse_ptr,
            B, Hq, Hkv, D, max_seq_len, bs, tstride, layer, kv_extent, _lib.i64(q3.stride(0), q3.stride(1)),
            _lib.i64(*kv_strides), _lib.i64(out.stride(0), out.stride(1)), float(scale), _lib.dtype_code(q.dtype),
            num_splits, workspace.data_ptr(), ws_bytes)
    return _Prepared(dev, "", args, keep, out, lse, None, None, q.dim() == 4)


def _prepare_decode_multi(q, k_cache, v_cache, seq_lens, *, block_tables, layer, scale, return_lse, num_splits,
                          max_seq_len, workspace, out, validate):
    """`_prepare_decode` for q (B, Hq, Nq, D), 2 <= Nq <= 16: one `pli_decode_fwd_multi` launch."""
    B, Hq, Nq, D = q.shape
    # q is read through its own strides (e.g. the (B, Nq, Hq, D).transpose(1, 2) view of a projection), never copied:
    # a DecodePlan re-reads the caller's q at every call and graph replay
    if q.stride(-1) != 1:
        raise RuntimeError("q must have a unit head_dim stride")
    dev = q.device
    st = _storage(q.dtype, B, Hq, D, k_cache, v_cache, seq_lens, block_tables, layer, max_seq_len, validate, scale, Nq)
    Hkv, lens, block_tables, bs, kv_strides, kv_extent, table_ptr, tstride, max_seq_len, scale = st
    lib = _lib.load()
    if num_splits is None:
        num_splits = decode_num_splits(B, Hkv, max_seq_len, group=Hq // Hkv, q_len=Nq)
    need = int(lib.pli_decode_workspace_bytes(B, Hq * Nq, D, num_splits))
    if workspace is None:
        workspace = torch.empty(need // 4, dtype=torch.float32, device=dev)
    elif workspace.numel() * workspace.element_size() < need or not workspace.is_cuda:
        raise RuntimeError(f"workspace too small: need {need} bytes")
    if out is None:
        out = torch.empty((B, Hq, Nq, D), dtype=q.dtype, device=dev)
    elif out.shape != (B, Hq, Nq, D) or out.dtype != q.dtype or out.stride(-1) != 1 or \
            (Hq > 1 and out.stride(1) != Nq * out.stride(2)):
        raise RuntimeError(f"out must be ({B}, {Hq}, {Nq}, {D}), q's dtype, contiguous in its last three dimensions")
    lse = torch.empty((B, Hq, Nq), dtype=torch.float32, device=dev) if return_lse else None
    keep = (q, k_cache, v_cache, block_tables, lens, workspace, lse)
    args = (q.data_ptr(), k_cache.data_ptr(), v_cache.data_ptr(), table_ptr, lens.data_ptr(), out.data_ptr(),
            lse.data_ptr() if lse is not None else None, B, Hq, Hkv, Nq, D, max_seq_len, bs, tstride, layer, kv_extent,
            _lib.i64(*q.stride()[:3]), _lib.i64(*kv_strides), _lib.i64(*out.stride()[:3]), float(scale),
            _lib.dtype_code(q.dtype), num_splits, workspace.data_ptr(), workspace.numel() * workspace.element_size())
    return _Prepared(dev, "", args, keep, out, lse, None, None, False, multi=True)


class _Prepared:
    """A validated, marshalled decode call: everything but the stream."""
    __slots__ = ("dev", "scatter", "args", "keep", "out", "lse", "peer_out", "ps", "four_d", "lib", "fwd")

    def __init__(self, dev, scatter, args, keep, out, lse, peer_out, ps, four_d, multi=False):
        self.dev, self.scatter, self.args, self.keep = dev, scatter, args, keep
        self.out, self.lse, self.peer_out, self.ps, self.four_d = out, lse, peer_out, ps, four_d
        self.lib = _lib.load()
        self.fwd = self.lib.pli_decode_fwd_multi if multi else self.lib.pli_decode_fwd

    def launch(self):
        with _lib.on_device(self.dev):
            stream = _lib.current_stream_ptr(self.dev)
            if self.scatter:
                import ctypes
                if self.scatter == "gather":
                    _lib.check(self.lib.pli_decode_fwd_gather(*self.args, stream))
                else:
                    _lib.check(self.lib.pli_decode_fwd_scatter(*self.args, stream))
                    _lib.check(self.lib.pli_peer_publish_wait(ctypes.byref(self.ps), stream))
                # eager: the buffer of this step; under stream capture (nothing ran yet): the fixed `stable` tensor the
                # captured step copies into — the caller accounts for replays with peer_out.advance(n)
                o = self.peer_out.finish_step(self.ps, stream)
            else:
                _lib.check(self.fwd(*self.args, stream))
                o = self.out.unsqueeze(2) if self.four_d else self.out
        return (o, self.lse) if self.lse is not None else o


def flash_decode(q, k_cache, v_cache, seq_lens, *, block_tables=None, layer: int = 0, scale: float | None = None,
                 return_lse: bool = False, num_splits: int | None = None, max_seq_len: int | None = None,
                 workspace: torch.Tensor | None = None, out: torch.Tensor | None = None, peer_out=None,
                 validate: bool = False):
    return _prepare_decode(q, k_cache, v_cache, seq_lens, block_tables=block_tables, layer=layer, scale=scale,
                           return_lse=return_lse, num_splits=num_splits, max_seq_len=max_seq_len, workspace=workspace,
                           out=out, peer_out=peer_out, validate=validate).launch()


flash_decode.__doc__ = _prepare_decode.__doc__


class DecodePlan:
    """`flash_decode` with the validation and argument marshalling done ONCE: `plan = DecodePlan(q, k_cache, v_cache,
    seq_lens, block_tables=..., out=..., ...)`, then `plan()` per step launches on the current stream with the same
    buffers (new queries / lengths are written into them in place, as a CUDA-graph runner does).  A decode step of a few
    tens of microseconds is otherwise bound by the ~30 us the Python wrapper spends per call; a plan call costs a few.
    Same arguments and results as `flash_decode`."""

    def __init__(self, q, k_cache, v_cache, seq_lens, **kw):
        if isinstance(seq_lens, int):
            raise TypeError("a plan needs seq_lens as a (B,) CUDA int32 tensor (it is read on the device at every step)")
        self._prep = _prepare_decode(q, k_cache, v_cache, seq_lens, **kw)

    def __call__(self):
        return self._prep.launch()


def decode_kernel_kind(k_cache: torch.Tensor, block_tables=None) -> str:
    """'mma_tma' or 'simt': which split-KV kernel serves this storage."""
    if block_tables is not None:
        bs, st = k_cache.shape[2], k_cache.stride()[:4]
    else:
        bs, st = 0, (k_cache.stride(0), 0, k_cache.stride(1), k_cache.stride(2))
    kind = _lib.load().pli_decode_kernel_kind(k_cache.shape[-1], _lib.dtype_code(k_cache.dtype), bs, _lib.i64(*st),
                                              k_cache.data_ptr(), k_cache.data_ptr())
    return _lib.KIND_NAMES[kind]


def decode_with_cache(q: torch.Tensor, cache, **kw):
    """flash_decode over a reference-style `KVCache` (ch02/kv_cache.py) or `LayerKVCache`
    (ch02/cached_generation.py) object: attends to the first cache.seq_len tokens."""
    if isinstance(cache, KVCache) or hasattr(cache, "k_cache"):
        k, v = cache.k_cache, cache.v_cache
    elif isinstance(cache, LayerKVCache) or hasattr(cache, "k"):
        k, v = cache.k, cache.v
    else:
        raise TypeError(f"unsupported cache object {type(cache)}")
    return flash_decode(q, k, v, int(cache.seq_len), **kw)


def decode_with_paged(q: torch.Tensor, paged: PagedKVCache, request_ids, *, layer: int = 0, **kw):
    """flash_decode over a `PagedKVCache` (ch07/paged_memory.py) for the given request ids."""
    if paged.k_cache is None:
        raise RuntimeError("PagedKVCache has no device pools (constructed without CUDA)")
    bt, lens = paged.block_table_tensor(request_ids, device=q.device)
    max_len = max(paged.block_tables[r].num_tokens for r in request_ids)
    return flash_decode(q, paged.k_cache, paged.v_cache, lens, block_tables=bt, layer=layer, max_seq_len=max_len, **kw)


def prefill_with_paged(q: torch.Tensor, paged: PagedKVCache, request_ids, *, layer: int = 0, **kw):
    """Chunked prefill (q (B, Hq, Nq, D), Nq >= 1 newest tokens) over a `PagedKVCache` for the given request ids:
    `flash_attention_paged` with the block tables / lengths taken from the allocator mirror."""
    from .flash_attention import flash_attention_paged
    if paged.k_cache is None:
        raise RuntimeError("PagedKVCache has no device pools (constructed without CUDA)")
    bt, lens = paged.block_table_tensor(request_ids, device=q.device)
    max_len = max(paged.block_tables[r].num_tokens for r in request_ids)
    return flash_attention_paged(q, paged.k_cache, paged.v_cache, bt, lens, layer=layer, max_seq_len=max_len, **kw)


def mixed_batch_attention(q: torch.Tensor, paged: PagedKVCache, prefill_ids, prefill_lens, decode_ids, *,
                          layer: int = 0, scale: float | None = None) -> torch.Tensor:
    """Attention of one mixed prefill/decode step (`MixedBatch` of ch08/mixed_batch.py:19-31: `prefill_requests`
    bringing `prompt_len`/chunk tokens each, `decode_requests` bringing one) over a `PagedKVCache` whose pages
    already hold this step's K/V.

    q (prefill_tokens + len(decode_ids), Hq, D): the prefill requests' new tokens in request order, then one row per
    decode request.  Two launches: the ragged prefill kernel for the prefill rows, the split-KV decode kernel
    (writing straight into the packed output) for the decode rows.  Returns o shaped like q."""
    from .flash_attention import flash_attention_varlen_paged
    if paged.k_cache is None:
        raise RuntimeError("PagedKVCache has no device pools (constructed without CUDA)")
    prefill_ids, decode_ids = list(prefill_ids), list(decode_ids)
    prefill_lens = [int(n) for n in prefill_lens]
    if len(prefill_lens) != len(prefill_ids):
        raise ValueError("one length per prefill request")
    tp = sum(prefill_lens)
    if q.dim() != 3 or q.shape[0] != tp + len(decode_ids):
        raise RuntimeError(f"q must be ({tp + len(decode_ids)}, Hq, D); got {tuple(q.shape)}")
    for r, n in zip(prefill_ids, prefill_lens):
        if not 0 < n <= paged.block_tables[r].num_tokens:
            raise ValueError(f"request {r}: {n} new tokens but {paged.block_tables[r].num_tokens} cached")
    out = torch.empty((q.shape[0], q.shape[1], q.shape[2]), dtype=q.dtype, device=q.device)
    if prefill_ids:
        bt, lens = paged.block_table_tensor(prefill_ids, device=q.device)
        cu = torch.tensor([0] + prefill_lens, dtype=torch.int32).cumsum(0, dtype=torch.int32).to(q.device)
        max_len = max(paged.block_tables[r].num_tokens for r in prefill_ids)
        out[:tp] = flash_attention_varlen_paged(q[:tp], paged.k_cache, paged.v_cache, bt, lens, cu, max(prefill_lens),
                                                layer=layer, scale=scale, max_seq_len=max_len)
    if decode_ids:
        decode_with_paged(q[tp:], paged, decode_ids, layer=layer, scale=scale, out=out[tp:])
    return out


def paged_gather(store: torch.Tensor, block_tables: torch.Tensor, seq_lens: torch.Tensor, max_len: int,
                 layer: int = 0) -> torch.Tensor:
    """Gather one layer of a paged pool to (B, max_len, Hkv, D) with the kernels' address rule
    (parity aid: lets tests assert page indexing bit-exactly; rows >= seq_len are zero)."""
    if store.dim() != 5 or not store.is_cuda:
        raise RuntimeError("store must be a CUDA pool (P, layers, bs, Hkv, D)")
    B = block_tables.shape[0]
    _, _, bs, Hkv, D = store.shape
    out = torch.empty((B, max_len, Hkv, D), dtype=store.dtype, device=store.device)
    lib = _lib.load()
    with _lib.on_device(store.device):
        rc = lib.pli_paged_gather(store.data_ptr(), out.data_ptr(), block_tables.data_ptr(), seq_lens.data_ptr(), B,
                                  max_len, Hkv, D, bs, block_tables.stride(0), layer, _lib.i64(*store.stride()[:4]),
                                  _lib.dtype_code(store.dtype), _lib.current_stream_ptr(store.device))
    _lib.check(rc)
    return out
