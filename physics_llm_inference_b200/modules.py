"""Callers of the hot path (SURVEY.md §8(f) F2/F4): the reference's GQA blocks and a CUDA-graph decode
step, with the attention core routed to the sm_100a kernels.

  GroupedQueryAttention   ch01/gqa.py:8-43            same ctor / forward(x, causal=True)
  CachedGQA               ch02/cached_generation.py:36-98   same ctor / forward(x, cache, start_pos)
  DecodeGraphRunner       ch08/cuda_graph.py:18-82 pattern around kv_append + flash_decode

The projections stay `nn.Linear` (dense GEMMs are not this path); what changes is that K/V are never
expanded with `repeat_interleave` (ch01/gqa.py:30-31), the N x N score matrix is never materialised
(ch01/gqa.py:32-36) and the (B,N,H,D)->(B,H,N,D) transposes (ch01/gqa.py:27-29) are only strides.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .decode import decode_num_splits, decode_workspace, flash_decode
from .flash_attention import flash_attention_forward
from .kv_cache import LayerKVCache, kv_append


class GroupedQueryAttention(nn.Module):
    def __init__(self, hidden_dim: int, num_heads: int, num_kv_heads: int):
        super().__init__()
        assert num_heads % num_kv_heads == 0
        self.num_heads = num_heads
        self.num_kv_heads = num_kv_heads
        self.num_groups = num_heads // num_kv_heads
        self.head_dim = hidden_dim // num_heads
        self.hidden_dim = hidden_dim
        self.q_proj = nn.Linear(hidden_dim, num_heads * self.head_dim, bias=False)
        self.k_proj = nn.Linear(hidden_dim, num_kv_heads * self.head_dim, bias=False)
        self.v_proj = nn.Linear(hidden_dim, num_kv_heads * self.head_dim, bias=False)
        self.o_proj = nn.Linear(hidden_dim, hidden_dim, bias=False)

    def forward(self, x: torch.Tensor, causal: bool = True) -> torch.Tensor:
        batch, seq_len, _ = x.shape
        q = self.q_proj(x).view(batch, seq_len, self.num_heads, self.head_dim).transpose(1, 2)
        k = self.k_proj(x).view(batch, seq_len, self.num_kv_heads, self.head_dim).transpose(1, 2)
        v = self.v_proj(x).view(batch, seq_len, self.num_kv_heads, self.head_dim).transpose(1, 2)
        attn_output = flash_attention_forward(q, k, v, causal=causal)        # (B, H, N, D), strides of q
        attn_output = attn_output.transpose(1, 2).reshape(batch, seq_len, self.hidden_dim)
        return self.o_proj(attn_output)

    def kv_cache_size_per_token(self, dtype: torch.dtype = torch.float16) -> int:
        return 2 * self.num_kv_heads * self.head_dim * torch.tensor([], dtype=dtype).element_size()


class CachedGQA(nn.Module):
    """GQA with KV-cache integration: prefill / chunk steps run the causal kernel over the cache with the
    offset mask (ch02/cached_generation.py:85-91), single-token steps run the split-KV decode kernel."""

    def __init__(self, hidden_dim: int, num_heads: int, num_kv_heads: int):
        super().__init__()
        self.num_heads = num_heads
        self.num_kv_heads = num_kv_heads
        self.num_groups = num_heads // num_kv_heads
        self.head_dim = hidden_dim // num_heads
        self.hidden_dim = hidden_dim
        self.q_proj = nn.Linear(hidden_dim, num_heads * self.head_dim, bias=False)
        self.k_proj = nn.Linear(hidden_dim, num_kv_heads * self.head_dim, bias=False)
        self.v_proj = nn.Linear(hidden_dim, num_kv_heads * self.head_dim, bias=False)
        self.o_proj = nn.Linear(hidden_dim, hidden_dim, bias=False)

    def forward(self, x: torch.Tensor, cache: LayerKVCache | None = None, start_pos: int = 0) -> torch.Tensor:
        batch, seq_len, _ = x.shape
        q = self.q_proj(x).view(batch, seq_len, self.num_heads, self.head_dim)
        k_new = self.k_proj(x).view(batch, seq_len, self.num_kv_heads, self.head_dim)
        v_new = self.v_proj(x).view(batch, seq_len, self.num_kv_heads, self.head_dim)
        if cache is not None:
            k_full, v_full = cache.update(k_new, v_new)
        else:
            k_full, v_full = k_new, v_new
        q = q.transpose(1, 2)
        if seq_len > 1:
            attn = flash_attention_forward(q, k_full.transpose(1, 2), v_full.transpose(1, 2), causal=True)
        else:
            attn = flash_decode(q, k_full, v_full, k_full.shape[1])          # no mask for one token (:85)
        attn = attn.transpose(1, 2).reshape(batch, seq_len, self.hidden_dim)
        return self.o_proj(attn)


class DecodeGraphRunner:
    """One decode step (append the new token's K/V, attend over the cache) captured in a CUDA graph.

    Follows the reference's `CUDAGraphRunner` (ch08/cuda_graph.py:30-76): static input buffers, warm-up,
    capture, then `copy_ -> replay -> clone`.  Works because the C-ABI launches make no host allocation
    or synchronisation and read the sequence lengths from device memory.

    tokens_per_step = k > 1: the step appends k tokens per sequence (q (B, Hq, k, D), k_new / v_new (B, k, Hkv, D))
    and attends all k in one launch with the offset causal mask, e.g. the verify step of speculative decoding
    (k - 1 draft tokens + 1); `run` returns (B, Hq, k, D).
    """

    def __init__(self, k_cache: torch.Tensor, v_cache: torch.Tensor, num_heads: int, *, block_tables=None, layer: int = 0,
                 warmup_iterations: int = 3, tokens_per_step: int = 1):
        if not 1 <= tokens_per_step <= 16:
            raise ValueError(f"tokens_per_step must be in [1, 16], got {tokens_per_step}")
        self.tokens_per_step = n = tokens_per_step
        self.k_cache, self.v_cache = k_cache, v_cache
        self.block_tables, self.layer = block_tables, layer
        self.num_heads = num_heads
        self.warmup_iterations = warmup_iterations
        paged = block_tables is not None
        self.batch = block_tables.shape[0] if paged else k_cache.shape[0]
        self.num_kv_heads, self.head_dim = k_cache.shape[-2], k_cache.shape[-1]
        self.capacity = block_tables.shape[1] * k_cache.shape[2] if paged else k_cache.shape[1]
        dev, dt = k_cache.device, k_cache.dtype
        self.static_q = torch.zeros(self.batch, num_heads, n, self.head_dim, device=dev, dtype=dt)
        self.static_k = torch.zeros(self.batch, n, self.num_kv_heads, self.head_dim, device=dev, dtype=dt)
        self.static_v = torch.zeros_like(self.static_k)
        self.seq_lens = torch.zeros(self.batch, dtype=torch.int32, device=dev)   # lengths BEFORE the step
        out_shape = (self.batch, num_heads, self.head_dim) if n == 1 else (self.batch, num_heads, n, self.head_dim)
        self.static_out = torch.empty(out_shape, device=dev, dtype=dt)
        splits = decode_num_splits(self.batch, self.num_kv_heads, self.capacity, group=num_heads // self.num_kv_heads,
                                   q_len=n)
        self.num_splits = splits
        self.workspace = decode_workspace(self.batch, num_heads * n, self.head_dim, splits, dev)
        self.graph: torch.cuda.CUDAGraph | None = None

    def _step(self):
        kv_append(self.k_cache, self.v_cache, self.static_k, self.static_v, self.seq_lens, block_tables=self.block_tables,
                  layer=self.layer)
        self.seq_lens.add_(self.tokens_per_step)
        flash_decode(self.static_q, self.k_cache, self.v_cache, self.seq_lens, block_tables=self.block_tables,
                     layer=self.layer, num_splits=self.num_splits, max_seq_len=self.capacity, workspace=self.workspace,
                     out=self.static_out)

    def capture(self, seq_lens: torch.Tensor) -> bool:
        """Capture the step.  `seq_lens` (B,) are the current lengths; warm-up steps are rolled back."""
        if not torch.cuda.is_available():
            return False
        start = seq_lens.to(device=self.seq_lens.device, dtype=torch.int32).clone()
        # warm-up and capture append tokens_per_step tokens from position seq_lens[b]: they must exist (cache rows /
        # allocated pages)
        n = self.tokens_per_step
        if int(start.max()) + n > self.capacity or int(start.min()) < 0:
            raise RuntimeError(f"cannot capture a decode step at lengths up to {int(start.max())}: the cache holds "
                               f"{self.capacity} tokens per sequence and the step appends "
                               f"{'one' if n == 1 else n}")
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(self.warmup_iterations):
                self.seq_lens.copy_(start)
                self._step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.seq_lens.copy_(start)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self._step()
        self.seq_lens.copy_(start)
        return True

    def run(self, q: torch.Tensor, k_new: torch.Tensor, v_new: torch.Tensor) -> torch.Tensor:
        if self.graph is None:
            raise RuntimeError("capture() first")
        self.static_q.copy_(q.reshape(self.static_q.shape))
        self.static_k.copy_(k_new.reshape(self.static_k.shape))
        self.static_v.copy_(v_new.reshape(self.static_v.shape))
        self.graph.replay()
        return self.static_out.clone()


class TensorParallelGQA(nn.Module):
    """`GroupedQueryAttention` sharded over KV-head groups (SURVEY.md §8(f) F4): q/k/v projections are
    column-parallel (`ColumnParallelLinear`, ch09/tensor_parallel.py:15-40: this rank's heads only), the
    attention kernels run on the local heads with no exchange, and the output projection is row-parallel
    (`RowParallelLinear`, ch09/tensor_parallel.py:43-68) followed by the all-reduce the reference only
    describes (ch09/nccl_primitives.py:45-67 models its cost).  `world_size` must divide num_kv_heads."""

    def __init__(self, hidden_dim: int, num_heads: int, num_kv_heads: int, world_size: int = 1, rank: int = 0,
                 process_group=None):
        super().__init__()
        assert num_heads % num_kv_heads == 0
        if num_kv_heads % world_size != 0:
            raise ValueError(f"world_size ({world_size}) must divide num_kv_heads ({num_kv_heads})")
        if not 0 <= rank < world_size:
            raise ValueError(f"rank {rank} outside [0, {world_size})")
        self.world_size, self.rank, self.process_group = world_size, rank, process_group
        self.hidden_dim = hidden_dim
        self.head_dim = hidden_dim // num_heads
        self.num_heads = num_heads // world_size              # local q heads
        self.num_kv_heads = num_kv_heads // world_size        # local kv heads
        self.q_proj = nn.Linear(hidden_dim, self.num_heads * self.head_dim, bias=False)
        self.k_proj = nn.Linear(hidden_dim, self.num_kv_heads * self.head_dim, bias=False)
        self.v_proj = nn.Linear(hidden_dim, self.num_kv_heads * self.head_dim, bias=False)
        self.o_proj = nn.Linear(self.num_heads * self.head_dim, hidden_dim, bias=False)

    @classmethod
    def from_full(cls, full: GroupedQueryAttention, world_size: int, rank: int, process_group=None):
        """This rank's shard of an unsharded block: rows of q/k/v weights, columns of the o weight."""
        tp = cls(full.hidden_dim, full.num_heads, full.num_kv_heads, world_size, rank, process_group)
        tp = tp.to(device=full.q_proj.weight.device, dtype=full.q_proj.weight.dtype)
        nq, nkv = tp.num_heads * tp.head_dim, tp.num_kv_heads * tp.head_dim
        with torch.no_grad():
            tp.q_proj.weight.copy_(full.q_proj.weight[rank * nq:(rank + 1) * nq])
            tp.k_proj.weight.copy_(full.k_proj.weight[rank * nkv:(rank + 1) * nkv])
            tp.v_proj.weight.copy_(full.v_proj.weight[rank * nkv:(rank + 1) * nkv])
            tp.o_proj.weight.copy_(full.o_proj.weight[:, rank * nq:(rank + 1) * nq])
        return tp

    def partial_forward(self, x: torch.Tensor, causal: bool = True) -> torch.Tensor:
        """This rank's summand of the block output (before the all-reduce)."""
        batch, seq_len, _ = x.shape
        q = self.q_proj(x).view(batch, seq_len, self.num_heads, self.head_dim).transpose(1, 2)
        k = self.k_proj(x).view(batch, seq_len, self.num_kv_heads, self.head_dim).transpose(1, 2)
        v = self.v_proj(x).view(batch, seq_len, self.num_kv_heads, self.head_dim).transpose(1, 2)
        attn = flash_attention_forward(q, k, v, causal=causal)
        return self.o_proj(attn.transpose(1, 2).reshape(batch, seq_len, self.num_heads * self.head_dim))

    def reduce(self, partial: torch.Tensor) -> torch.Tensor:
        if self.world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(partial, op=dist.ReduceOp.SUM, group=self.process_group)
        return partial

    def forward(self, x: torch.Tensor, causal: bool = True) -> torch.Tensor:
        return self.reduce(self.partial_forward(x, causal))
