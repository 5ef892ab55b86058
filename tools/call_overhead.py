import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import physics_llm_inference_b200 as pli
B, Hq, Hkv, L, D, bs = 256, 4, 1, 1024, 128, 16
pages = B * L // bs
kp = torch.randn(pages, 1, bs, Hkv, D, device="cuda").bfloat16(); vp = torch.randn(pages, 1, bs, Hkv, D, device="cuda").bfloat16()
table = torch.randperm(pages).to(torch.int32).view(B, L // bs).cuda()
lens = torch.full((B,), L, dtype=torch.int32, device="cuda")
q = torch.randn(B, Hq, 1, D, device="cuda").bfloat16()
ws = pli.decode_workspace(B, Hq, D, 1, "cuda"); out = torch.empty(B, Hq, D, device="cuda", dtype=torch.bfloat16)
f = lambda: pli.flash_decode(q, kp, vp, lens, block_tables=table, max_seq_len=L, num_splits=1, workspace=ws, out=out)
for _ in range(10): f()
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(2000): f()
t1 = time.perf_counter()
torch.cuda.synchronize()
t2 = time.perf_counter()
print(f"CPU issue time per call {(t1 - t0) / 2000 * 1e6:.1f} us; total per call incl. drain {(t2 - t0) / 2000 * 1e6:.1f} us")
g = torch.cuda.CUDAGraph()
s = torch.cuda.Stream()
with torch.cuda.stream(s):
    f()
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        for _ in range(20): f()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
g.replay(); torch.cuda.synchronize()
e0.record()
for _ in range(10): g.replay()
e1.record(); torch.cuda.synchronize()
us = e0.elapsed_time(e1) / 200 * 1e3
nbytes = 2 * B * L * Hkv * D * 2
print(f"graph replay: {us:.1f} us per decode  {nbytes / us / 1e3:.0f} GB/s")
qq = torch.randn(4, 32, 8192, 128, device="cuda").bfloat16(); kk = torch.randn(4, 8, 8192, 128, device="cuda").bfloat16()
for _ in range(3): pli.flash_attention_forward(qq, kk, kk, causal=True)
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(50): pli.flash_attention_forward(qq, kk, kk, causal=True)
t1 = time.perf_counter(); torch.cuda.synchronize()
print(f"prefill CPU issue time per call {(t1 - t0) / 50 * 1e6:.1f} us")
