"""Decode with Nq new tokens per sequence (speculative-decoding verify step), three routes timed the way
tools/decode_trace.py times one-token decode -- plans graph-replayed over >= 2 rotating K/V pools, so that HBM, not L2,
is measured:
    (a) multi   one pli_decode_fwd_multi launch (DecodePlan with q (B, Hq, Nq, D));
    (b) paged   flash_attention_paged over the same Nq rows (the tcgen05 prefill kernel, 128-row Q tiles);
    (c) loop    Nq one-token DecodePlans, token i with seq_lens - (Nq - 1 - i).
GB/s are on the algorithmic bytes 2*B*L*Hkv*D*2 + 2*B*Hq*Nq*D*2 + 4*B*ceil(L/bs).  Route (a) is checked against the
oracle on sampled sequences.
    python tools/decode_multi_perf.py
"""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import physics_llm_inference_b200 as pli
from oracle import attention_oracle as orc


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{name}, power limit / max SM clock: {pl}"


def timed(fn, reps=10):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def graph_us(steps_fns):
    """us per step of a CUDA graph that replays the step functions in order."""
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for f in steps_fns:
            f()
        torch.cuda.synchronize()
        with torch.cuda.graph(g):
            for f in steps_fns:
                f()
    torch.cuda.current_stream().wait_stream(side)
    return timed(g.replay) / len(steps_fns)


def case(B, Hq, Hkv, L, Nq, D=128, bs=16, tag=""):
    pages = B * L // bs
    npools = max(2, min(4, int(5e9 // (2 * pages * bs * Hkv * D * 2))))
    pools = [(torch.randn(pages, 1, bs, Hkv, D, device="cuda").bfloat16(),
              torch.randn(pages, 1, bs, Hkv, D, device="cuda").bfloat16()) for _ in range(npools)]
    table = torch.randperm(pages).to(torch.int32).view(B, L // bs).cuda()
    lens = torch.full((B,), L, dtype=torch.int32, device="cuda")
    q = torch.randn(B, Hq, Nq, D, device="cuda").bfloat16()
    nbytes = 2 * B * L * Hkv * D * 2 + 2 * B * Hq * Nq * D * 2 + 4 * B * ((L + bs - 1) // bs)
    steps = 12 // npools * npools

    # (a) one launch
    S = pli.decode_num_splits(B, Hkv, L, group=Hq // Hkv, q_len=Nq)
    ws = pli.decode_workspace(B, Hq * Nq, D, S, "cuda")
    out = torch.empty((B, Hq, Nq, D) if Nq > 1 else (B, Hq, D), device="cuda", dtype=torch.bfloat16)
    plans = [pli.DecodePlan(q, kp, vp, lens, block_tables=table, max_seq_len=L, num_splits=S, workspace=ws, out=out)
             for kp, vp in pools]
    us_a = graph_us([plans[i % npools] for i in range(steps)])
    # parity of (a) on sampled sequences: their pages gathered on the GPU, the oracle on the CPU
    plans[0]()
    torch.cuda.synchronize()
    err = 0.0
    for b in (0, B - 1):
        idx = table[b].long()
        kb, vb = pools[0][0][idx].cpu(), pools[0][1][idx].cpu()
        local = torch.arange(L // bs, dtype=torch.int32).view(1, -1)
        ro, _ = orc.paged_decode_oracle(q[b:b + 1], kb, vb, local, [L])
        err = max(err, (out.view(B, Hq, Nq, D)[b:b + 1].float().cpu() - ro).abs().max().item())

    # (b) the paged prefill kernel over the same rows
    def paged_step(kp, vp):
        return lambda: pli.flash_attention_paged(q, kp, vp, table, lens, max_seq_len=L)
    us_b = graph_us([paged_step(*pools[i % npools]) for i in range(steps)])

    # (c) Nq one-token launches with shifted lengths
    loop_lens = [lens - (Nq - 1 - i) for i in range(Nq)]
    S1 = pli.decode_num_splits(B, Hkv, L)
    ws1 = pli.decode_workspace(B, Hq, D, S1, "cuda")
    outs = [torch.empty(B, Hq, D, device="cuda", dtype=torch.bfloat16) for _ in range(Nq)]
    loops = [[pli.DecodePlan(q[:, :, i].contiguous(), kp, vp, loop_lens[i], block_tables=table, max_seq_len=L,
                             num_splits=S1, workspace=ws1, out=outs[i]) for i in range(Nq)] for kp, vp in pools]

    def loop_step(j):
        return lambda: [pl() for pl in loops[j]]
    us_c = graph_us([loop_step(i % npools) for i in range(steps)])

    name = f"{tag}B{B} Hq{Hq} Hkv{Hkv} L{L} Nq{Nq}"
    chunks = (Hq // Hkv * Nq + 15) // 16
    print(f"{name:36s} splits {S:2d} chunks {chunks} | (a) multi {us_a:7.1f} us {nbytes / us_a / 1e3:5.0f} GB/s | "
          f"(b) paged prefill {us_b:7.1f} us {nbytes / us_b / 1e3:5.0f} GB/s | (c) {Nq} x one-token {us_c:7.1f} us "
          f"{nbytes / us_c / 1e3:5.0f} GB/s | (a) vs oracle max|dO| {err:.2e}", flush=True)
    assert err <= 2e-2, f"{name}: route (a) differs from the oracle by {err}"
    del pools, plans, loops


if __name__ == "__main__":
    print(gpu_info(), flush=True)
    for nq in (1, 2, 4, 8, 16):
        case(64, 32, 8, 4096, nq, tag="C3 ")
    for nq in (2, 4):
        case(256, 4, 1, 1024, nq, tag="C5/8 ")
    case(1, 32, 8, 32768, 4)
