"""Graph-timed adp_conv_gemm on the README net's GEMM shapes at B=8, for every N tile that divides N
(bias + residual + GroupNorm statistics, as the conv3 of a ResnetItem runs).  20 launches captured
in a CUDA graph, replayed (device time only).  usage: python tools/time_gemm.py"""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from audio_diffusion_pytorch_b200 import ops
dev = "cuda"

def run(M, K, N, taps, bn, res=True, stats=False, B=8, reps=20):
    x = torch.randn(B, M // B, K, device=dev).bfloat16()
    w = torch.randn(N, K, taps, device=dev) * (K * taps) ** -0.5
    out = torch.empty(B, M // B, N, device=dev, dtype=torch.bfloat16)
    r = torch.randn_like(out) if res else None
    bias = torch.randn(N, device=dev)
    st = torch.zeros(B, 8, 2, device=dev, dtype=torch.float64) if stats else None
    wp = ops.pack_conv(w)
    tp = (-1, 0, 1) if taps == 3 else (0,)
    f = lambda: ops.conv_gemm(x, wp, out, c_in=K, n_valid=N, taps=tp, bias=bias, residual=r, stats=st, block_n=bn)
    for _ in range(3): f()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()          # host launch cost (~30 us via ctypes) must not be timed
    with torch.cuda.graph(g):
        for _ in range(reps): f()
    g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    g.replay(); g.replay()
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (2 * reps)
    fl = 2.0 * M * K * N * taps
    return us, fl / us / 1e6

if __name__ == "__main__":
    shapes = [("L1 conv3", 524288, 32, 32, 3), ("L2 conv3", 131072, 64, 64, 3), ("L3 conv3", 32768, 128, 128, 3),
              ("L4 conv3", 16384, 256, 256, 3), ("L5 conv3", 8192, 512, 512, 3), ("L6 conv3", 4096, 512, 512, 3),
              ("L7 conv3", 2048, 1024, 1024, 3), ("L8 conv3", 1024, 1024, 1024, 3),
              ("L7 qkv", 2048, 1024, 1536, 1), ("L5 qkv", 8192, 512, 1536, 1), ("L7 out", 2048, 512, 1024, 1),
              ("L5 out", 8192, 512, 512, 1)]
    for name, M, K, N, taps in shapes:
        row = []
        for bn in (32, 64, 128, 256):
            if N % bn:
                continue
            try:
                us, tf = run(M, K, N, taps, bn, res=True, stats=True)
                row.append(f"bn{bn}: {us:6.1f}us {tf:5.0f}TF")
            except Exception as e:
                row.append(f"bn{bn}: ERR {str(e)[:30]}")
        print(f"{name:9s} | " + " | ".join(row), flush=True)
