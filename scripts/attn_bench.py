"""Attention kernel timing at the evaluation's shape (B x 1024 tokens x 64): python scripts/attn_bench.py [B]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from mcedm_b200 import _lib as L
lib = L.lib(); dev = torch.device("cuda:0")
B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
qkv = (torch.randn(B, 1024, 192, device=dev) * 0.8).half()
out = torch.empty(B, 1024, 64, device=dev, dtype=torch.float16)
run = lambda: L.check(lib.mcedm_attention(L.ptr(qkv), B, 1024, L.ptr(out), None, 1, L.stream_ptr()))
for _ in range(3):
    run()
torch.cuda.synchronize(); L.check_watchdog()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20):
    run()
e1.record(); torch.cuda.synchronize()
us = e0.elapsed_time(e1) / 20 * 1e3
print(f"B={B}: {us:.1f} us per call, {4.0 * B * 1024 * 1024 * 64 / us / 1e6:.0f} TFLOP/s")
