"""conv_rows_fused 64->64 at 128x128: time with the transform and / or the epilogue's work removed (bring-up switches),
to see which role bounds a row.  python scripts/rows_ablate.py [B]"""
import ctypes as C, os, sys, subprocess
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if len(sys.argv) > 2:
    import torch
    from mcedm_b200 import _lib as L
    from mcedm_b200.engine import pack_conv3x3
    lib = L.lib(); dev = torch.device("cuda:0"); dt = torch.float16
    B, H = int(sys.argv[1]), 128
    xf = sys.argv[2] == "1"
    res = sys.argv[3] == "1"
    x = torch.randn(B, H, 128, 64, device=dev).to(dt)
    r = torch.randn(B, H, 128, 64, device=dev).to(dt)
    coef = torch.cat([torch.rand(B, 64, device=dev) + 0.5, torch.randn(B, 64, device=dev) * 0.3], 1).contiguous()
    w = pack_conv3x3(torch.randn(64, 64, 3, 3, device=dev) / 24, dtype=dt); bias = torch.randn(64, device=dev)
    out = torch.empty(B, H, 128, 64, device=dev, dtype=dt); st = torch.empty(B * H, 4, 16, 2, device=dev)
    cptr = (C.c_void_p * 1)(coef.data_ptr()) if xf else None
    def run():
        L.check(lib.mcedm_conv_rows_fused(L.ptr_array([x]), cptr, 1, None, 0, L.ptr(w), L.ptr(bias), B, H, 64, 0, 64, L.ptr(out), 1,
                                          L.ptr(r) if res else None, 1 if res else 0, 0, 0, L.ptr(st), 1, L.stream_ptr()))
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        run()
    e1.record(); torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 10 * 1e3
    print(f"DBG={os.environ.get('MCEDM_DBG', '0'):>2} transform={int(xf)} residual={int(res)}: {us:7.1f} us  {2.0 * B * H * 128 * 64 * 576 / us / 1e6:6.0f} TFLOP/s")
else:
    B = sys.argv[1] if len(sys.argv) > 1 else "128"
    for dbg in ("0", "2"):
        for xf in ("1", "0"):
            for res in ("0", "1"):
                subprocess.run([sys.executable, __file__, B, xf, res], env=dict(os.environ, MCEDM_DBG=dbg))
