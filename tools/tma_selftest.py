"""TMA-fed tcgen05 engine self-test: planar FP16 hi/lo operands, 1x1 and 3x3, vs fp64."""
import ctypes, os, sys, time
import torch
import torch.nn.functional as F
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from mmmot_b200 import _lib
from mmmot_b200.weights import pack_tc
lib = _lib.load()
_lib.check(lib.mmmot_set_debug(int(os.environ.get('TC_DBG', '0'))), "mmmot_set_debug")
if os.environ.get('MMMOT_KSEG'): lib.mmmot_set_kseg(int(os.environ['MMMOT_KSEG']))
vp = lambda t: ctypes.c_void_p(t.data_ptr())
g = torch.Generator().manual_seed(0)


def planes(x):
    hi = x.half()
    lo = (x - hi.float()).half()
    return torch.stack([hi, lo]).contiguous()


LIN = ((128, 32, 256), (256, 64, 512), (512, 512, 4099), (64, 64, 300), (1024, 128, 1000), (512, 512, 148 * 256 * 4))
if os.environ.get('TMA_ONLY'):
    LIN = ()
for (M, K, rows) in LIN:
    Wt = torch.randn(K, M, generator=g); X = torch.randn(rows, K, generator=g); b = torch.randn(M, generator=g)
    ref = X.double() @ Wt.double() + b.double()
    Wp, wps = pack_tc(Wt)
    Wp_d, b_d, Xp = Wp.cuda(), b.cuda(), planes(X).cuda()
    Y = torch.full((rows, M), float("nan"), device="cuda")
    rc = lib.mmmot_debug_linear_planar(vp(Wp_d), wps, vp(b_d), vp(Xp), vp(Y), M, K, rows, None)
    torch.cuda.synchronize()
    t0 = time.time()
    for _ in range(3):
        lib.mmmot_debug_linear_planar(vp(Wp_d), wps, vp(b_d), vp(Xp), vp(Y), M, K, rows, None)
    torch.cuda.synchronize()
    dt = (time.time() - t0) / 3
    err = float((Y.double().cpu() - ref).abs().max() / ref.abs().max())
    print(f"linear M={M} K={K} rows={rows}: rc={rc} err={err:.2e} {2.0*M*K*rows/dt/1e12:.1f} TF/s", flush=True)

CONVS = ((4, 8, 8, 32, 64), (2, 64, 64, 64, 64), (3, 32, 32, 64, 128), (5, 16, 16, 128, 256), (9, 8, 8, 256, 512), (33, 4, 4, 512, 512),
                        (2, 24, 40, 32, 64), (1024, 16, 16, 256, 256), (4096, 8, 8, 512, 512))
if os.environ.get('TMA_ONLY'):
    CONVS = ((1024, 64, 64, 64, 64), (1024, 32, 32, 128, 128), (1024, 16, 16, 256, 256))
for (n, H, W, C, M) in CONVS:
    w = torch.randn(M, C, 3, 3, generator=g) * (2.0 / (9 * C)) ** 0.5
    b = torch.randn(M, generator=g) * 0.1
    x = torch.randn(n, C, H, W, generator=g)
    ref = F.relu(F.conv2d(x.double(), w.double(), b.double(), padding=1)) if n <= 64 else None
    Wt = w.permute(2, 3, 1, 0).reshape(9 * C, M)           # [(ky*3+kx)*C + ci][co]
    Wp, wps = pack_tc(Wt)
    Xp = planes(x.permute(0, 2, 3, 1).contiguous()).cuda()    # NHWC planes
    Yp = torch.zeros(2, n, H, W, M, dtype=torch.half, device="cuda")
    Wp_d, b_d = Wp.cuda(), b.cuda()
    scr = torch.zeros((n + 16) * H * W * M + 256 * M, device="cuda")
    for seg, sp in (("1pass", None), ("kseg", vp(scr))):
        rc = lib.mmmot_debug_conv_planar(vp(Wp_d), wps, vp(b_d), vp(Xp), vp(Yp), n, H, W, C, M, sp, None)
        torch.cuda.synchronize()
        t0 = time.time()
        for _ in range(3):
            lib.mmmot_debug_conv_planar(vp(Wp_d), wps, vp(b_d), vp(Xp), vp(Yp), n, H, W, C, M, sp, None)
        torch.cuda.synchronize()
        dt = (time.time() - t0) / 3
        if ref is not None:
            y = (Yp[0].double() + Yp[1].double()).cpu().permute(0, 3, 1, 2)
            err = float((y - ref).abs().max() / ref.abs().max())
        else:
            err = float("nan")
        print(f"conv n={n} {H}x{W} C={C} M={M} [{seg}]: rc={rc} err={err:.2e} {2.0*M*9*C*n*H*W/dt/1e12:.1f} TF/s", flush=True)
