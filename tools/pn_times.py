"""PointNet stage alone: per-kernel device times from the library's tagged timing hook (and a target for ncu).
Run on a GPU box:  python tools/pn_times.py [n] [pts] [pairs]     TC_DBG=... sets mmmot_set_debug bits."""
import ctypes
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mmmot_b200 as mb          # noqa: E402
from mmmot_b200 import _lib      # noqa: E402
from mmmot_b200.synthetic import synthetic_state_dict   # noqa: E402
from tools.aff_times import collect                     # noqa: E402


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 128
    pts = int(sys.argv[2]) if len(sys.argv) > 2 else 512
    pairs = int(sys.argv[3]) if len(sys.argv) > 3 else 32
    L = 2 * n
    net = mb.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch="C", test_mode=2, dropblock=0)
    net.load_state_dict(synthetic_state_dict("C", seed=0))
    net.cuda().eval()
    lib = _lib.load()
    wts = net.prepared()
    dev = wts.flat.device
    g = torch.Generator(device=dev).manual_seed(1)
    points = torch.randn(pairs * L * pts, 3, device=dev, generator=g)
    split = torch.arange(0, pairs * L * pts + 1, pts, dtype=torch.int32)
    split_d = split.to(dev)
    feats = torch.empty(pairs, 3, 512, L, device=dev)
    ws = torch.empty(int(lib.mmmot_pointnet_workspace(pairs, L, pairs * L * pts)), dtype=torch.uint8, device=dev)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    hs = split.numpy()
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def run():
        _lib.check(lib.mmmot_pointnet_fwd(wts.ptr, vp(points), vp(split_d), ctypes.c_void_p(hs.ctypes.data), pairs, L, vp(feats),
                                          vp(ws), ws.numel(), st), "mmmot_pointnet_fwd")
    for dbg in [int(x) for x in os.environ.get("TC_DBG", "0").split(",")]:
        _lib.check(lib.mmmot_set_debug(dbg), "mmmot_set_debug")
        for _ in range(2):
            run()
        torch.cuda.synchronize()
        lib.mmmot_timing_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        torch.cuda.synchronize()
        lib.mmmot_timing_enable(0)
        print(f"n={n} pts={pts} pairs={pairs} dbg={dbg}: PointNet stage {e0.elapsed_time(e1):.3f} ms")
        for name, (ms, fl, by, cnt) in collect(lib).items():
            print(f"   {name:32s} {ms:8.3f} ms  {fl / ms / 1e9 if ms else 0:8.1f} TFLOP/s  {by / ms / 1e6 if ms else 0:8.1f} GB/s")
    lib.mmmot_set_debug(0)


if __name__ == "__main__":
    main()
