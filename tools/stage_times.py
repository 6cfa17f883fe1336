"""Per-stage device time of one bench step (CUDA events around every C-ABI stage call).
Run on a GPU box:  python tools/stage_times.py [pairs]"""
import collections
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mmmot_b200 as mb          # noqa: E402
from mmmot_b200 import _lib      # noqa: E402
import bench                     # noqa: E402


def main():
    pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    dev = torch.device("cuda:0")
    CFG = bench.CFG
    n, pts, hw = CFG["n"], CFG["pts"], CFG["hw"]
    L, B = 2 * n, pairs
    net = mb.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch=CFG["fusion"],
                         affinity_op=CFG["affinity_op"], softmax_mode=CFG["softmax_mode"],
                         neg_threshold=CFG["neg_threshold"], test_mode=2, dropblock=0)
    from mmmot_b200.synthetic import synthetic_state_dict
    net.load_state_dict(synthetic_state_dict(CFG["fusion"], seed=0))
    net.cuda(dev).eval()
    g = torch.Generator(device=dev).manual_seed(1234)
    crops = torch.randn(B * L, 3, hw, hw, device=dev, generator=g)
    points = torch.randn(B * L * pts, 3, device=dev, generator=g)
    split = torch.arange(0, B * L * pts + 1, pts, dtype=torch.int32)
    batch = (crops, points, split, n)
    lib = _lib.load()
    _lib.check(lib.mmmot_set_debug(int(os.environ.get('TC_DBG', '0'))), "mmmot_set_debug")
    spans = collections.defaultdict(list)
    names = ["mmmot_appearance_fwd", "mmmot_pointnet_fwd", "mmmot_fusion_det_fwd", "mmmot_affinity_fwd",
             "mmmot_lp_assign"]
    for nm in names:
        orig = getattr(lib, nm)

        def wrap(*a, _o=orig, _n=nm):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = _o(*a)
            e1.record()
            spans[_n].append((e0, e1))
            return r
        setattr(lib, nm, wrap)
    for it in range(3):
        spans.clear()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0.record()
        net.predict_batch(*batch)
        t1.record()
        torch.cuda.synchronize()
    tot = t0.elapsed_time(t1)
    print(f"pairs={pairs} step {tot:.2f} ms -> {pairs / tot * 1e3:.1f} pairs/s")
    acc = 0.0
    for nm in names:
        ms = sum(a.elapsed_time(b) for a, b in spans[nm])
        acc += ms
        print(f"  {nm:24s} {ms:8.2f} ms  {100 * ms / tot:5.1f}%  ({len(spans[nm])} calls)")
    print(f"  {'host glue / other':24s} {tot - acc:8.2f} ms  {100 * (tot - acc) / tot:5.1f}%")
    if os.environ.get("KPROF"):
        # per-launch device durations of a normal (un-serialised) run through CUPTI
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            net.predict_batch(*batch)
            torch.cuda.synchronize()
        evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        evs.sort(key=lambda e: e.time_range.start)
        for e in evs:
            print(f"    {e.time_range.elapsed_us() / 1e3:9.3f} ms  {e.name[:70]}")


if __name__ == "__main__":
    main()
