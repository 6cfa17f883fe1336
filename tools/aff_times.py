"""Affinity stage alone (BASELINE cfg5): per-kernel device times from the library's tagged timing hook.
Run on a GPU box:  python tools/aff_times.py [n] [pairs]      TC_DBG=0,4,8 runs with those mmmot_set_debug bits (0-3)."""
import ctypes
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mmmot_b200 as mb          # noqa: E402
from mmmot_b200 import _lib      # noqa: E402
from mmmot_b200.synthetic import synthetic_state_dict   # noqa: E402


def collect(lib):
    n = lib.mmmot_timing_tag_count()
    ms, fl, by = (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_double * n)()
    cnt = (ctypes.c_long * n)()
    lib.mmmot_timing_collect_tags(ms, fl, by, cnt)
    return {lib.mmmot_timing_tag_name(t).decode(): (ms[t], fl[t], by[t], cnt[t]) for t in range(n) if cnt[t]}


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 128
    pairs = int(sys.argv[2]) if len(sys.argv) > 2 else 32
    op, sm = os.environ.get("AFF_OP", "minus_abs"), os.environ.get("AFF_SM", "dual_add")
    net = mb.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch="C", affinity_op=op,
                         softmax_mode=sm, neg_threshold=0.2, test_mode=2, dropblock=0)
    net.load_state_dict(synthetic_state_dict("C", seed=0))
    net.cuda().eval()
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(1)
    feats = torch.relu(torch.randn(pairs, 3, 512, 2 * n, device="cuda", generator=g))
    for dbg in [int(x) for x in os.environ.get("TC_DBG", "0").split(",")]:
        _lib.check(lib.mmmot_set_debug(dbg), "mmmot_set_debug")
        for _ in range(2):
            net.associate_batch(feats, n)
        torch.cuda.synchronize()
        lib.mmmot_timing_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        net.associate_batch(feats, n)
        e1.record()
        torch.cuda.synchronize()
        lib.mmmot_timing_enable(0)
        print(f"n={n} pairs={pairs} dbg={dbg}: affinity stage {e0.elapsed_time(e1):.3f} ms")
        for name, (ms, fl, by, cnt) in collect(lib).items():
            print(f"   {name:32s} {ms:8.3f} ms  {fl / ms / 1e9 if ms else 0:8.1f} TFLOP/s  {by / ms / 1e6 if ms else 0:8.1f} GB/s")
    lib.mmmot_set_debug(0)


if __name__ == "__main__":
    main()
