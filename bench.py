#!/usr/bin/env python
"""Throughput benchmark of the association hot path (driver contract: one JSON line on stdout).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg2|cfg3|cfg4|cfg5] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Default workload = BASELINE.json configs[3] / SURVEY §8d cfg4, the configuration the metric is quoted on:
pp_pv_40e_dualadd_subabs_C (Fusion C, minus_abs, dual_add), N = M = 128 detections per frame, P = 512 LiDAR points per
detection, 64x64 crops.  A "step" = one pass of forward + association LP over `--pairs` frame-pairs per GPU (weak
scaling: per-GPU work fixed; `--total-pairs T` fixes the total instead = strong scaling, BASELINE's "B=4096 sharded 8x").
Frame-pairs are independent units, sharded over ranks with no data-path collective; the only collective is the final
gather of the assignment indices (mmmot_b200.parallel.gather_pairs, SURVEY §8e), inside the timed region.
--config cfg2 / cfg3: BASELINE configs[1] / [2] (Fusion A N=32 B=64; Fusion C multiply/none N=64 P=512 B=256).
--config cfg5: BASELINE configs[4], the N sweep 8 -> 256 of the affinity + LP kernels alone (value = the N=128 point).

value   : frame-pairs/s with inputs resident in HBM (CUDA events, max over ranks).
e2e     : same metric through the public API with HOST (pinned) inputs: H2D of crops/points and D2H of the assignment
          results inside the timed region.
roofline: dominant kernel = the TMA-fed tcgen05 3x3-conv contraction of the VGG trunk (layers 1..12, 83 % of the
          algorithmic FLOPs), timed per launch with CUDA events on the launching stream (library hook mmmot_timing_*).
kernels : the same per-launch timing for EVERY hot kernel of the path, tagged (stage, layer): algorithmic FLOPs and
          compulsory HBM bytes of the launch / its measured duration, against the measured tensor / HBM peak.
cpu_baseline / --impl reference: the oracle port of the reference's PyTorch-CPU path (the reference is pure Python and
          is not needed at run time) on the host cores (thread count swept on the real shape); --impl reference times one
          frame-pair per step, --steps of them.
--dump-outputs DIR: after the timed steps, every array the timed path returned in its last step, as DIR/<name>.npy
          (float32, or float64 for integer outputs; cfg5: per sweep point, prefixed n<N>_).  Inputs and weights are
          seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: model / shape of SURVEY §8d ("pairs" = frame-pairs per GPU per step)
    "cfg2": dict(fusion="A", affinity_op="multiply", softmax_mode="none", neg_threshold=0.2, n=32, pts=128, hw=64, pairs=64,
                 what="cfg2 pp_pv_40e_mul_A: Fusion A, multiply, no softmax, N=M=32 dets/frame, P=128 LiDAR pts/det, 64x64 crops"),
    "cfg3": dict(fusion="C", affinity_op="multiply", softmax_mode="none", neg_threshold=0.2, n=64, pts=512, hw=64, pairs=256,
                 what="cfg3 pp_pv_40e_mul_C: Fusion C, multiply, no softmax, N=M=64 dets/frame, P=512 LiDAR pts/det, 64x64 crops"),
    "cfg4": dict(fusion="C", affinity_op="minus_abs", softmax_mode="dual_add", neg_threshold=0.2, n=128, pts=512, hw=64, pairs=128,
                 what="cfg4 pp_pv_40e_dualadd_subabs_C: Fusion C, minus_abs, dual_add, N=M=128 dets/frame, P=512 LiDAR pts/det, "
                      "64x64 crops"),
    "cfg5": dict(fusion="C", affinity_op="minus_abs", softmax_mode="dual_add", neg_threshold=0.2, n=128, pts=0, hw=0, pairs=32,
                 what="cfg5 N sweep 8..256 of the affinity + new/end + softmax + LP kernels alone (inputs = 3x512x2N feature stacks)"),
}
CFG = CONFIGS["cfg4"]          # tools/ import this
SWEEP_N = (8, 16, 32, 64, 128, 256)


def flop_per_pair(c):
    """Algorithmic FLOPs per frame-pair (SURVEY §8d), minimal work (no dead STN, split head)."""
    n, L = c["n"], 2 * c["n"]
    aff = 3 * n * n * 1.7042e6 + 3 * L * 0.655e6
    if not c["hw"]:
        return aff
    vgg = L * 30.693e9 * (c["hw"] / 224.0) ** 2 + L * 0.41e6
    pn = L * c["pts"] * 0.369e6 + L * 1.57e6
    fus = L * (1.05e6 if c["fusion"] in "AB" else 2.10e6) + 3 * L * 0.787e6
    return vgg + pn + fus + aff


def bytes_in_per_pair(c):
    L = 2 * c["n"]
    return L * 3 * c["hw"] * c["hw"] * 4 + L * c["pts"] * 12 + (L + 1) * 8 if c["hw"] else 3 * 512 * L * 4


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def _nvml(self):
        """In-process NVML handle (cheap queries).  A nvidia-smi subprocess per sample re-initialises the driver every
        time (~0.5 s each on these boxes) and was seen to stall the launching thread's CUDA calls; kept as fallback only."""
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                idx = int(vis.split(",")[self.index])
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(idx)
        except Exception:
            return None, None

    def run(self):
        nv, h = self._nvml()
        while not self.stop_flag and nv is not None:
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                act = lambda bit: "Active" if r & bit else "Not Active"
                self.rows.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)),
                                  str(nv.nvmlDeviceGetPowerUsage(h) / 1000.0), act(nv.nvmlClocksEventReasonHwSlowdown),
                                  act(nv.nvmlClocksEventReasonHwThermalSlowdown), act(nv.nvmlClocksEventReasonSwThermalSlowdown),
                                  act(nv.nvmlClocksEventReasonSwPowerCap)])
            except Exception:
                pass
            time.sleep(0.1)
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        self.stop_flag = True
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = max([int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = sorted(float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit())
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons, "samples": len(sm),
                "power_w": pw[len(pw) // 2] if pw else None}


# --------------------------------------------------------------------------------------- CPU legs (oracle port)
def pick_cpu_threads(c):
    """torch's intra-op scaling on many-core hosts is poor for these shapes (128 threads were 14x slower than 8 on the
    GPU box), so the thread count is swept on the REAL shape: the dominant CPU stage of the workload (the VGG trunk on
    the pair's 2N crops; the affinity MLP for cfg5) is timed at a few counts up to all host cores, fastest wins."""
    from mmmot_b200.synthetic import synthetic_pair, synthetic_state_dict
    from oracle import torch_ref
    ncpu = os.cpu_count() or 1
    sd = synthetic_state_dict(c["fusion"], seed=0)
    if c["hw"]:
        dets, _, _ = synthetic_pair(c["n"], c["n"], 8, c["hw"], seed=0)
        probe = lambda: torch_ref.appearance(sd, dets)
    else:
        f = torch.relu(torch.randn(3, 512, 2 * c["n"], generator=torch.Generator().manual_seed(0)))
        probe = lambda: torch_ref.associate(sd, f[:, :, :c["n"]], f[:, :, c["n"]:], c["affinity_op"], c["softmax_mode"])
    best, best_t, sweep = 1, float("inf"), {}
    for th in sorted({min(ncpu, t) for t in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(th)
        with torch.no_grad():
            t = time.perf_counter()
            probe()
            dt = time.perf_counter() - t
        sweep[th] = round(dt, 3)
        if dt < best_t:
            best, best_t = th, dt
        if dt > 4 * best_t:
            break
    return best, sweep


def oracle_pairs_per_s(c, n_pairs, threads, budget_s=60.0):
    """The reference's CPU path (oracle port of TrackingNet.forward + HiGHS restatement of the LP; cfg5: associate +
    LP only).  Bounded sample: stops early once `budget_s` seconds of CPU work are spent (>= 1 pair is always timed;
    budget_s=None times all n_pairs)."""
    from mmmot_b200.synthetic import synthetic_pair, synthetic_state_dict
    from oracle import lp_ref, torch_ref
    torch.set_num_threads(threads)
    sd = synthetic_state_dict(c["fusion"], seed=0)
    n = c["n"]
    t_tot = 0.0
    for p in range(n_pairs):
        if c["hw"]:
            dets, info, split = synthetic_pair(n, n, c["pts"], c["hw"], seed=p)
            t = time.perf_counter()
            det, link, new, end, _ = torch_ref.forward(sd, dets, info, split, c["fusion"], c["affinity_op"], c["softmax_mode"],
                                                       c["neg_threshold"])
            lp_ref.milp_solve(det[2], [link[0][2:3]], new[2], end[2], [n, n])
        else:
            f = torch.relu(torch.randn(3, 512, 2 * n, generator=torch.Generator().manual_seed(p)))
            det = torch.rand(2 * n, generator=torch.Generator().manual_seed(p))
            t = time.perf_counter()
            with torch.no_grad():
                link, new, end = torch_ref.associate(sd, f[:, :, :n], f[:, :, n:], c["affinity_op"], c["softmax_mode"])
            z = torch.zeros(n)
            lp_ref.milp_solve(det, [link[2]], torch.cat([z, new[2]]), torch.cat([end[2], z]), [n, n])
        t_tot += time.perf_counter() - t
        if budget_s is not None and t_tot > budget_s:
            n_pairs = p + 1
            break
    return n_pairs / t_tot, t_tot, n_pairs


def cpu_leg(c, n_pairs, budget_s=60.0):
    threads, sweep = pick_cpu_threads(c)
    rate, secs, done = oracle_pairs_per_s(c, n_pairs, threads, budget_s)
    what = "forward + LP" if c["hw"] else "affinity stage + LP"
    return {"value": rate, "unit": "frame-pairs/s", "cores": threads, "host_cores": os.cpu_count(), "kind": "port",
            "thread_sweep_s": sweep,
            "sample": f"{done} frame-pair(s) of the same workload ({what}, {secs:.1f} s of CPU work): oracle port of the reference "
                      "PyTorch-CPU path + HiGHS MILP restatement of ortools_solve (OR-tools absent); torch threads = the fastest "
                      "of the sweep in thread_sweep_s (seconds of the dominant CPU stage on this shape per thread count)"}, secs, done


def config_dict(c, name, pairs, world, scaling):
    d = {"workload": c["what"] + ("; forward + association LP" if c["hw"] else ""),
         "config": name, "pairs_per_gpu_per_step": pairs, "global_pairs_per_step": pairs * world,
         "parallelism": f"frame-pair sharding x{world}, final gather only", "scaling_mode": scaling,
         "l2_policy": "inputs larger than L2 (%.2f GB per GPU per step vs 126 MB L2)" % (pairs * bytes_in_per_pair(c) / 1e9)}
    return d


DUMP_LIMIT = 64 << 20          # bytes written by --dump-outputs, all arrays together


def _dump_bytes(t):
    return t.numel() * (4 if t.dtype == torch.float32 else 8)


def dump_outputs(out_dir, sets):
    """--dump-outputs: every output of the last timed step as <out_dir>/<name>.npy, float32 as computed and every other
    dtype (int32 indices, the status word) as float64, which holds it exactly.  `sets` is a list of
    (prefix, per_pair, shared, B): per_pair maps names (prefix included) to tensors whose leading axis is the B
    frame-pairs, shared to tensors without one.  When the whole would exceed DUMP_LIMIT, every per-pair array keeps the
    same fixed, seeded subset of its frame-pairs, and the indices kept are written as <prefix>pair_index.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    limit = DUMP_LIMIT - (1 << 20)                       # headroom for the .npy headers
    total = sum(_dump_bytes(t) for _, pp, sh, _ in sets for t in list(pp.values()) + list(sh.values()))
    shared = sum(_dump_bytes(t) for _, _, sh, _ in sets for t in sh.values())
    index = 8 * sum(B for _, _, _, B in sets)            # the pair_index arrays, when sampling
    frac = 1.0 if total <= limit else (limit - shared) / (total - shared + index)
    for prefix, per_pair, sh, B in sets:
        arrays = dict(sh)
        if frac < 1.0:
            keep = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:max(1, int(B * frac))].sort().values
            arrays[prefix + "pair_index"] = keep
            arrays.update({k: v[keep.to(v.device)] for k, v in per_pair.items()})
        else:
            arrays.update(per_pair)
        for k, v in arrays.items():
            v = v.detach().cpu()
            np.save(os.path.join(out_dir, k + ".npy"), (v if v.dtype == torch.float32 else v.double()).numpy())


def run_reference(args, c, name, rank):
    if rank != 0:
        return
    cpu, secs, done = cpu_leg(c, args.steps, budget_s=None)       # one frame-pair per step, every step timed
    line = {"impl": "reference", "metric": metric_name(c), "value": cpu["value"], "unit": "frame-pairs/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(done, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the same config as the GPU arm; every CPU "step" is a bounded sample of it (cpu_baseline.sample)
            "config": dict(config_dict(c, name, args.pairs or c["pairs"], max(args.gpus, 1), "weak"), engine="auto"),
            "cpu_baseline": cpu,
            "e2e": {"value": cpu["value"], "unit": "frame-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def metric_name(c):
    return f"frame-pairs/sec at N={c['n']} dets" + ("" if c["hw"] else " (affinity + LP kernels only)")


# --------------------------------------------------------------------------------------- per-kernel rooflines
TENSOR_TAGS = ("vgg.conv", "pointnet.l2", "pointnet.l3", "pointnet.l4", "pointnet.l5", "pointnet.head", "affinity.l1",
               "affinity.l2", "affinity.l3")


def collect_tags(lib):
    n = lib.mmmot_timing_tag_count()
    ms, fl, by = (ctypes.c_double * n)(), (ctypes.c_double * n)(), (ctypes.c_double * n)()
    cnt = (ctypes.c_long * n)()
    rc = lib.mmmot_timing_collect_tags(ms, fl, by, cnt)
    assert rc == 0, rc
    return {lib.mmmot_timing_tag_name(t).decode(): (ms[t], fl[t], by[t], cnt[t]) for t in range(n) if cnt[t]}


def kernel_table(tags, steps, peaks):
    """One row per (stage, layer): algorithmic work of its launches / their measured duration vs the binding peak."""
    tpeak, hpeak = peaks.get("bf16_tflops_sustained", 1400.0), peaks.get("hbm_gbs", 6650.0)
    rows = []
    for name, (ms, fl, by, cnt) in tags.items():
        if ms <= 0:
            continue
        tf, gb = fl / ms / 1e9, by / ms / 1e6
        # vgg.pool_mean_heads: the per-image fixed-point sums it reads were written by the preceding conv epilogue's atomics
        # and are still L2-resident (100 MB per launch in ~20 us), so an HBM fraction would be meaningless
        bound = "latency" if name == "lp.assign" else "l2" if name == "vgg.pool_mean_heads" else \
            ("tensor" if name.startswith(TENSOR_TAGS) and name != "vgg.conv0" else "hbm")
        row = {"kernel": name, "launches_per_step": cnt / steps, "ms_per_step": ms / steps, "bound": bound,
               "algorithmic_tflops": round(tf, 1), "algorithmic_gbs": round(gb, 1)}
        if bound == "tensor":
            row.update(frac=round(tf / tpeak, 3), mma_issue_frac=round(3 * tf / tpeak, 3))
        elif bound == "hbm":
            row.update(frac=round(gb / hpeak, 3))
        rows.append(row)
    return rows


# --------------------------------------------------------------------------------------- cfg5: affinity + LP sweep
def run_sweep(args, c, name, rank, world, local):
    import mmmot_b200
    from mmmot_b200 import _lib
    from mmmot_b200.synthetic import synthetic_state_dict
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    net = mmmot_b200.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch=c["fusion"],
                                 affinity_op=c["affinity_op"], softmax_mode=c["softmax_mode"], neg_threshold=c["neg_threshold"],
                                 test_mode=2, dropblock=0)
    net.load_state_dict(synthetic_state_dict(c["fusion"], seed=0))
    net.cuda(dev).eval()
    peaks, how = load_peaks()
    sampler = ClockSampler(local)
    sampler.start()
    points, main, dumps = [], None, []
    for n in SWEEP_N:
        # batch sized so that one step is >= ~100 ms of device work and inputs exceed L2 where they can
        B = args.pairs if args.pairs else max(16, min(4096, int(32 * (128 / n) ** 2)))
        g = torch.Generator(device=dev).manual_seed(1234 + n)
        feats = torch.relu(torch.randn(B, 3, 512, 2 * n, device=dev, generator=g))
        det = torch.rand(B, 2 * n, device=dev, generator=g)
        h_feats = torch.empty(feats.shape, dtype=torch.float32, pin_memory=True).copy_(feats)
        h_match = torch.empty(B, n, dtype=torch.int32, pin_memory=True)
        d_feats = torch.empty_like(feats)
        zn = torch.zeros(B, n, device=dev)

        last = {}

        def step(f):
            link, new, end = net.associate_batch(f, n)
            r = mmmot_b200.solve_batch(det, link[:, 2], torch.cat([zn, new[:, 2]], 1), torch.cat([end[:, 2], zn], 1), n, n)
            last.update(r, link=link, new=new, end=end)
            return r

        def step_e2e():
            d_feats.copy_(h_feats, non_blocking=True)
            r = step(d_feats)
            h_match.copy_(r["match"], non_blocking=True)

        def timed(fn, hooks):
            for _ in range(max(args.warmup, 3)):
                fn()
            torch.cuda.synchronize(dev)
            l0 = lib.mmmot_launch_count()
            if hooks:
                lib.mmmot_timing_enable(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            torch.cuda.synchronize(dev)
            lib.mmmot_timing_enable(0)
            return e0.elapsed_time(e1), lib.mmmot_launch_count() - l0, (collect_tags(lib) if hooks else None)
        ms, launches, tags = timed(lambda: step(feats), True)
        if args.dump_outputs:
            dumps.append((f"n{n}_", {f"n{n}_{k}": v for k, v in last.items()}, {}, B))
        ms2, _, _ = timed(step_e2e, False)
        pt = {"n": n, "pairs_per_step": B, "value": B * args.steps / (ms / 1e3), "e2e": B * args.steps / (ms2 / 1e3),
              "ms_per_step": ms / args.steps, "gpu_launches": int(launches),
              "algorithmic_tflops": B * args.steps / (ms / 1e3) * flop_per_pair(dict(c, n=n)) / 1e12,
              "kernels": kernel_table(tags, args.steps, peaks)}
        points.append(pt)
        if n == c["n"]:
            main = (pt, ms, ms2, launches, tags, B, h_feats.numel() * 4, h_match.numel() * 4)
    clocks = sampler.summary()
    pt, ms, ms2, launches, tags, B, h2d, d2h = main
    l1 = next(k for k in pt["kernels"] if k["kernel"].startswith("affinity.l1"))
    cpu = None
    if not args.no_cpu:
        cpu, _, _ = cpu_leg(c, args.cpu_pairs)
    line = {"metric": metric_name(c), "value": pt["value"], "unit": "frame-pairs/s", "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": pt["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (tcgen05 engine: FP16 hi/lo split operands, fp32 accumulate; LP in f64)",
            "data": "synthetic", "config": config_dict(c, name, B, 1, "weak"), "clocks": clocks,
            "e2e": {"value": pt["e2e"], "unit": "frame-pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms2 / args.steps},
            "gpu_launches": pt["gpu_launches"], "algorithmic_tflops": pt["algorithmic_tflops"],
            "roofline": {"bound": "tensor", "kernel": "gen::gemm_gen_kernel (affinity layer 1: pairwise operand generated in-kernel, "
                                                      "512 -> 1024, FP16 hi/lo split: 3 MMAs per algorithmic MAC)",
                         "achieved": l1["algorithmic_tflops"], "peak": peaks.get("bf16_tflops_sustained", 1400.0), "unit": "TFLOP/s",
                         "frac": l1["frac"], "peak_source": f"{how} bf16_tflops_sustained", "traffic": None},
            "kernels": pt["kernels"], "sweep": points, "cpu_baseline": cpu}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumps)
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- full forward + LP
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="cfg4", choices=sorted(CONFIGS))
    ap.add_argument("--pairs", type=int, default=int(os.environ.get("MMMOT_BENCH_PAIRS", "0")),
                    help="frame-pairs per GPU per step (default: the config's own batch)")
    ap.add_argument("--total-pairs", type=int, default=0, help="strong scaling: total frame-pairs per step, sharded over the ranks")
    ap.add_argument("--cpu-pairs", type=int, default=2, help="frame-pairs timed for cpu_baseline (rank 0)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--kseg", type=int, default=-1, help="tcgen05 conv K-segment length in 32-chunks (0 = off; default: library default)")
    ap.add_argument("--engine", default="auto", choices=["auto", "fp32", "tcgen05"],
                    help="contraction engine (A/B runs; default auto = tcgen05 for this workload)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0; at most "
                         "64 MB in all, a fixed seeded sample of the frame-pairs beyond that); the inputs are seeded, so two "
                         "builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's outputs; the reference arm has none")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    name = args.config
    c = CONFIGS[name]

    if args.impl == "reference":
        run_reference(args, c, name, rank)
        return
    if name == "cfg5":
        if rank == 0:
            run_sweep(args, c, name, rank, world, local)
        return

    import mmmot_b200
    from mmmot_b200 import _lib
    from mmmot_b200.parallel import gather_pairs, shard_range
    from mmmot_b200.synthetic import synthetic_state_dict
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the first communicator is created: keep stdout for the one
        # JSON line (the banner goes to stderr)
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            os.dup2(saved, 1)
            os.close(saved)
    lib = _lib.load()
    mmmot_b200.set_engine(args.engine)
    if args.kseg >= 0:
        lib.mmmot_set_kseg(args.kseg)

    n, pts, hw = c["n"], c["pts"], c["hw"]
    L = 2 * n
    if args.total_pairs:
        scaling, total = "strong", args.total_pairs
        lo, hi = shard_range(total, rank, world)
        B = hi - lo
    else:
        scaling, B = "weak", (args.pairs or c["pairs"])
        total = B * world
    net = mmmot_b200.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch=c["fusion"],
                                 affinity_op=c["affinity_op"], softmax_mode=c["softmax_mode"],
                                 neg_threshold=c["neg_threshold"], test_mode=2, dropblock=0)
    net.load_state_dict(synthetic_state_dict(c["fusion"], seed=0))
    net.cuda(dev).eval()

    def make_inputs(seed_rank, pairs):
        """synthetic inputs of the config's shape, generated on the device (seeded per rank)"""
        g = torch.Generator(device=dev).manual_seed(1234 + seed_rank)
        crops = torch.randn(pairs * L, 3, hw, hw, device=dev, generator=g)
        centre = torch.rand(pairs * L, 1, 3, device=dev, generator=g) * torch.tensor([60.0, 40.0, 2.0], device=dev) + \
            torch.tensor([0.0, -20.0, -2.0], device=dev)
        points = (torch.randn(pairs * L, pts, 3, device=dev, generator=g) * torch.tensor([2.0, 1.0, 0.8], device=dev) + centre).reshape(-1, 3)
        return crops, points, torch.arange(0, pairs * L * pts + 1, pts, dtype=torch.int32)
    crops, points, split = make_inputs(rank, B)
    # mirrored to pinned host memory for the end-to-end leg
    h_crops = torch.empty(crops.shape, dtype=torch.float32, pin_memory=True).copy_(crops)
    h_points = torch.empty(points.shape, dtype=torch.float32, pin_memory=True).copy_(points)

    last = {}

    def step_resident():
        o = net.predict_batch(crops, points, split, n, check=False)
        if world > 1:
            last["match"] = gather_pairs(o["match"], total)      # the path's only collective (SURVEY §8e)
        else:
            last["match"] = o["match"]
        last["status"] = o["status"]
        last["out"] = o
        return o

    # e2e = the package's own host pipeline (mmmot_b200.HostPipeline): pinned host -> device copies overlapped with
    # compute in sub-batches, results device -> host; every byte of every step's inputs crosses PCIe inside the timed
    # region.
    pipe = mmmot_b200.HostPipeline(net, n, sub_batches=4)

    def step_e2e():
        r = pipe.run(h_crops, h_points, split, sync=False)
        if world > 1:
            gather_pairs(r["match_device"], total)
        return r

    def timed(fn, steps, warmup, with_hooks=False):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        l0 = lib.mmmot_launch_count()
        if with_hooks:
            lib.mmmot_timing_enable(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        tags = None
        if with_hooks:
            lib.mmmot_timing_enable(0)
            tags = collect_tags(lib)
        launches = lib.mmmot_launch_count() - l0
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, launches, tags

    warm = max(args.warmup, 3)            # timing rule: >= 3 warm-up steps
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches, tags = timed(step_resident, args.steps, warm, with_hooks=True)
    clocks = sampler.summary() if sampler else None
    status = int(last["status"])
    sampler2 = ClockSampler(local) if rank == 0 else None
    if sampler2:
        sampler2.start()
    ms_e2e, _, _ = timed(step_e2e, args.steps, warm)
    clocks_e2e = sampler2.summary() if sampler2 else None
    status |= int(pipe.h_status.max())

    # N-GPU result == 1-GPU result: rank 0 recomputes rank 1's shard from the same seeded inputs and compares it bit
    # for bit with what the gather returned (outside the timed region)
    shard_equal = None
    if world > 1 and rank == 0:
        if scaling == "strong":
            l1, h1 = shard_range(total, 1, world)
        else:
            l1, h1 = B, 2 * B
        c1, p1, s1 = make_inputs(1, h1 - l1)
        o1 = net.predict_batch(c1, p1, s1, n)
        shard_equal = bool(torch.equal(o1["match"], last["match"][l1:h1]))

    if rank == 0:
        peaks, how = load_peaks()
        value = total * args.steps / (ms / 1e3)
        e2e = total * args.steps / (ms_e2e / 1e3)
        conv = [v for k, v in tags.items() if k.startswith("vgg.conv") and k != "vgg.conv0"]
        conv_ms, conv_flop, conv_n = sum(v[0] for v in conv), sum(v[1] for v in conv), sum(v[3] for v in conv)
        achieved = conv_flop / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        tc_engine = args.engine != "fp32"
        traffic, traffic_note = None, None
        for f in ("r02_conv_traffic.json", "r01_conv_traffic.json"):
            try:    # dram bytes per frame-pair of the 12 conv launches, from a committed ncu --set full capture of cfg4
                with open(os.path.join(ROOT, "profiles", f)) as fh:
                    tr = json.load(fh)
                if tc_engine and name == "cfg4":
                    traffic = tr["dram_bytes_per_pair"] * (B * args.steps * 12 / max(conv_n, 1)) / 12
                    traffic_note = f"avg dram bytes per launch, scaled from profiles/{f} (ncu --set full, dram__bytes_read+write)"
                break
            except Exception:
                continue
        roofline = {"bound": "tensor",
                    "kernel": ("tma::gemm_tma_kernel / gemm_tma_px_kernel, conv mode (TMA-fed tcgen05 3x3-conv contraction of the VGG "
                               "trunk, layers 1..12, FP16 hi/lo split: 3 MMAs per algorithmic MAC)") if tc_engine else
                              "gemm_simt_kernel<XM_CONV3> (VGG 3x3 conv contraction, FP32 FFMA engine)",
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "mma_issue_tflops": 3 * achieved if tc_engine else None,
                    "mma_issue_frac": 3 * achieved / peak if tc_engine else None,
                    "peak_source": f"{how} bf16_tflops_sustained (kernel timed inside a long step); 'achieved' counts "
                                   "ALGORITHMIC FLOPs (2*Cout*9Cin*pixels per launch); the tensor pipe executes 3x that",
                    "launches_timed": conv_n, "avg_launch_ms": conv_ms / max(conv_n, 1),
                    "share_of_step": conv_ms / ms, "traffic": traffic, "traffic_note": traffic_note}
        cpu = None
        if not args.no_cpu and world == 1:      # the CPU baseline is reported at N=1 only
            cpu, _, _ = cpu_leg(c, args.cpu_pairs)
        h2d, d2h = pipe.bytes_per_batch(h_crops, h_points, split)
        line = {"metric": metric_name(c), "value": value, "unit": "frame-pairs/s", "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None,
                "dtype": "f32 (tcgen05 engine: FP16 hi/lo split operands, fp32 accumulate)" if tc_engine else "f32",
                "data": "synthetic", "config": dict(config_dict(c, name, B, world, scaling), engine=args.engine),
                "clocks": clocks, "clocks_e2e": clocks_e2e,
                "e2e": {"value": e2e, "unit": "frame-pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "range_status": status,
                "algorithmic_tflops": value * flop_per_pair(c) / 1e12 / world,
                "roofline": roofline, "kernels": kernel_table(tags, args.steps, peaks), "cpu_baseline": cpu}
        if world > 1:
            line["shard_equal"] = shard_equal
        assert status == 0, "MMMOT_E_RANGE raised during the benchmark"
        if args.dump_outputs:
            o = last["out"]
            per_pair = {k: o[k] for k in ("det", "link", "new", "end", "assign_det", "assign_link", "assign_new",
                                          "assign_end", "match")}
            sets = [("", per_pair, {"trans1": o["trans"][0], "trans2": o["trans"][1], "status": o["status"]}, B)]
            if world > 1:        # what the final gather hands rank 0: every rank's assignment indices
                sets.append(("gathered_", {"gathered_match": last["match"]}, {}, total))
            dump_outputs(args.dump_outputs, sets)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
