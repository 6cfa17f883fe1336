"""GPU (-m gpu): the CUDA path, called through the C ABI, against the oracle and the committed
golden fixtures.  Tolerance: 1e-4 relative (BASELINE.json north_star) with the metric
max|a-b| / max|ref|; assignment outputs bit-exact."""
import pytest
import torch

from helpers import TOL, case_tol, check_close, det_close, frac_outside, golden_cases, relerr
import mmmot_b200
from mmmot_b200.synthetic import synthetic_batch, synthetic_pair, synthetic_state_dict
from oracle import lp_ref, torch_ref

pytestmark = pytest.mark.gpu
CASES = golden_cases()
# fraction of elements allowed outside the element-wise bound |a-b| <= 1e-4|ref| + 1e-6 (helpers.frac_outside; reported by
# every test that uses it).  Measured on the cfg4 pair: 2e-5 of the dual_add link entries, the worst by a factor 1.003 —
# softmax outputs of ~5e-3 whose absolute error (1.5e-6) is what the 4e-5 max-norm error leaves at that magnitude.
ELEM_OUTSIDE = 1e-3


def make_net(fusion, op, sm, thr, seed):
    net = mmmot_b200.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch=fusion,
                                 affinity_op=op, softmax_mode=sm, neg_threshold=thr, test_mode=2, dropblock=0)
    sd = synthetic_state_dict(fusion, seed=seed)
    net.load_state_dict(sd)
    return net.cuda().eval(), sd


@pytest.fixture(params=["fp32", "tcgen05"])
def engine(request):
    """Both contraction engines must meet the same parity bound."""
    mmmot_b200.set_engine(request.param)
    yield request.param
    mmmot_b200.set_engine("auto")


def _planes(x):
    """fp32 -> FP16 (hi, lo) planes stacked on a new leading axis (the tcgen05 engines' operand format)."""
    hi = x.half()
    return torch.stack([hi, (x - hi.float()).half()]).contiguous()


@pytest.mark.parametrize("M,K,S", [(128, 32, 256), (256, 96, 512), (64, 64, 300), (512, 512, 4099), (1024, 128, 1000),
                                   (128, 4608, 2048)])
def test_contraction_engines_vs_fp64(M, K, S):
    """Each contraction engine alone (C ABI test hooks) against an fp64 matmul: the FP32 FFMA engine, the TMA-fed
    tcgen05 engine (FP16 hi/lo planes in, fp32 out) and the generated-operand tcgen05 engine (GroupNorm+ReLU producer,
    fp32 channels-last in / out)."""
    import ctypes
    from mmmot_b200 import _lib
    from mmmot_b200.weights import pack_tc
    lib = _lib.load()
    g = torch.Generator().manual_seed(M + K + S)
    Wt, X, b = torch.randn(K, M, generator=g), torch.randn(K, S, generator=g), torch.randn(M, generator=g)
    ref = Wt.double().t() @ X.double() + b.double()[:, None]
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    Wt_d, X_d, b_d = Wt.cuda(), X.cuda(), b.cuda()
    Wp, wps = pack_tc(Wt)
    Wp = Wp.cuda()
    Y = torch.full((M, S), float("nan"), device="cuda")
    assert lib.mmmot_debug_linear(vp(Wt_d), None, 0.0, vp(b_d), vp(X_d), vp(Y), M, K, S, 1, None) == 0
    assert relerr(Y, ref) < 3e-5, "fp32 engine"
    # TMA-fed engine: X as channels-last planes [2][S][K], Y [S][M]
    Xp = _planes(X.t().contiguous()).cuda()
    Y2 = torch.full((S, M), float("nan"), device="cuda")
    assert lib.mmmot_debug_linear_planar(vp(Wp), wps, vp(b_d), vp(Xp), vp(Y2), M, K, S, None) == 0
    assert relerr(Y2.t(), ref) < 3e-5, "tma engine"
    # generated-operand engine: Y[S][M] = relu(X[S][K]*sc + sh) W^T + b, fp32 channels-last in and out
    if K <= 512 and K % 32 == 0:
        sc, sh = torch.rand(K, generator=g) + 0.5, torch.randn(K, generator=g) * 0.3
        ref3 = Wt.double().t() @ torch.relu(X.double() * sc.double()[:, None] + sh.double()[:, None]) + b.double()[:, None]
        Xc = X.t().contiguous().cuda()
        Y3 = torch.full((S, M), float("nan"), device="cuda")
        assert lib.mmmot_debug_linear_gen(vp(Wp), wps, vp(b_d), vp(Xc), vp(sc.cuda()), vp(sh.cuda()), vp(Y3), M, K, S, None) == 0
        torch.cuda.synchronize()
        assert relerr(Y3.t(), ref3) < 3e-5, "gen engine"


def test_fp16_range_is_reported_not_clamped():
    """VERDICT r1 weak #10: activations >= 65504 saturate in the FP16 hi/lo conversion of the tensor-core path; the
    library raises MMMOT_E_RANGE instead of returning clamped results.  The FP32 engine has no such limit."""
    from mmmot_b200 import _lib
    net, sd = make_net("C", "minus_abs", "dual_add", 0.2, 3)
    dets, info, split = synthetic_pair(16, 16, 32, 32, seed=8)
    args = (info["points"][0].cuda(), info["points_split"][0], 16, 16)
    mmmot_b200.set_engine("tcgen05")
    try:
        o = net.forward_batch(dets.cuda(), *args)
        assert int(o["status"]) == 0
        with pytest.raises(_lib.MmmotError, match="MMMOT_E_RANGE"):
            net.forward_batch(dets.cuda() * 1e6, *args)
        o = net.forward_batch(dets.cuda() * 1e6, *args, check=False)     # deferred check: the flag travels with the outputs
        assert int(o["status"]) & 1
        mmmot_b200.set_engine("fp32")
        o = net.forward_batch(dets.cuda() * 1e6, *args)
        assert int(o["status"]) == 0 and torch.isfinite(o["link"]).all()
    finally:
        mmmot_b200.set_engine("auto")


def test_fetch_pinned_i32():
    """mmmot_fetch_pinned_i32: stream-ordered host -> device transfer of the CSR offsets by a kernel reading pinned host
    memory (no copy engine, no host synchronisation); pageable memory is refused loudly."""
    import ctypes
    from mmmot_b200 import _lib
    lib = _lib.load()
    for n in (1, 257, 8193, 100001):
        src = torch.empty(n, dtype=torch.int32, pin_memory=True).copy_(torch.arange(n, dtype=torch.int32) * 3 - 7)
        dst = torch.full((n + 1,), -1, dtype=torch.int32, device="cuda")
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        assert lib.mmmot_fetch_pinned_i32(ctypes.c_void_p(dst.data_ptr()), ctypes.c_void_p(src.data_ptr()), n, st) == 0
        assert torch.equal(dst[:n].cpu(), src) and int(dst[n]) == -1
    pageable = torch.arange(16, dtype=torch.int32)
    dst = torch.zeros(16, dtype=torch.int32, device="cuda")
    assert lib.mmmot_fetch_pinned_i32(ctypes.c_void_p(dst.data_ptr()), ctypes.c_void_p(pageable.data_ptr()), 16, None) == -1
    torch.cuda.synchronize()


def test_score_arch_branch_reg_has_no_sigmoid():
    """reference tracking_net.py:153-156: the sigmoid is applied only when 'cls' is in score_arch."""
    dets, info, split = synthetic_pair(6, 6, 24, 32, seed=2)
    outs = {}
    for arch in ("branch_cls", "branch_reg"):
        net = mmmot_b200.TrackingNet(2, appear_skippool=True, score_arch=arch, score_fusion_arch="A", neg_threshold=-10.0,
                                     test_mode=2, dropblock=0)
        net.load_state_dict(synthetic_state_dict("A", seed=6))
        net.cuda().eval()
        outs[arch] = net(dets.cuda(), {k: v.cuda() for k, v in info.items()}, split)[0]
    assert torch.allclose(torch.sigmoid(outs["branch_reg"]), outs["branch_cls"], atol=1e-6)
    assert (outs["branch_reg"].abs() > 1e-3).any()


@pytest.mark.parametrize("g", CASES, ids=[c["case"][0] for c in CASES])
def test_forward_matches_reference_golden(g, engine):
    """Reference signature, one frame-pair, against outputs of the UNMODIFIED reference."""
    name, fusion, op, sm, thr, n, m, pts, hw, ragged, seed = g["case"]
    net, sd = make_net(fusion, op, sm, thr, seed)
    dets, info, split = synthetic_pair(n, m, pts, hw, seed=seed, ragged=ragged)
    det, link, new, end, trans = net(dets.cuda(), {k: v.cuda() for k, v in info.items()}, split)
    tol = case_tol(g["case"])
    assert link[0].shape == g["link"].shape and det.shape == g["det"].shape
    assert relerr(link[0], g["link"]) < tol
    assert relerr(new, g["new"]) < tol and relerr(end, g["end"]) < tol
    assert det_close(det, g["det"], thr, tol)
    assert relerr(trans[0], g["trans1"]) < 1e-5 and relerr(trans[1], g["trans2"]) < 1e-5
    assert torch.all(new[:, :n] == 0) and torch.all(end[:, n:] == 0)


@pytest.mark.parametrize("fusion,op,sm", [("A", "multiply", "none"), ("C", "minus_abs", "dual_add"), ("B", "multiply", "none")])
def test_features_match_oracle(fusion, op, sm, engine):
    """Stage check: the 3x512xL feature stack (appearance | PointNet | fusion), N=M=16, 64x64 crops."""
    net, sd = make_net(fusion, op, sm, 0.2, 31)
    dets, info, split = synthetic_pair(16, 16, 48, 64, seed=31, ragged=True)
    o = net.forward_batch(dets.cuda(), info["points"][0].cuda(), info["points_split"][0], 16, 16, keep_feats=True)
    _, st = torch_ref.forward(sd, dets, info, split, fusion, op, sm, 0.2, return_stages=True)
    for s in range(3):
        assert relerr(o["feats"][0, s], st["feats"][s]) < TOL, f"stack {s}"


@pytest.mark.parametrize("n,m", [(8, 8), (32, 32), (64, 64), (20, 45), (128, 128)])
@pytest.mark.parametrize("op,sm", [("multiply", "none"), ("minus_abs", "dual_add")])
def test_affinity_stage_matches_oracle(n, m, op, sm, engine):
    """BASELINE config 5 (N sweep): affinity + start/end + softmax alone on identical feature tensors."""
    net, sd = make_net("C", op, sm, 0.2, 7)
    g = torch.Generator().manual_seed(n * 1000 + m)
    feats = torch.relu(torch.randn(2, 3, 512, n + m, generator=g))
    link, new, end = net.associate_batch(feats.cuda(), n, m)
    for b in range(2 if n <= 64 else 1):
        rl, rn, re = torch_ref.associate(sd, feats[b, :, :, :n], feats[b, :, :, n:], op, sm)
        assert relerr(link[b], rl.squeeze(1)) < TOL
        assert relerr(new[b], rn) < TOL and relerr(end[b], re) < TOL


@pytest.mark.parametrize("hw,n", [(96, 3), (224, 1), (576, 1)])
def test_non_power_of_two_crops(hw, n, engine):
    """Crop sizes that are multiples of 32 but not powers of two (224 is the reference's real crop size,
    dataset/test_seq_dataset.py:217-218): partial TMA boxes / tile tails.  576 is wider than the first VGG layer's
    in-kernel operand producers stage (512), so the tcgen05 engine takes the im2col27 pre-pass there."""
    net, sd = make_net("A", "multiply", "none", 0.2, 12)
    dets, info, split = synthetic_pair(n, n, 32, hw, seed=50 + hw)
    o = net.forward_batch(dets.cuda(), info["points"][0].cuda(), info["points_split"][0], n, n, keep_feats=True)
    _, st = torch_ref.forward(sd, dets, info, split, "A", "multiply", "none", 0.2, return_stages=True)
    assert relerr(o["feats"][0, 0], st["feats"][0]) < TOL


def test_affinity_n256_top_of_sweep():
    """BASELINE config 5, N = 256 (top of the N sweep), one pair, tensor-core engine vs oracle."""
    net, sd = make_net("C", "minus_abs", "dual_add", 0.2, 7)
    g = torch.Generator().manual_seed(256)
    feats = torch.relu(torch.randn(1, 3, 512, 512, generator=g))
    link, new, end = net.associate_batch(feats.cuda(), 256, 256)
    rl, rn, re = torch_ref.associate(sd, feats[0, :, :, :256], feats[0, :, :, 256:], "minus_abs", "dual_add")
    assert relerr(link[0], rl.squeeze(1)) < TOL and relerr(new[0], rn) < TOL and relerr(end[0], re) < TOL


def test_batched_equals_looped():
    """forward_batch over B pairs == B single-pair forwards (pairs are independent GroupNorm domains)."""
    net, sd = make_net("C", "minus_abs", "dual_add", 0.2, 5)
    B, n = 3, 8
    crops, pts, split = synthetic_batch(B, n, pts=24, hw=32, seed=40)
    net.chunk_pairs = 2          # also exercises chunking
    o = net.forward_batch(crops.cuda(), pts.cuda(), split, n)
    net.chunk_pairs = None
    for b in range(B):
        dets, info, ds = synthetic_pair(n, n, 24, 32, seed=40 + b)
        det, link, new, end, _ = net(dets.cuda(), {k: v.cuda() for k, v in info.items()}, ds)
        assert torch.equal(o["link"][b], link[0]) and torch.equal(o["det"][b], det)
        assert torch.equal(o["new"][b], new[:, n:]) and torch.equal(o["end"][b], end[:, :n])


def test_host_pipeline_equals_predict_batch():
    """HostPipeline (pinned host -> overlapped H2D -> predict_batch per sub-batch -> D2H; what bench.py times as e2e)
    returns exactly what predict_batch returns on device-resident inputs, on ragged point counts, across repeated runs
    (buffer / pinned-slot reuse) and for a batch that cannot be cut into sub-batches."""
    net, sd = make_net("C", "minus_abs", "dual_add", 0.2, 5)
    n = 8
    for B, seed in ((8, 50), (3, 60)):
        ds, ps, sp, off = [], [], [torch.zeros(1, dtype=torch.int64)], 0
        for b in range(B):
            d, info, _ = synthetic_pair(n, n, 24, 32, seed=seed + b, ragged=True)
            ds.append(d); ps.append(info["points"][0])
            s_ = info["points_split"][0].long()
            sp.append(s_[1:] + off); off += int(s_[-1])
        crops, pts, split = torch.cat(ds), torch.cat(ps), torch.cat(sp)
        ref = net.predict_batch(crops.cuda(), pts.cuda(), split, n)
        pipe = mmmot_b200.HostPipeline(net, n, sub_batches=4)
        h_crops, h_pts = crops.pin_memory(), pts.pin_memory()
        for _ in range(3):
            r = pipe.run(h_crops, h_pts, split)
            assert torch.equal(r["match"], ref["match"].cpu()) and torch.equal(r["match_device"], ref["match"])
            for k in ("assign_det", "assign_new", "assign_end"):
                assert torch.equal(r[k], ref[k].cpu()), k
        assert pipe.nsub == (4 if B == 8 else 1)
        h2d, d2h = pipe.bytes_per_batch(h_crops, h_pts, split)
        assert h2d == crops.numel() * 4 + pts.numel() * 4 + split.numel() * 4 and d2h > 0
    # the range flag travels through the pipeline too
    from mmmot_b200 import _lib
    mmmot_b200.set_engine("tcgen05")
    try:
        with pytest.raises(_lib.MmmotError, match="MMMOT_E_RANGE"):
            pipe.run((h_crops * 1e6).pin_memory(), h_pts, split)
    finally:
        mmmot_b200.set_engine("auto")


# ------------------------------------------------------------------ LP
def _rand_lp(g, n, m, B=1):
    L = n + m
    det = torch.rand(B, L, generator=g) - (torch.rand(B, L, generator=g) < 0.3).float()
    link = torch.rand(B, n, m, generator=g)
    new = torch.cat([torch.zeros(B, n), torch.rand(B, m, generator=g)], 1)
    end = torch.cat([torch.rand(B, n, generator=g), torch.zeros(B, m)], 1)
    return det, link, new, end


def _assert_same_assignment(got, ref):
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1][0], ref[1][0])
    assert torch.equal(got[2], ref[2]) and torch.equal(got[3], ref[3])


@pytest.mark.parametrize("n,m", [(1, 1), (3, 2), (8, 8), (7, 19), (16, 16), (32, 32), (64, 64), (128, 128), (100, 128),
                                 (256, 256)])
def test_lp_bit_exact_vs_milp_oracle(n, m):
    """Every N of BASELINE's sweep (8..256, plus ragged shapes): the warp-per-pair Hungarian kernel returns the
    SAME 0/1 tensors as the MILP restatement of solvers.py:17-111 (HiGHS) and as the independent assignment
    reduction solved by scipy.linear_sum_assignment.  Random continuous scores: the optimum is unique."""
    g = torch.Generator().manual_seed(100 + n + m)
    B = 6 if n <= 64 else 4
    det, link, new, end = _rand_lp(g, n, m, B)
    r = mmmot_b200.solve_batch(det.cuda(), link.cuda(), new.cuda(), end.cuda(), n, m)
    for b in range(B):
        (a, obj, y) = lp_ref.milp_solve(det[b], [link[b:b + 1]], new[b], end[b], [n, m])
        a2, obj2 = lp_ref.assignment_solve(det[b], [link[b:b + 1]], new[b], end[b], [n, m])
        got = (r["assign_det"][b].cpu(), [r["assign_link"][b:b + 1].cpu()], r["assign_new"][b].cpu(), r["assign_end"][b].cpu())
        assert abs(lp_ref.objective(det[b], [link[b:b + 1]], new[b], end[b], got) - obj) < 1e-9
        assert abs(obj - obj2) < 1e-8
        _assert_same_assignment(got, a)
        _assert_same_assignment(got, a2)
        mt = r["match"][b].cpu()
        assert torch.equal(mt >= 0, a[1][0][0].sum(1) > 0)
        assert torch.equal(mt.clamp_min(0)[mt >= 0].long(), a[1][0][0].argmax(1)[mt >= 0])


def test_lp_reference_signature_on_forward_outputs():
    """ortools_solve drop-in on the oracle's own score tensors (identical inputs -> identical indices)."""
    g = CASES[3]
    name, fusion, op, sm, thr, n, m = g["case"][:7]
    t = 2
    a = mmmot_b200.ortools_solve(g["det"][t].cuda(), [g["link"][t:t + 1].cuda()], g["new"][t].cuda(), g["end"][t].cuda(),
                                 [torch.tensor([n]), torch.tensor([m])])
    b, obj, _ = lp_ref.milp_solve(g["det"][t], [g["link"][t:t + 1]], g["new"][t], g["end"][t], [n, m])
    assert a[1][0].shape == (1, n, m) and a[0].dtype == torch.float32 and a[0].is_cuda
    assert torch.equal(a[0].cpu(), b[0]) and torch.equal(a[1][0].cpu(), b[1][0])
    assert torch.equal(a[2].cpu(), b[2]) and torch.equal(a[3].cpu(), b[3])


@pytest.mark.parametrize("n", [128, 256])
def test_lp_large_optimality_and_feasibility(n):
    """Full-size instances (BASELINE N=128, sweep top 256): objective equals scipy's assignment optimum
    of the (N+M)^2 reduction, and the flow constraints of solvers.py:83-111 hold."""
    import numpy as np
    from scipy.optimize import linear_sum_assignment
    g = torch.Generator().manual_seed(n)
    B = 4
    det, link, new, end = _rand_lp(g, n, n, B)
    r = mmmot_b200.solve_batch(det.cuda(), link.cuda(), new.cuda(), end.cuda(), n, n)
    for b in range(B):
        ad, al, an, ae = [r[k][b].cpu() for k in ("assign_det", "assign_link", "assign_new", "assign_end")]
        assert torch.equal(ae[:n] + al.sum(1), ad[:n]) and torch.equal(an[:n], ad[:n])
        assert torch.equal(an[n:] + al.sum(0), ad[n:]) and torch.equal(ae[n:], ad[n:])
        d, l, nw, e = [t.double().numpy() for t in (det[b], link[b], new[b], end[b])]
        aj, bk = d[:n] + nw[:n], d[n:] + e[n:]
        C = np.full((2 * n, 2 * n), -1e9)
        C[:n, :n] = aj[:, None] + bk[None, :] + l
        C[:n, n:][np.arange(n), np.arange(n)] = np.maximum(aj + e[:n], 0)
        C[n:, :n][np.arange(n), np.arange(n)] = np.maximum(bk + nw[n:], 0)
        C[n:, n:] = 0
        rr, cc = linear_sum_assignment(C, maximize=True)
        got = lp_ref.objective(det[b], [link[b:b + 1]], new[b], end[b], (ad, [al.unsqueeze(0)], an, ae))
        assert abs(got - C[rr, cc].sum()) < 1e-8


def test_predict_batch_full_size_property():
    """BASELINE N=128 shape end to end (1 pair): every output finite, softmax rows/cols consistent,
    assignment feasible."""
    net, sd = make_net("C", "minus_abs", "dual_add", 0.2, 9)
    n = 128
    crops, pts, split = synthetic_batch(1, n, pts=64, hw=64, seed=77)
    o = net.predict_batch(crops.cuda(), pts.cuda(), split, n)
    for k in ("det", "link", "new", "end"):
        assert torch.isfinite(o[k]).all(), k
    assert (o["link"] >= 0).all() and (o["link"] <= 1).all()      # dual_add of two softmaxes
    al, ad = o["assign_link"][0], o["assign_det"][0]
    assert al.sum(1).max() <= 1 and al.sum(0).max() <= 1
    assert torch.equal(o["assign_end"][0][:n] + al.sum(1), ad[:n])


def test_cfg4_full_size_pair_matches_oracle():
    """One frame-pair at exactly the bench configuration (BASELINE configs[3] / SURVEY cfg4: Fusion C, minus_abs, dual_add,
    N=M=128, P=512 points per detection, 64x64 crops) against the oracle — the size the throughput is quoted on.
    The oracle needs ~10 s of host time for this pair."""
    net, sd = make_net("C", "minus_abs", "dual_add", 0.2, 4)
    n = 128
    dets, info, split = synthetic_pair(n, n, 512, 64, seed=123)
    torch.set_num_threads(min(16, torch.get_num_threads()))
    ref_det, ref_link, ref_new, ref_end, _ = torch_ref.forward(sd, dets, info, split, "C", "minus_abs", "dual_add", 0.2)
    det, link, new, end, _ = net(dets.cuda(), {k: v.cuda() for k, v in info.items()}, split)
    rep = []
    check_close(link[0], ref_link[0], TOL, "link", rep, max_outside=ELEM_OUTSIDE)
    check_close(new, ref_new, TOL, "new", rep, max_outside=ELEM_OUTSIDE)
    check_close(end, ref_end, TOL, "end", rep, max_outside=ELEM_OUTSIDE)
    assert det_close(det, ref_det, 0.2, TOL)
    print("cfg4 pair (what, max-norm rel err, fraction outside element-wise bound, worst ratio):", rep)
    # (1) identical inputs -> identical indices: the GPU solver on the ORACLE's score tensors equals the MILP
    #     restatement and the assignment reduction bit for bit (north_star: "assignment indices bit-exact")
    t = 2
    b = mmmot_b200.ortools_solve(ref_det[t].cuda(), [ref_link[0][t:t + 1].cuda()], ref_new[t].cuda(), ref_end[t].cuda(), split)
    b = (b[0].cpu(), [b[1][0].cpu()], b[2].cpu(), b[3].cpu())
    (mil, obj, y) = lp_ref.milp_solve(ref_det[t], [ref_link[0][t:t + 1]], ref_new[t], ref_end[t], [n, n])
    lsa, _ = lp_ref.assignment_solve(ref_det[t], [ref_link[0][t:t + 1]], ref_new[t], ref_end[t], [n, n])
    _assert_same_assignment(b, mil)
    _assert_same_assignment(b, lsa)
    # (2) end to end (GPU scores -> GPU solver) against (oracle scores -> oracle solver): the two score sets differ by
    #     fp32 round-off, so the optimum can only move if the gap to the second-best solution is smaller than the
    #     total score perturbation.  Measure both; demand exact equality whenever the gap exceeds the perturbation.
    a = mmmot_b200.ortools_solve(det[t], [link[0][t:t + 1]], new[t], end[t], split)
    a = (a[0].cpu(), [a[1][0].cpu()], a[2].cpu(), a[3].cpu())
    perturb = float((det[t].cpu() - ref_det[t]).abs().sum() + (link[0][t].cpu() - ref_link[0][t]).abs().sum()
                    + (new[t].cpu() - ref_new[t]).abs().sum() + (end[t].cpu() - ref_end[t]).abs().sum())
    (_, obj2, _) = lp_ref.milp_solve(ref_det[t], [ref_link[0][t:t + 1]], ref_new[t], ref_end[t], [n, n], exclude=y)
    gap = obj - obj2
    same = all(torch.equal(p, q) for p, q in ((a[0], mil[0]), (a[1][0], mil[1][0]), (a[2], mil[2]), (a[3], mil[3])))
    print(f"cfg4 pair: LP optimum {obj:.6f}, second-best gap {gap:.3e}, L1 score perturbation {perturb:.3e}, identical={same}")
    if gap > perturb:
        assert same, (gap, perturb)
    else:   # near-tie: the GPU-side optimum must still be optimal to within the perturbation under the oracle's scores
        got = lp_ref.objective(ref_det[t], [ref_link[0][t:t + 1]], ref_new[t], ref_end[t], a)
        assert obj - got <= perturb + 1e-9, (obj, got, perturb)


# ------------------------------------------------------------------ BASELINE configs at their stated shapes
@pytest.mark.parametrize("name,fusion,op,sm,n,pts,hw", [
    ("cfg2", "A", "multiply", "none", 32, 128, 64),       # BASELINE configs[1]: pp_pv_40e_mul_A, N=32, 64x64 crops
    ("cfg3", "C", "multiply", "none", 64, 512, 64),       # BASELINE configs[2]: pp_pv_40e_mul_C, N=64, P=512
    ("crop224", "C", "minus_abs", "dual_add", 4, 96, 224),  # the reference's real crop size (test_seq_dataset.py:217-218)
])
def test_full_forward_at_baseline_config(name, fusion, op, sm, n, pts, hw):
    """Full forward (all five outputs + the feature stacks) of one frame-pair at the shapes BASELINE.json states for
    cfg2 / cfg3, and a multi-detection pair at 224x224 crops, against the oracle; max-norm and element-wise metrics."""
    net, sd = make_net(fusion, op, sm, 0.2, 21)
    dets, info, split = synthetic_pair(n, n, pts, hw, seed=300 + n, ragged=(name == "crop224"))
    torch.set_num_threads(min(16, torch.get_num_threads()))
    (rdet, rlink, rnew, rend, _), st = torch_ref.forward(sd, dets, info, split, fusion, op, sm, 0.2, return_stages=True)
    o = net.forward_batch(dets.cuda(), info["points"][0].cuda(), info["points_split"][0], n, n, keep_feats=True)
    rep = []
    for s_ in range(3):     # intermediate feature stacks: max-norm metric (GroupNorm outputs cross zero, so a bound relative to
        e = relerr(o["feats"][0, s_], st["feats"][s_])          # each element's own magnitude is meaningless there)
        rep.append((f"{name} feats[{s_}]", e))
        assert e < TOL, rep[-1]
    check_close(o["link"][0], rlink[0], TOL, f"{name} link", rep, max_outside=ELEM_OUTSIDE)
    check_close(o["new"][0], rnew[:, n:], TOL, f"{name} new", rep, max_outside=ELEM_OUTSIDE)
    check_close(o["end"][0], rend[:, :n], TOL, f"{name} end", rep, max_outside=ELEM_OUTSIDE)
    assert det_close(o["det"][0], rdet, 0.2, TOL)
    print(name, rep)


# ------------------------------------------------------------------ training mode (SURVEY §8f N4)
from helpers import LOSS_KW, synthetic_gt, train_cases  # noqa: E402

TRAIN = train_cases()


@pytest.mark.parametrize("g", TRAIN, ids=[c["case"][0] for c in TRAIN])
def test_training_mode_forward_and_loss_match_reference_golden(g):
    """TrackingNet.train(): BatchNorm batch statistics in the VGG trunk and w_det, raw det logits, unpadded new/end
    scores, running-average update, and TrackingModule.step's loss — against the UNMODIFIED reference in .train() mode."""
    name, fusion, op, sm, n, m, pts, hw, ragged, seed = g["case"]
    net = mmmot_b200.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch=fusion, affinity_op=op,
                                 softmax_mode=sm, neg_threshold=0.2, test_mode=2, **g.get("drop", dict(dropblock=0, use_dropout=False)))
    net.load_state_dict(synthetic_state_dict(fusion, seed=seed))
    net.cuda().train()
    # the golden ran the reference on the CPU, so its Dropout mask came from the CPU generator too: draw it there
    net._dropout_mask = lambda shape, dev, p=0.5: torch.nn.functional.dropout(torch.ones(shape), p=p, training=True).to(dev)
    dets, info, split = synthetic_pair(n, m, pts, hw, seed=seed, ragged=ragged)
    cls, ids = synthetic_gt(n, m, seed)
    tm = mmmot_b200.TrackingModule(net, None, mmmot_b200.TrackingLoss(**LOSS_KW))
    dinfo = {k: v.cuda() for k, v in info.items()}
    torch.manual_seed(seed)       # DropBlock / Dropout draws start where the golden's did (make_goldens.py)
    det, link, new, end, trans = net(dets.cuda(), dinfo, split)
    assert det.shape == (3, n + m) and new.shape == (3, m) and end.shape == (3, n)
    assert relerr(det, g["det"]) < TOL and relerr(link[0], g["link"]) < TOL
    assert relerr(new, g["new"]) < TOL and relerr(end, g["end"]) < TOL
    sd_after = net.state_dict()
    for k, v in g["running"].items():
        if k.startswith("appearance.layers") or k.startswith("w_det"):
            if k.endswith("num_batches_tracked"):
                assert int(sd_after[k]) == int(v), k
            else:
                assert relerr(sd_after[k], v) < 1e-4, k
    # the loss through TrackingModule.step (second training-mode forward: the outputs do not depend on running stats)
    torch.manual_seed(seed)
    loss = tm.step(dets.cuda(), dinfo, ids, cls, split)
    assert abs(float(loss) - float(g["loss"])) < 2e-4 * abs(float(g["loss"]))
    # back to eval: the eval forward still works and pads / squashes as before
    net.eval()
    d2, l2, n2, e2, _ = net(dets.cuda(), dinfo, split)
    assert n2.shape == (3, n + m) and (d2 <= 1).all()


def test_multi_frame_sample_and_end_mode_max():
    """VERDICT r1 missing #6: samples of more than two frames (tracking_net.py:170-182) and NewEndIndicator_v2 mode 'max'
    (new_end.py:73-74), against the oracle."""
    fusion, op, sm = "C", "minus_abs", "dual_add"
    splits = [5, 7, 4]
    L = sum(splits)
    g = torch.Generator().manual_seed(77)
    for end_mode in ("avg", "max"):
        net = mmmot_b200.TrackingNet(3, appear_skippool=True, score_arch="branch_cls", score_fusion_arch=fusion, affinity_op=op,
                                     softmax_mode=sm, neg_threshold=0.2, test_mode=2, dropblock=0, end_mode=end_mode)
        sd = synthetic_state_dict(fusion, seed=13)
        net.load_state_dict(sd)
        net.cuda().eval()
        dets, info, _ = synthetic_pair(splits[0], L - splits[0], 24, 32, seed=61, ragged=True)
        ds = [torch.tensor([k]) for k in splits]
        det, link, new, end, _ = net(dets.cuda(), {k: v.cuda() for k, v in info.items()}, ds)
        rdet, rlink, rnew, rend, _ = torch_ref.forward(sd, dets, info, ds, fusion, op, sm, 0.2, end_mode=end_mode)
        assert len(link) == 2 and link[1].shape == (3, 7, 4) and new.shape == (3, L)
        for a, b in zip(link, rlink):
            assert relerr(a, b) < TOL
        assert relerr(new, rnew) < TOL and relerr(end, rend) < TOL and det_close(det, rdet, 0.2, TOL)
        assert torch.all(new[:, :5] == 0) and torch.all(end[:, -4:] == 0)
    # end_mode 'max' on a shape that takes the tensor-core path (N*M >= 256)
    net2, sd2 = make_net("C", "multiply", "none", 0.2, 7)
    net2.end_mode = "max"
    feats = torch.relu(torch.randn(1, 3, 512, 40, generator=g))
    lk, nw, en = net2.associate_batch(feats.cuda(), 20, 20)
    rl, rn, re = torch_ref.associate(sd2, feats[0, :, :, :20], feats[0, :, :, 20:], "multiply", "none", end_mode="max")
    assert relerr(lk[0], rl.squeeze(1)) < TOL and relerr(nw[0], rn) < TOL and relerr(en[0], re) < TOL
