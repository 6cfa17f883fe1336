"""CPU: the oracle restatement against the golden fixtures produced by the UNMODIFIED reference
(oracle/make_goldens.py), plus known-answer tests the reference never had (SURVEY §4)."""
import numpy as np
import os
import types

import pytest
import torch

from helpers import GOLDEN_DIR, case_tol, golden_cases, relerr
from mmmot_b200.synthetic import synthetic_pair, synthetic_state_dict
from oracle import lp_ref, torch_ref

CASES = golden_cases()


def test_goldens_present():
    assert len(CASES) >= 8


@pytest.mark.parametrize("g", CASES, ids=[c["case"][0] for c in CASES])
def test_oracle_matches_reference_golden(g):
    name, fusion, op, sm, thr, n, m, pts, hw, ragged, seed = g["case"]
    sd = synthetic_state_dict(fusion, seed=seed)
    dets, info, split = synthetic_pair(n, m, pts, hw, seed=seed, ragged=ragged)
    (det, link, new, end, trans), st = torch_ref.forward(sd, dets, info, split, fusion, op, sm, thr,
                                                         return_stages=True)
    tol = case_tol(g["case"])
    assert relerr(st["feats"], g["feats"]) < tol
    assert relerr(det, g["det"]) < tol
    assert relerr(link[0], g["link"]) < tol
    assert relerr(new, g["new"]) < tol
    assert relerr(end, g["end"]) < tol
    assert relerr(trans[0], g["trans1"]) < 1e-5 and relerr(trans[1], g["trans2"]) < 1e-5
    # eval-mode zero padding (tracking_net.py:183-189)
    assert torch.all(new[:, :n] == 0) and torch.all(end[:, n:] == 0)


@pytest.mark.parametrize("g", CASES[:3], ids=[c["case"][0] for c in CASES[:3]])
def test_stn_is_input_independent_constant(g):
    """SURVEY F4: the STN output equals I + reshape(W_out relu(beta) + b_out) for any input."""
    fusion, seed = g["case"][1], g["case"][10]
    sd = synthetic_state_dict(fusion, seed=seed)
    assert relerr(torch_ref.stn_constant(sd, "point_net.feat.stn1", 3), g["trans1"]) < 1e-6
    assert relerr(torch_ref.stn_constant(sd, "point_net.feat.stn2", 64), g["trans2"]) < 1e-6
    from mmmot_b200.weights import stn_constant
    assert relerr(stn_constant(sd, "point_net.feat.stn2", 64).float(), g["trans2"][0]) < 1e-6


def test_oracle_vs_live_reference_cfg1():
    """BASELINE config[0]: Fusion-A, N=8 plumbing case at 64x64 crops, against the outputs the unmodified reference
    computed for it (oracle/make_goldens.py::live_golden)."""
    from oracle.make_goldens import LIVE_CASE
    name, fusion, op, sm, thr, n, m, pts, hw, ragged, seed = LIVE_CASE
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    ref = {k: torch.from_numpy(g[k]) for k in ("det", "link", "new", "end")}
    sd = synthetic_state_dict(fusion, seed=seed)
    dets, info, split = synthetic_pair(n, m, pts, hw, seed=seed, ragged=ragged)
    det, link, new, end, _ = torch_ref.forward(sd, dets, info, split, fusion, op, sm, thr)
    assert relerr(link[0], ref["link"]) < 1e-4 and relerr(det, ref["det"]) < 1e-4
    assert relerr(new, ref["new"]) < 1e-4 and relerr(end, ref["end"]) < 1e-4


# ------------------------------------------------------------------ LP oracle
def _rand_lp(g, n, m):
    L = n + m
    det = torch.rand(L, generator=g) - (torch.rand(L, generator=g) < 0.3).float()
    link = torch.rand(1, n, m, generator=g)
    new = torch.cat([torch.zeros(n), torch.rand(m, generator=g)])
    end = torch.cat([torch.rand(n, generator=g), torch.zeros(m)])
    return det, link, new, end


def test_milp_restatement_matches_brute_force():
    g = torch.Generator().manual_seed(0)
    for _ in range(25):
        n = int(torch.randint(1, 4, (1,), generator=g))
        m = int(torch.randint(1, 4, (1,), generator=g))
        det, link, new, end = _rand_lp(g, n, m)
        a, obj, _ = lp_ref.milp_solve(det, [link], new, end, [n, m])
        b, best, gap = lp_ref.brute_force(det, [link], new, end, [n, m])
        assert abs(obj - best) < 1e-9
        if gap > 1e-6:
            assert all(torch.equal(x, y) for x, y in zip([a[0], a[1][0], a[2], a[3]], [b[0], b[1][0], b[2], b[3]]))
        assert abs(lp_ref.objective(det, [link], new, end, a) - obj) < 1e-9


def test_milp_equals_assignment_reduction():
    """SURVEY F9: for 2 frames the MIP equals an (N+M)x(M+N) assignment problem."""
    from scipy.optimize import linear_sum_assignment
    g = torch.Generator().manual_seed(5)
    for n, m in ((8, 8), (12, 7), (5, 16)):
        det, link, new, end = _rand_lp(g, n, m)
        a, obj, _ = lp_ref.milp_solve(det, [link], new, end, [n, m])
        d, l, nw, e = [t.double().numpy() for t in (det, link[0], new, end)]
        aj, bk = d[:n] + nw[:n], d[n:] + e[n:]
        C = np.full((n + m, m + n), -1e9)
        C[:n, :m] = aj[:, None] + bk[None, :] + l
        C[:n, m:][np.arange(n), np.arange(n)] = np.maximum(aj + e[:n], 0)
        C[n:, :m][np.arange(m), np.arange(m)] = np.maximum(bk + nw[n:], 0)
        C[n:, m:] = 0
        r, c = linear_sum_assignment(C, maximize=True)
        assert abs(C[r, c].sum() - obj) < 1e-9


# ------------------------------------------------------------------ training mode (SURVEY §8f N4)
from helpers import LOSS_KW, synthetic_gt, train_cases  # noqa: E402

TRAIN = train_cases()


@pytest.mark.parametrize("g", TRAIN, ids=[c["case"][0] for c in TRAIN])
def test_train_oracle_matches_reference_golden(g):
    """oracle/train_ref.py (training-mode forward, running-average update, loss) against the UNMODIFIED reference in
    .train() mode; and the product's host-side pieces (generate_gt, TrackingLoss) against the same fixtures."""
    import mmmot_b200
    from oracle import train_ref
    name, fusion, op, sm, n, m, pts, hw, ragged, seed = g["case"]
    sd = synthetic_state_dict(fusion, seed=seed)
    dets, info, split = synthetic_pair(n, m, pts, hw, seed=seed, ragged=ragged)
    torch.manual_seed(seed)       # the DropBlock / Dropout draws of the golden start from this state (make_goldens.py)
    (det, link, new, end, trans), stats = train_ref.forward_train(sd, dets, info, split, fusion, op, sm, **g.get("drop", {}))
    assert relerr(det, g["det"]) < 5e-5 and relerr(link[0], g["link"]) < 5e-5
    assert relerr(new, g["new"]) < 5e-5 and relerr(end, g["end"]) < 5e-5
    assert new.shape == (3, m) and end.shape == (3, n)                 # no zero padding in training mode
    run = train_ref.running_after(sd, stats)
    for k, v in run.items():
        assert relerr(v, g["running"][k]) < 1e-5, k
    assert all(int(v) == 1 for k, v in g["running"].items() if k.endswith("num_batches_tracked")
               and (k.startswith("appearance.layers") or k.startswith("w_det")))
    # ground truth + loss: oracle restatement and the product's torch modules, on the reference's own outputs
    cls, ids = synthetic_gt(n, m, seed)
    tm = mmmot_b200.TrackingModule(types.SimpleNamespace(test_mode=2), None, mmmot_b200.TrackingLoss(**LOSS_KW))
    gt_det, gt_link, gt_new, gt_end = tm.generate_gt(g["det"][0], cls, ids, split)
    assert torch.equal(gt_det, g["gt_det"]) and torch.equal(gt_link[0], g["gt_link"])
    assert torch.equal(gt_new, g["gt_new"]) and torch.equal(gt_end, g["gt_end"])
    args = (split, gt_det, gt_link, gt_new, gt_end, g["det"], [g["link"]], g["new"], g["end"], [g["trans1"], g["trans2"]])
    kw = {k: LOSS_KW[k] for k in ("det_ratio", "trans_ratio", "trans_last")}
    assert abs(float(train_ref.tracking_loss(*args, **kw)) - float(g["loss"])) < 1e-6 * abs(float(g["loss"]))
    assert abs(float(tm.criterion(*args)) - float(g["loss"])) < 1e-6 * abs(float(g["loss"]))


def test_dropblock_weights_match_oracle_dropblock():
    """The host-side DropBlock mask generator of the product (TrackingNet._dropblock_weights) draws the same Bernoulli
    seeds and builds the same block weights as the oracle's restatement of modules/dropblock.py (itself pinned by the
    train_drop golden), for odd and even block sizes and 1x1 maps."""
    import mmmot_b200
    from oracle import torch_ref
    for (n, h, w, bs) in ((5, 4, 4, 5), (3, 14, 14, 5), (7, 7, 7, 4), (2, 1, 1, 5)):
        x = torch.rand(n, 6, h, w, generator=torch.Generator().manual_seed(n * 100 + h))
        torch.manual_seed(900 + h)
        ref = torch_ref.drop_block(x, bs)
        torch.manual_seed(900 + h)
        wts = mmmot_b200.TrackingNet._dropblock_weights(n, h, w, bs)
        assert wts.shape == (n, h, w)
        assert torch.allclose(x * wts[:, None], ref, rtol=1e-6, atol=0)
