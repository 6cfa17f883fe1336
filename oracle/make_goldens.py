"""ORACLE fixture generator — run in the build container only (needs /root/reference).

    python -m oracle.make_goldens

Runs the UNMODIFIED reference ``modules.TrackingNet`` (imported in place, shimmed per SURVEY
F3) on seeded synthetic frame-pairs with seeded synthetic weights and stores inputs' seeds +
the reference outputs under tests/golden/.  Weights/inputs are regenerated from seeds by
``mmmot_b200.synthetic`` at test time (an 85 MB state_dict cannot be committed), so a fixture
is ~10-100 KB.  The reference ships no golden vectors of its own (SURVEY F2) — these are them.
"""
import os

import torch

from mmmot_b200.synthetic import synthetic_pair, synthetic_state_dict
from oracle import ref_loader

# (name, fusion, affinity_op, softmax_mode, neg_threshold, N, M, pts, hw, ragged, seed)
CASES = [
    ("mul_A_n8", "A", "multiply", "none", 0.2, 8, 8, 32, 32, False, 1),
    ("mul_B_n6x9", "B", "multiply", "none", 0.2, 6, 9, 24, 32, True, 2),
    ("mul_C_n8", "C", "multiply", "none", 0.2, 8, 8, 32, 32, False, 3),
    ("subabs_dualadd_C_n8", "C", "minus_abs", "dual_add", 0.2, 8, 8, 32, 32, True, 4),
    ("rrc_subabs_dualadd_C_n5x3", "C", "minus_abs", "dual_add", 0.0, 5, 3, 16, 64, True, 5),
    ("single_C_n4", "C", "minus", "single", 0.2, 4, 4, 16, 32, False, 6),
    ("dual_B_n1x1", "B", "multiply", "dual", 0.2, 1, 1, 16, 32, True, 7),
    ("dualmax_A_n3x7", "A", "minus_abs", "dual_max", 0.2, 3, 7, 20, 32, True, 8),
]

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def reference_forward(case, want_feats=False):
    name, fusion, op, sm, thr, n, m, pts, hw, ragged, seed = case
    net = ref_loader.load_tracking_net(
        seq_len=2, score_arch="branch_cls", appear_arch="vgg", appear_len=512,
        appear_skippool=True, appear_fpn=False, point_arch="v1", point_len=512,
        without_reflectivity=True, softmax_mode=sm, affinity_op=op, end_arch="v2",
        end_mode="avg", test_mode=2, score_fusion_arch=fusion, neg_threshold=thr,
        dropblock=0, use_dropout=False)
    sd = synthetic_state_dict(fusion, seed=seed)
    net.load_state_dict(sd, strict=True)          # also pins the key/shape schema
    dets, info, split = synthetic_pair(n, m, pts, hw, seed=seed, ragged=ragged)
    with torch.no_grad():
        feats, _ = net.feature(dets, info)
        det, link, new, end, trans = net(dets, info, split)
    return {"det": det, "link": link[0], "new": new, "end": end,
            "trans1": trans[0], "trans2": trans[1], "feats": feats}


# BASELINE config[0]: the Fusion-A N=8 plumbing case at 64x64 crops
LIVE_CASE = ("cfg1_mul_A_n8", "A", "multiply", "none", 0.2, 8, 8, 64, 64, False, 21)


def live_golden():
    """The reference's eval-mode outputs of LIVE_CASE (det, link, new, end), stored as float32 arrays so that
    tests/test_oracle.py checks the oracle against them without the reference tree."""
    import numpy as np
    ref = reference_forward(LIVE_CASE)
    np.savez_compressed(os.path.join(OUT, LIVE_CASE[0] + ".npz"),
                        **{k: ref[k].numpy().astype(np.float32) for k in ("det", "link", "new", "end")})
    print(LIVE_CASE[0], {k: tuple(ref[k].shape) for k in ("det", "link", "new", "end")})


def crop_goldens():
    """LiDAR cropping (SURVEY §8f N1) through the UNMODIFIED reference functions (numba):
    box_np_ops.box_camera_to_lidar + preprocess.remove_points_outside_boxes, per box, empty box -> zero point."""
    import numpy as np
    import sys
    sys.path.insert(0, ref_loader.REF)
    from point_cloud import box_np_ops
    from point_cloud.preprocess import remove_points_outside_boxes
    for name, P, n, seed in (("crop_small", 3000, 7, 1), ("crop_mid", 20000, 24, 7)):
        rng = np.random.default_rng(seed)
        centers = rng.uniform([0, -20, -2], [60, 20, 0], size=(n, 3)).astype(np.float32)
        pts = np.concatenate([centers[rng.integers(0, n, P)] + rng.normal(size=(P, 3)) * [2.0, 1.2, 0.9],
                              rng.uniform(size=(P, 1))], 1).astype(np.float32)
        boxes = np.concatenate([centers, rng.uniform([1.2, 2.5, 1.2], [2.2, 5.0, 2.0], size=(n, 3)),
                                rng.uniform(-3.14, 3.14, size=(n, 1))], 1).astype(np.float32)
        boxes[n // 2, :3] += 1000.0                       # one empty box
        out, split = [], [0]
        for i in range(n):
            bp = remove_points_outside_boxes(pts, boxes[i:i + 1])
            if bp.shape[0] == 0:
                bp = np.zeros((1, 4))
            split.append(split[-1] + bp.shape[0])
            out.append(bp)
        out = np.concatenate(out, 0)[:, :3].astype(np.float32)
        # camera -> lidar box conversion with a KITTI-like calibration
        rect = np.eye(4, dtype=np.float32)
        rect[:3, :3] = np.array([[0.9999, 0.0098, -0.0074], [-0.0099, 0.9999, -0.0043], [0.0074, 0.0044, 0.9999]], np.float32)
        v2c = np.eye(4, dtype=np.float32)
        v2c[:3, :] = np.array([[0.0075, -0.9999, -0.0006, -0.0041], [0.0148, 0.0007, -0.9998, -0.0763],
                               [0.9998, 0.0075, 0.0148, -0.2718]], np.float32)
        cam = np.concatenate([rng.uniform([-20, 0, 5], [20, 2, 60], size=(n, 3)), rng.uniform(1, 4, size=(n, 3)),
                              rng.uniform(-3, 3, size=(n, 1))], 1).astype(np.float32)
        lid = box_np_ops.box_camera_to_lidar(cam, rect, v2c)
        # the reference's real pipeline: float64 boxes out of box_camera_to_lidar -> float64 predicate (numba).
        # Boxes: the same ones, moved camera -> LiDAR in float64 like preprocess.py:72-75 does
        boxes64 = boxes.astype(np.float64) + rng.uniform(-1e-7, 1e-7, size=boxes.shape)      # genuinely float64 values
        out64, split64 = [], [0]
        for i in range(n):
            bp = remove_points_outside_boxes(pts, boxes64[i:i + 1])
            if bp.shape[0] == 0:
                bp = np.zeros((1, 4))
            split64.append(split64[-1] + bp.shape[0])
            out64.append(bp)
        out64 = np.concatenate(out64, 0)[:, :3].astype(np.float32)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), points=pts, boxes=boxes, out=out,
                            split=np.asarray(split, np.int64), rect=rect, v2c=v2c, cam=cam, lidar=lid,
                            boxes64=boxes64, out64=out64, split64=np.asarray(split64, np.int64))
        print(name, out.shape, split[-1])


def resize_goldens():
    """Image crop-and-resize (SURVEY §8f N2) with the reference's own calls: PIL crop + BILINEAR resize
    (dataset/test_seq_dataset.py:212-218) and the evaluation transform of utils/build_util.py:137-142.  The frame is
    regenerated from tests.helpers.synthetic_image; stored: float outputs at 32x32 for every box, sha256 of the
    224x224 float outputs, and two full 224x224 uint8 crops."""
    import hashlib
    import numpy as np
    import torchvision.transforms as transforms
    from PIL import Image
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(OUT)))
    from helpers import RESIZE_BOXES, synthetic_image
    img = Image.fromarray(synthetic_image(), "RGB")
    normalize = transforms.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])
    store = {"boxes": np.asarray(RESIZE_BOXES, np.float64)}
    for S in (224, 32):
        tf = transforms.Compose([transforms.Resize(S), transforms.CenterCrop(S), transforms.ToTensor(), normalize])
        outs, u8 = [], []
        for b in RESIZE_BOXES:
            x1, y1, x2, y2 = np.floor(b[0]), np.floor(b[1]), np.ceil(b[2]), np.ceil(b[3])
            crop = img.crop((x1, y1, x2, y2)).resize((S, S), Image.BILINEAR)
            u8.append(np.asarray(crop))
            outs.append(tf(crop).unsqueeze(0))
        outs = torch.cat(outs, 0).numpy()
        if S == 32:
            store["out32"] = outs
        else:
            store["sha224"] = np.asarray([hashlib.sha256(o.tobytes()).hexdigest() for o in outs])
            store["u8_224_first"] = u8[0]
            store["u8_224_full"] = u8[9]
    np.savez_compressed(os.path.join(OUT, "resize_kitti.npz"), **store)
    print("resize_kitti", store["out32"].shape)


def stitch_goldens():
    """Track-id assignment + stitching + KITTI text (SURVEY §8f N3) through the UNMODIFIED reference
    tracking_model.TrackingModule.assign_det_id / align_id and utils.data_util.write_kitti_result.  Absent
    third-party imports of those modules (ortools behind `solvers`, pyproj) are stubbed: neither is used here."""
    import copy
    import json
    import sys
    import tempfile
    import types
    sys.path.insert(0, ref_loader.REF)
    sys.path.insert(0, os.path.join(os.path.dirname(OUT)))
    sys.modules.setdefault("pyproj", types.ModuleType("pyproj"))
    if "solvers" not in sys.modules:
        sys.modules["solvers"] = types.SimpleNamespace(ortools_solve=None)
    from helpers import stitch_scenario
    import tracking_model as ref_tm
    from utils.data_util import write_kitti_result
    gold = {}
    for seed in (0, 1, 2):
        dets, samples = stitch_scenario(seed)
        tm = ref_tm.TrackingModule(types.SimpleNamespace(test_mode=0), None, None, det_type="3D")
        steps = []
        for (a, b), split, a_det, a_link, a_new, a_end in samples:
            pair = [copy.deepcopy(dets[a]), copy.deepcopy(dets[b])]
            ids, boxes = tm.assign_det_id(a_det, a_link, a_new, a_end, split, pair)
            local = [[int(v) for v in x] for x in ids]
            aligned, adets, start = tm.align_id(ids, boxes)
            steps.append({"local": local, "aligned": [[int(v) for v in x] for x in aligned], "frame_start": int(start),
                          "frames": [int(d["frame_idx"][0]) for d in adets], "last_id": int(tm.last_id)})
        with tempfile.TemporaryDirectory() as tmp:
            write_kitti_result(tmp, "0000", "step", tm.frames_id, copy.deepcopy(tm.frames_det), part="val")
            text = open(os.path.join(tmp, "step", "val", "0000.txt")).read()
        gold[str(seed)] = {"steps": steps, "frames_id": [[int(v) for v in x] for x in tm.frames_id], "kitti": text}
    with open(os.path.join(OUT, "stitch.json"), "w") as f:
        json.dump(gold, f)
    print("stitch", {k: len(v["steps"]) for k, v in gold.items()})


# training-mode cases (SURVEY §8f N4): (name, fusion, affinity_op, softmax_mode, N, M, pts, hw, ragged, seed)
TRAIN_CASES = [
    ("train_mul_A_n6x5", "A", "multiply", "none", 6, 5, 24, 32, True, 21),
    ("train_subabs_dualadd_C_n7", "C", "minus_abs", "dual_add", 7, 7, 32, 32, False, 22),
    # experiments/rrc_pfv_40e_subabs_dualadd_C/config.yaml:32-33: dropblock 5, use_dropout True (64-px crops: 4x4 and 2x2
    # head maps, so blocks really differ per pixel); torch.manual_seed(seed) right before the forward
    ("train_drop_subabs_dualadd_C_n9x6", "C", "minus_abs", "dual_add", 9, 6, 40, 64, True, 23),
]
TRAIN_DROP = {"train_drop_subabs_dualadd_C_n9x6": dict(dropblock=5, use_dropout=True)}


# experiments/pp_pv_40e_dualadd_subabs_C/config.yaml:39-45 through utils/build_util.py:147-155
LOSS_KW = dict(smooth_ratio=0, detloss_type="bce", det_ratio=1.5, trans_ratio=0.001, trans_last=True, linkloss_type="l2")


def synthetic_gt(n, m, seed):
    """Seeded class flags / track ids in the DataLoader layout generate_gt reads (per frame: 1 x n_i)."""
    g = torch.Generator().manual_seed(4000 + seed)
    cls = [(torch.rand(1, k, generator=g) < 0.75).long() for k in (n, m)]
    ids0 = torch.randperm(n + 3, generator=g)[:n]
    ids1 = torch.randperm(n + 3, generator=g)[:m]          # overlaps ids0 partly: links, births and deaths
    return cls, [ids0.unsqueeze(0), ids1.unsqueeze(0)]


def train_goldens():
    """The UNMODIFIED reference in .train() mode (BatchNorm batch statistics, raw det logits, unpadded new/end) and its
    TrackingLoss / generate_gt.  Shims: F._verify_batch_size (SURVEY F3); `Tensor.eq` returning uint8 while the loss
    runs, because cost.py:122 computes `1 - gt_score.eq(...)`, which reference-era torch allowed on a byte mask and
    modern torch rejects on bool; `solvers` stubbed (ortools absent; not used here)."""
    import sys
    import types
    sys.path.insert(0, ref_loader.REF)
    sys.modules.setdefault("pyproj", types.ModuleType("pyproj"))
    if "solvers" not in sys.modules:
        sys.modules["solvers"] = types.SimpleNamespace(ortools_solve=None)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        import tracking_model as ref_tm
        from cost import TrackingLoss
    for case in TRAIN_CASES:
        name, fusion, op, sm, n, m, pts, hw, ragged, seed = case
        net = ref_loader.load_tracking_net(
            seq_len=2, score_arch="branch_cls", appear_arch="vgg", appear_len=512, appear_skippool=True, appear_fpn=False,
            point_arch="v1", point_len=512, without_reflectivity=True, softmax_mode=sm, affinity_op=op, end_arch="v2",
            end_mode="avg", test_mode=2, score_fusion_arch=fusion, neg_threshold=0.2,
            **TRAIN_DROP.get(name, dict(dropblock=0, use_dropout=False)))
        sd = synthetic_state_dict(fusion, seed=seed)
        net.load_state_dict(sd, strict=True)
        net.train()
        dets, info, split = synthetic_pair(n, m, pts, hw, seed=seed, ragged=ragged)
        torch.manual_seed(seed)              # the DropBlock / Dropout draws (CPU generator) start from here
        with torch.no_grad():
            det, link, new, end, trans = net(dets, info, split)
        after = {k: v.clone() for k, v in net.state_dict().items() if "running_" in k or "num_batches" in k}
        cls, ids = synthetic_gt(n, m, seed)
        with contextlib.redirect_stdout(io.StringIO()):
            tm = ref_tm.TrackingModule(net, None, TrackingLoss(**LOSS_KW))
        gt_det, gt_link, gt_new, gt_end = tm.generate_gt(det[0], cls, ids, split)
        orig_eq = torch.Tensor.eq
        torch.Tensor.eq = lambda a, b: orig_eq(a, b).to(torch.uint8)
        try:
            with torch.no_grad():
                loss = tm.criterion(split, gt_det, gt_link, gt_new, gt_end, det, link, new, end, trans)
        finally:
            torch.Tensor.eq = orig_eq
        out = {"case": case, "det": det, "link": link[0], "new": new, "end": end, "trans1": trans[0], "trans2": trans[1],
               "running": after, "gt_det": gt_det, "gt_link": gt_link[0], "gt_new": gt_new, "gt_end": gt_end,
               "loss": loss.detach().clone(), "drop": TRAIN_DROP.get(name, dict(dropblock=0, use_dropout=False))}
        torch.save(out, os.path.join(OUT, name + ".pt"))
        print(name, float(loss), tuple(det.shape), tuple(new.shape), tuple(end.shape))


def main():
    os.makedirs(OUT, exist_ok=True)
    train_goldens()
    crop_goldens()
    resize_goldens()
    stitch_goldens()
    live_golden()
    torch.set_num_threads(os.cpu_count())
    for case in CASES:
        out = reference_forward(case)
        out = {k: v.clone().contiguous() for k, v in out.items()}
        out["case"] = case
        torch.save(out, os.path.join(OUT, case[0] + ".pt"))
        print(case[0], {k: tuple(v.shape) for k, v in out.items() if hasattr(v, "shape")})


if __name__ == "__main__":
    main()
