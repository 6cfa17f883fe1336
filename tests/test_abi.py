"""CPU: the C-ABI library loads and exports every symbol include/mmmot_b200.h declares; the Python
mirror of the enums/weight ids matches the header; host-side logic (schema, weight packing,
config surface, error behaviour without a GPU)."""
import collections
import ctypes
import os
import re
import shutil
import subprocess

import pytest
import torch

import mmmot_b200
from mmmot_b200 import _lib
from mmmot_b200.schema import state_schema
from mmmot_b200.synthetic import synthetic_batch, synthetic_pair, synthetic_state_dict
from mmmot_b200.weights import prepare


def test_library_exports_every_declared_symbol(lib_built):
    names = _lib.header_functions()
    assert set(names) == set(_lib.SIGNATURES), (sorted(set(names) ^ set(_lib.SIGNATURES)))
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert getattr(lib, n) is not None
    lib.mmmot_abi_version.restype = ctypes.c_int
    assert lib.mmmot_abi_version() == _lib.ABI_VERSION == int(re.search(r"MMMOT_ABI_VERSION (\d+)", open(_lib.HEADER_PATH).read()).group(1))


def test_python_enums_match_header():
    src = open(_lib.HEADER_PATH).read()
    ids = dict((k, int(v)) for k, v in re.findall(r"MMMOT_W_([A-Z0-9_]+)\s*=\s*(\d+)", src))
    for k, v in _lib.W.items():
        assert ids[k] == v, k
    for table, prefix in ((_lib.FUSION, "MMMOT_FUSION_"), (_lib.AFFINITY, "MMMOT_AFF_"), (_lib.SOFTMAX, "MMMOT_SM_")):
        for k, v in table.items():
            assert re.search(rf"{prefix}{k.upper()}\s*=\s*{v}\b", src), (prefix, k)


def test_workspace_queries_need_no_gpu(lib_built):
    lib = _lib.load()
    assert lib.mmmot_appearance_workspace(16, 64, 64) > 16 * 64 * 64 * 64 * 4
    assert lib.mmmot_affinity_workspace(1, 128, 128) > 3 * 1024 * 128 * 128 * 4
    # tensor-core path (L >= 16): fp32 trunk activations + FP16 hi/lo planes, but never the 1024-wide layer
    tc_ws = lib.mmmot_pointnet_workspace(1, 16, 4096)
    assert (64 + 128 + 64) * 4096 * 4 < tc_ws < 1024 * 4096 * 4
    lib.mmmot_set_engine(1)                              # FP32 engine materialises it
    try:
        assert lib.mmmot_pointnet_workspace(1, 16, 4096) > 1024 * 4096 * 4
    finally:
        lib.mmmot_set_engine(0)
    assert lib.mmmot_fusion_det_workspace(2, 16) > 0 and lib.mmmot_lp_workspace(4, 8, 8) > 0
    # argument validation happens before any CUDA call
    assert lib.mmmot_lp_assign(None, 0, None, 0, None, 0, None, 0, 1, 1, 1, None, None, None, None, None, None, 0, None) == -1


def test_set_debug_accepts_only_the_profiling_bits(lib_built):
    """mmmot_set_debug takes bits 0-3 (skip epilogue / weight loads / operand loads / MMA issue) and refuses any other
    bit, so a stale flag from a removed experiment fails instead of silently measuring the default path."""
    lib = _lib.load()
    try:
        for flags in range(16):
            assert lib.mmmot_set_debug(flags) == 0, flags
        for flags in (16, 4096, 16384):
            assert lib.mmmot_set_debug(flags) == -1, flags
    finally:
        lib.mmmot_set_debug(0)


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="needs cuobjdump")
def test_every_kernel_is_compiled_once(lib_built):
    """The kernels are compiled in one translation unit (engines.cu), so the library holds one body per kernel."""
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    names = re.findall(r"Function : (\S+)", sass)
    assert names
    dups = sorted(n for n, c in collections.Counter(names).items() if c > 1)
    assert not dups, dups


@pytest.mark.parametrize("fusion,nkeys,numel",[("C", 263, 21218212), ("A", 255, None), ("B", 259, None)])
def test_state_dict_schema(fusion, nkeys, numel):
    """SURVEY §8b: 263 keys / 21 218 212 elements for Fusion C; key names are the drop-in contract."""
    sch = state_schema(fusion)
    assert len(sch) == nkeys
    net = mmmot_b200.TrackingNet(2, appear_skippool=True, score_arch="branch_cls", score_fusion_arch=fusion)
    sd = net.state_dict()
    assert list(sd.keys()) == list(sch.keys())
    for k, (shape, _) in sch.items():
        assert tuple(sd[k].shape) == tuple(shape), k
    if numel:
        assert sum(v.numel() for v in sd.values()) == numel
    res = net.load_state_dict(synthetic_state_dict(fusion, 3), strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert not dict(net.named_parameters())["point_net.feat.stn1.idt"].requires_grad


def test_prepare_folds_bn_and_stn():
    sd = synthetic_state_dict("C", seed=2)
    w, t1, t2, scales = prepare(sd, "C")
    assert sum(t is not None for t in w) == _lib.W["COUNT"]
    # BN fold of the first VGG conv: y = conv(x)*s + shift, checked on a random input
    x = torch.randn(2, 3, 8, 8)
    ref = torch.nn.functional.conv2d(x, sd["appearance.layers.0.0.weight"], sd["appearance.layers.0.0.bias"], padding=1)
    ref = torch.nn.functional.batch_norm(ref, sd["appearance.layers.0.1.running_mean"], sd["appearance.layers.0.1.running_var"],
                                         sd["appearance.layers.0.1.weight"], sd["appearance.layers.0.1.bias"], False, 0.0, 1e-5)
    wt = w[_lib.W["VGG_WT0"]].reshape(3, 3, 3, 64).permute(3, 2, 0, 1)     # [(ky,kx),ci][co] -> [co][ci][ky][kx]
    got = torch.nn.functional.conv2d(x, wt, w[_lib.W["VGG_B0"]], padding=1)
    assert (got - ref).abs().max() < 1e-4
    # STN fold: conv1(T1^T x) == (W1 T1^T) x
    pts = torch.randn(1, 3, 50)
    w1 = sd["point_net.feat.conv1.weight"]
    ref = torch.nn.functional.conv1d(torch.bmm(pts.transpose(2, 1), t1.unsqueeze(0)).transpose(2, 1), w1)
    got = torch.einsum("kc,bkp->bcp", w[_lib.W["PN_L1"]], pts)
    assert (got - ref).abs().max() < 1e-5
    # stacked affinity / new-end first layer
    assert w[_lib.W["AF_W01T"]].shape == (512, 1024)
    assert torch.equal(w[_lib.W["AF_W01T"]][:, 512:].t(), sd["w_link.w_new_end.conv0.0.weight"].reshape(512, 512))


def test_config_surface_of_shipped_experiments():
    """The five shipped configs' model sections (reference experiments/*/config.yaml:2-33)."""
    base = dict(sample_max_len=2, without_reflectivity=True, dropblock=0, use_dropout=False,
                model=dict(point_arch="v1", point_len=512, appear_arch="vgg", appear_len=512, appear_skippool=True,
                           appear_fpn=False, end_arch="v2", end_mode="avg", affinity_op="multiply", softmax_mode="none",
                           score_arch="branch_cls", neg_threshold=0.2, score_fusion_arch="A", test_mode=2))
    for fusion, op, sm, thr in (("A", "multiply", "none", 0.2), ("B", "multiply", "none", 0.2), ("C", "multiply", "none", 0.2),
                                ("C", "minus_abs", "dual_add", 0.2), ("C", "minus_abs", "dual_add", 0)):
        cfg = dict(base, model=dict(base["model"], score_fusion_arch=fusion, affinity_op=op, softmax_mode=sm, neg_threshold=thr))
        net = mmmot_b200.build_model({"common": cfg})
        assert (net.score_fusion_arch, net.affinity_op, net.softmax_mode, net.test_mode) == (fusion, op, sm, 2)
    with pytest.raises(NotImplementedError):
        mmmot_b200.TrackingNet(2, appear_skippool=False, score_arch="branch_cls")   # broken in the reference too (SURVEY §8b)


def test_no_cpu_fallback():
    net = mmmot_b200.TrackingNet(2, appear_skippool=True, score_arch="branch_cls").eval()
    dets, info, split = synthetic_pair(2, 2, 4, 32)
    with pytest.raises(_lib.MmmotError):
        net(dets, info, split)
    with pytest.raises(_lib.MmmotError):
        mmmot_b200.ortools_solve(torch.zeros(4), [torch.zeros(1, 2, 2)], torch.zeros(4), torch.zeros(4), [2, 2])


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.abspath(mmmot_b200.__file__))
    for f in os.listdir(root):
        if f.endswith(".py"):
            assert "oracle" not in open(os.path.join(root, f)).read().replace("the oracle", ""), f


def test_synthetic_batch_layout():
    crops, pts, split = synthetic_batch(3, 4, pts=8, hw=32, seed=0)
    assert crops.shape == (24, 3, 32, 32) and split.shape == (25,) and pts.shape == (int(split[-1]), 3)
    d, info, _ = synthetic_pair(4, 4, 8, 32, seed=1)
    assert torch.equal(crops[8:16], d) and torch.equal(pts[64:128], info["points"][0])
