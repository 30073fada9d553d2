"""CPU-only checks: the C-ABI library loads and exports every symbol include/hnr.h declares; host
logic that needs no GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "hnr.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hnr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from hybridneuralrendering_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    L = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/hnr.h but not exported"
    assert set(_lib.EXPORTED) == set(names), set(_lib.EXPORTED) ^ set(names)
    L.hnr_abi_version.restype = ctypes.c_int
    assert L.hnr_abi_version() == 1
    _lib.lib()    # argtypes bind without error


def test_product_path_refuses_cpu_tensors():
    from hybridneuralrendering_b200 import ops
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.linear([torch.zeros(4, 3)], torch.zeros(2, 3), torch.zeros(2), 1)
    from hybridneuralrendering_b200 import lighting_fast_querier, make_opt
    with pytest.raises(RuntimeError, match="CUDA"):
        lighting_fast_querier(torch.device("cpu"), make_opt())


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "hybridneuralrendering_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in re.sub(r'""".*?"""', "", src, flags=re.S).replace("# ", ""), fn


def test_blur_wrappers_reject_bad_shapes_before_launch():
    """the blur kernels index the raster from patch_num / patch_size alone: every wrapper checks its shapes on the host (CPU
    tensors here, so a check that came after the CUDA guard would raise RuntimeError instead)"""
    from hybridneuralrendering_b200 import ops
    PN, PS, KS = 2, 3, 5
    n = (PN * PS) ** 2
    ok, ker, raw = torch.zeros(n, 3), torch.zeros(4, KS, KS), torch.zeros(PN * PN, KS * KS + 1)
    bad_rasters = [torch.zeros(n - 1, 3), torch.zeros(n + PS, 3), torch.zeros(n, 4), torch.zeros(n, 1), torch.zeros(n * 3),
                   torch.zeros(1, n, 3)]
    for bad in bad_rasters:
        with pytest.raises(ValueError, match="pred"):
            ops.BlurSelectFn.apply(bad, ok, ker, PN, PS)
        with pytest.raises(ValueError, match="gt"):
            ops.BlurSelectFn.apply(ok, bad, ker, PN, PS)
        with pytest.raises(ValueError, match="pred"):
            ops.BlurGrayFn.apply(bad, ok, PN, PS)
        with pytest.raises(ValueError, match="gt"):
            ops.BlurGrayFn.apply(ok, bad, PN, PS)
        with pytest.raises(ValueError, match="pred"):
            ops.BlurLearnFn.apply(bad, raw, PN, PS, KS, 0, 4, 1)
    with pytest.raises(ValueError, match="pred"):                # the raster of a 1-patch-larger grid
        ops.BlurSelectFn.apply(torch.zeros(((PN + 1) * PS) ** 2, 3), torch.zeros(((PN + 1) * PS) ** 2, 3), ker, PN, PS)
    for bad in (torch.zeros(4, KS, KS - 1), torch.zeros(4, KS - 1, KS - 1), torch.zeros(KS, KS), torch.zeros(1, 4, KS, KS)):
        with pytest.raises(ValueError, match="kernels"):
            ops.BlurSelectFn.apply(ok, ok, bad, PN, PS)
    for bad in (torch.zeros(PN * PN - 1, KS * KS + 1), torch.zeros(PN * PN + 1, KS * KS + 1), torch.zeros(PN * PN * (KS * KS + 1))):
        with pytest.raises(ValueError, match="raw"):
            ops.BlurLearnFn.apply(ok, bad, PN, PS, KS, 0, 4, 1)
    # well-formed CPU tensors pass the shape checks and stop at the CUDA guard
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.BlurSelectFn.apply(ok, ok, ker, PN, PS)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.BlurGrayFn.apply(ok, ok, PN, PS)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.BlurLearnFn.apply(ok, raw, PN, PS, KS, 0, 4, 1)


def test_aggregator_state_dict_matches_reference_layout():
    from hybridneuralrendering_b200 import PointAggregator, make_opt
    from oracle import render_oracle as ro
    agg = PointAggregator(make_opt())
    sd = agg.state_dict()
    assert sum(v.numel() for v in sd.values()) == 449381          # SURVEY.md §8c: parameter count of the reference class
    for name, shp in {**ro.LAYER_SHAPES, **ro.CONV_SHAPES}.items():
        assert tuple(sd[name + ".weight"].shape) == shp and tuple(sd[name + ".bias"].shape) == (shp[0],)
    with pytest.raises(NotImplementedError):
        PointAggregator(make_opt(agg_distance_kernel="quadric"))


def test_drop_patch_positions_and_kernel_bank():
    from hybridneuralrendering_b200.blur import predefined_blur_kernels
    from hybridneuralrendering_b200.point_aggregators import drop_patch_rays
    pos = drop_patch_rays(8, 7, 0.5)
    assert len(pos) == 24 * 64 and pos.max() == 1759               # SURVEY.md Appendix B.16
    K = predefined_blur_kernels(3)
    assert K.shape == (36, 9, 9) and np.allclose(K.sum(axis=(1, 2)), 1, atol=1e-6) and (K >= 0).all()
    nz = (K > 0).sum(axis=(1, 2))
    assert nz.min() >= 2 and nz.max() <= 25


def test_synthetic_scenes_respect_cell_capacity():
    from hybridneuralrendering_b200 import make_opt
    from hybridneuralrendering_b200 import synthetic as syn
    from oracle import query_oracle as qo
    for kind, gen in (("lego", syn.lego_scene), ("scannet", syn.room_scene)):
        opt = make_opt(kind)
        xyz = gen(20000, 0)
        gp = qo.grid_params(xyz, opt.vsize, opt.vscale, opt.kernel_size, opt.ranges, opt.radius_limit_scale)
        g = qo.build_grid(xyz, gp, opt.P, opt.query_size, opt.max_o)
        assert g.max_cell_count <= opt.P
        assert xyz.shape == (20000, 3) and xyz.dtype == np.float32


def test_query_oracle_layered_rule_small():
    """hand-checkable case: early exit after layer 0 when the own voxel already holds >= K in-radius points"""
    from oracle import query_oracle as qo
    rng = np.random.default_rng(0)
    base = np.array([0.5, 0.5, 0.5], np.float32)
    own = base + rng.uniform(0.001, 0.007, (5, 3)).astype(np.float32) * 0 + rng.uniform(-0.003, 0.003, (5, 3)).astype(np.float32)
    far = base + np.array([[0.012, 0, 0], [0, 0.012, 0]], np.float32)
    pad = np.array([[0, 0, 0], [1, 1, 1]], np.float32)
    xyz = np.concatenate([pad[:1], own, far, pad[1:]]).astype(np.float32)
    gp = qo.grid_params(xyz, [0.004] * 3, [2, 2, 2], [3, 3, 3], None, 4.0)
    g = qo.build_grid(xyz, gp, 12, [3, 3, 3])
    own_cells = set(qo.lin_index(qo.cell_of(own, gp), gp).tolist())
    if len(own_cells) == 1:
        slots, canon, visited = qo.layered_knn(xyz, g, base, 4, [3, 3, 3])
        assert set(canon.tolist()) <= set(range(1, 6)) and (canon >= 0).sum() == 4      # never looks at the far shell
        slots8, canon8, _ = qo.layered_knn(xyz, g, base, 8, [3, 3, 3])
        assert set(range(1, 8)) == set(canon8[canon8 >= 0].tolist())                    # K=8 > 5: walks layer 1 too


def test_frame_producer_host_logic_matches_reference_golden():
    """N4 host side of the PRODUCT (no GPU needed): nearest-view choice and the patch draws reproduce the unmodified reference's
    choices for the seeded golden cases; both RNG streams are consumed in the reference's order."""
    import random
    from frame_cases import FRAME_CASES, FRAME_CASES_CPU
    from hybridneuralrendering_b200 import frame_producer as fp
    from hybridneuralrendering_b200 import synthetic as syn
    G = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frame.npz")))
    images, c2w, vids, K, train_ids, test_ids = syn.frame_scene()
    H, W = images.shape[1:3]
    for name, split, idx, over, seed, bg in FRAME_CASES + FRAME_CASES_CPU:
        random.seed(seed)
        np.random.seed(seed)
        vid = (train_ids if split == "train" else test_ids)[idx]
        V = over["use_nearest"]
        if over.get("dynamic_nearest"):
            V = int(np.random.randint(2, 8)) if split == "train" else 4
        vn = fp.select_nearest_views(train_ids, vid, V, over["find_nearest_mode"], split)
        assert vn.tolist() == G[f"{name}_vid_nearest"].tolist(), name
        pix = G[f"{name}_pixel_idx"]
        m = over["edge_filter"]
        if over["random_sample"] == "dilated":
            st = over["dilation_setup"].split("_")
            PN, PS = int(st[0]), int(st[1])
            p = fp.draw_dilated_patches(W, H, m, PN, PS, np.arange(float(st[2]), float(st[3]) + 1))
            for i in range(PN):
                for j in range(PN):
                    blk = pix[i * PS:(i + 1) * PS, j * PS:(j + 1) * PS]
                    x0, y0, d = p[i * PN + j]
                    assert (blk[0, 0] == (x0, y0)).all() and (blk[1, 1] == (x0 + d, y0 + d)).all(), (name, i, j)


def test_frame_producer_item_host_path_with_stubbed_device_ops(monkeypatch):
    """runs FrameProducer.item on the CPU with the two device entry points replaced by recorders (the real kernels are covered by
    tests/test_gpu_frame_producer.py): key set, shapes, the patch table handed to the kernel and the RNG state after the item."""
    import random
    from frame_cases import FRAME_CASES, FRAME_CASES_CPU
    from hybridneuralrendering_b200 import frame_producer as fp
    from hybridneuralrendering_b200 import synthetic as syn
    G = dict(np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frame.npz")))
    images, c2w, vids, K, train_ids, test_ids = syn.frame_scene()
    H, W = images.shape[1:3]
    seen = {}

    def fake_rays(patches, PN, PS, width, height, margin, intrinsic, c2w_, dir_norm, frame_u8):
        seen.update(patches=None if patches is None else patches.numpy().copy(), PN=PN, PS=PS, margin=margin, dir_norm=dir_norm)
        rows, cols = (height - 2 * margin, width - 2 * margin) if patches is None else (PN * PS, PN * PS)
        return torch.zeros(rows, cols, 2), torch.zeros(rows * cols, 3), torch.zeros(rows * cols, 3)

    monkeypatch.setattr(fp, "frame_rays", fake_rays)
    monkeypatch.setattr(fp, "frame_views", lambda bank, ids: bank[ids.long()].float() / 255.0)
    for name, split, idx, over, seed, bg in FRAME_CASES + FRAME_CASES_CPU:
        bank = fp.FrameBank(images, c2w, vids, K, "cpu")
        prod = fp.FrameProducer(bank, train_ids if split == "train" else test_ids, train_ids, fp.default_opt(**over), split=split,
                                bg_color=bg, blur_kernels=np.zeros((1, 9, 9), np.float32), total_num_image=vids[-1] + 1)
        random.seed(seed)
        np.random.seed(seed)
        it = prod.item(idx)
        np.testing.assert_array_equal(np.array([random.random(), np.random.rand()]), G[f"{name}_after"], err_msg=name)
        assert it["vid_nearest"].tolist() == G[f"{name}_vid_nearest"].tolist()
        V = len(it["vid_nearest"])
        assert it["images_nearest"].shape == (1, V, H, W, 3) and it["c2w_nearest"].shape == (1, V, 4, 4)
        assert np.float32(it["images_nearest"].abs().max()) == G[f"{name}_images_nearest_absmax"]
        assert it["campos_nearest"].shape == (1, V, 3) and it["campos"].shape == (1, 3) and it["camrotc2w"].shape == (1, 3, 3)
        np.testing.assert_array_equal(it["c2w_nearest"][0].numpy(), G[f"{name}_c2w_nearest"])
        np.testing.assert_array_equal(it["bg_color"][0].numpy(), G[f"{name}_bg_color"])
        pix = G[f"{name}_pixel_idx"]
        assert seen["margin"] == over["edge_filter"] and seen["dir_norm"] == (over["dir_norm"] > 0)
        if seen["patches"] is None:
            assert it["pixel_idx"].shape[1:3] == pix.shape[:2]
        else:
            PN, PS = seen["PN"], seen["PS"]
            assert PN * PS == pix.shape[0]
            for p, (x0, y0, d) in enumerate(seen["patches"]):
                blk = pix[(p // PN) * PS:(p // PN + 1) * PS, (p % PN) * PS:(p % PN + 1) * PS]
                xs, ys = np.meshgrid(x0 + d * np.arange(PS), y0 + d * np.arange(PS))
                np.testing.assert_array_equal(blk[..., 0], xs)
                np.testing.assert_array_equal(blk[..., 1], ys)


def test_step_roofline_formula():
    """SURVEY 8(d): roofline time = sum over stages of max(bytes / HBM peak, FLOPs / tensor peak).  Hand-checked numbers for the
    configs[1] frame of round 1 (28.2 M neighbour rows, 3.95 M valid samples, 163,570 kept rays)."""
    from hybridneuralrendering_b200 import profiling
    pk = {"hbm_gbs": 6553.3, "bf16_tflops_sustained": 1370.7}
    u = {"valid_neighbours": 28233702, "valid_samples": 3945903, "kept_rays": 163570}
    r = profiling.step_roofline(u, 4, 640000, 400, 80, 800, 800, 72.9, pk)
    nbr = 542720 * 28233702 / (1370.7e12 / 3) * 1e3
    smp = (154184 + 4 * 39040) * 3945903 / (1370.7e12 / 3) * 1e3
    assert abs(r["stages"]["per-neighbour MLP"]["roofline_ms"] - nbr) < 1e-3 and abs(nbr - 33.537) < 0.01
    assert abs(r["stages"]["per-sample MLPs"]["roofline_ms"] - smp) < 1e-3
    gather = (168 * 28233702 + 40 * 3945903) / 6553.3e9 * 1e3
    assert abs(r["stages"]["gather + weights"]["roofline_ms"] - gather) < 1e-3
    assert abs(r["roofline_ms"] - sum(s["roofline_ms"] for s in r["stages"].values())) < 1e-2
    assert abs(r["frac"] - r["roofline_ms"] / 72.9) < 1e-9 and 0.5 < r["frac"] < 0.53
    t = profiling.step_roofline({"valid_neighbours": 562096, "valid_samples": 75272, "kept_rays": 4096}, 8, 4096, 400, 24, 480, 640, 25.9, pk,
                                train=True, points=2_000_000)
    # round 2: the fused backward runs on the kind::f16 pipe (3 bf16 MMAs per product) like the forward -> same tensor peak;
    # `frac_tf32_basis` keeps round 1's backward denominator (3 TF32 MMAs per product, TF32 = bf16 / 2 when not measured)
    fwd, bwd = 542720 * 562096 / (1370.7e12 / 3), 2 * 542720 * 562096 / (1370.7e12 / 3)
    assert abs(t["stages"]["per-neighbour MLP"]["roofline_ms"] - (fwd + bwd) * 1e3) < 1e-3
    assert "dense point-gradient tables (zero fill)" in t["stages"] and 0.08 < t["frac"] < 0.10
    assert 0.14 < t["frac_tf32_basis"] < 0.16 and abs(t["tensor_peak_bwd_tf32_basis_tflops"] - 1370.7 / 6) < 1e-6
