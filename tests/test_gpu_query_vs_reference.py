"""Bit-exact parity of the product query (and of the numpy oracle) against the REFERENCE's own CUDA
kernels, compiled from the reference source into oracle/_ref/ (oracle/build_ref_query_cubin.py) and
launched here through cuda.bindings.  This is what pins the query oracle (north_star: "the
reference pycuda kernel on the same box")."""
import os

import numpy as np
import pytest
import torch

from helpers import cuda
from hybridneuralrendering_b200 import make_opt
from hybridneuralrendering_b200 import synthetic as syn
from oracle import build_ref_query_cubin as rb
from oracle import query_oracle as qo
from oracle import ref_query_runner as rq

pytestmark = pytest.mark.gpu


def _canon(p):
    p = np.asarray(p).copy()
    big = np.iinfo(np.int32).max
    p[p < 0] = big
    p.sort(axis=-1)
    p[p == big] = -1
    return p


@pytest.mark.parametrize("kind,N,seed", [("lego", 60000, 0), ("room", 80000, 1)])
def test_product_and_oracle_match_reference_kernels(kind, N, seed):
    if not rq.available():
        # the kernels are compiled from the original project's source, which the repository does not contain: without that source
        # there is nothing to compare with; with it, a missing cubin means its build failed
        if not os.path.isfile(rb.SRC):
            pytest.skip(f"original project's query source {rb.SRC} not found: set HNR_REFERENCE_ROOT to a checkout of it and run "
                        "__graft_entry__.build()")
        pytest.fail(f"{rq.CUBIN} missing although {rb.SRC} exists: run __graft_entry__.build() (it reports why the build failed)")
    from hybridneuralrendering_b200 import lighting_fast_querier
    if kind == "lego":
        xyz, fr, opt = syn.lego_scene(N, seed), syn.lego_frame(H=40, W=40, V=1, seed=seed), make_opt("lego")
    else:
        xyz, fr, opt = syn.room_scene(N, seed), syn.room_frame(H=48, W=64, V=1, patch_num=4, patch_size=4, seed=seed), make_opt("scannet")
    near, far = float(fr["near"].min()), float(fr["far"].max())
    q = lighting_fast_querier(torch.device("cuda"), opt)
    R = fr["raydir"].shape[1]
    ts = q.candidate_ts(R, near, far, "cuda")
    gp = qo.grid_params(xyz, opt.vsize, opt.vscale, opt.kernel_size, opt.ranges, opt.radius_limit_scale)
    # candidate positions exactly as the reference forms them: campos + raydir * t (two torch ops)
    raypos = (cuda(fr["campos"])[:, None, None, :] + cuda(fr["raydir"])[:, :, None, :] * ts.view(1, 1, -1, 1)).contiguous()
    ref = rq.reference_query(cuda(xyz)[None].contiguous(), raypos, gp, SR=opt.SR, K=opt.K, P=opt.P, max_o=opt.max_o,
                             kernel_size=opt.kernel_size, query_size=opt.query_size)
    assert ref["max_cell_count"] <= opt.P and ref["n_occupied"] <= opt.max_o          # off the reference's random paths
    # the voxel that won occupied-slot 0 in THIS run of the reference (atomic order) stores no points
    q.skip_cell_override = ref["slot0_cell"]
    out = q.query_points(None, None, cuda(xyz)[None], None, fr["h"], fr["w"], fr["intrinsic"], near, far, cuda(fr["raydir"]),
                         cuda(fr["campos"]), cuda(fr["camrotc2w"]), ts=ts)
    pidx, loc, loc_w, dirs, ray_mask, _, _ = out
    assert q._grid.info[0] == ref["n_occupied"]
    np.testing.assert_array_equal(ray_mask.cpu().numpy(), ref["ray_mask"].cpu().numpy())                    # ray mask: bit-exact
    np.testing.assert_array_equal(loc_w.cpu().numpy(), ref["sample_loc_w"].cpu().numpy())                  # sample positions: same floats
    a, b = _canon(pidx.cpu().numpy()), _canon(ref["sample_pidx"].cpu().numpy())
    assert a.shape == b.shape and a.shape[1] > 50
    np.testing.assert_array_equal(a, b)                                                                    # neighbour sets: bit-exact
    # and the numpy oracle agrees with the reference kernels too (pins oracle/query_oracle.py)
    o = qo.query(xyz, fr["campos"], fr["camrotc2w"], fr["raydir"], ts.cpu().numpy().reshape(-1), vsize=opt.vsize, vscale=opt.vscale,
                 kernel_size=opt.kernel_size, query_size=opt.query_size, ranges=opt.ranges, radius_limit_scale=opt.radius_limit_scale,
                 SR=opt.SR, K=opt.K, P=opt.P, max_o=opt.max_o, skip_cell=ref["slot0_cell"])
    np.testing.assert_array_equal(o["ray_mask"], ref["ray_mask"].cpu().numpy())
    np.testing.assert_array_equal(_canon(o["sample_pidx"]), b)
    # with ascending stored order the oracle's emulation of the reference's slot order is exact whenever the
    # reference's voxel lists happen to be ascending too; as sets they always agree
    np.testing.assert_array_equal(_canon(o["sample_pidx_visit_order"]), b)
