"""GPU tests (-m gpu) against what the ORIGINAL kaolin-wisp CUDA operators returned on the same inputs:
    hashgrid_interpolate_cuda / _backward_cuda  (A14)      uniform_sample_cuda  (A8)      find_depth_bound_cuda  (B1)
The outputs are stored under tests/golden/ref_*.npz by oracle/ref_kernels/golden.py (run on a B200 against the operators built from the
original sources); the inputs are rebuilt here by the same functions.  This pins those three operators to the code they replace, not
to a restatement of it."""
import os

import numpy as np
import pytest
import torch

from oracle.ref_kernels import golden as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def W():
    import wisp_b200
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return wisp_b200


def _golden(name):
    path = G.golden_path(name)
    assert os.path.exists(path), f"{path} missing (python -m oracle.ref_kernels.golden regenerates it)"
    return dict(np.load(path))


@pytest.mark.parametrize("F", G.HASHGRID_FEATURE_DIMS)
def test_hashgrid_kernels_vs_reference_cuda(W, F):
    """wb_hashgrid_fwd / _bwd (one launch, all LODs) vs wisp._C.ops.hashgrid_interpolate_cuda / _backward_cuda (one launch per LOD):
    dense and hashed levels, points on cell faces and at the +-1 borders.  Forward: same arithmetic -> 2 ulp-level agreement;
    backward: same products, different atomic order."""
    g = _golden(f"hashgrid_f{F}")
    grid, coords, go, feat_rows, table_rows = G.hashgrid_case(W, F)
    assert np.array_equal(feat_rows, g["feat_rows"]) and np.array_equal(table_rows, g["table_rows"])
    mine = W.ops.hashgrid(coords, grid.codebook_bitwidth, len(grid.resolutions) - 1, grid.codebook)
    assert abs(float(mine.abs().max()) - float(g["feats_absmax"])) <= 2e-6 * float(g["feats_absmax"])
    err = float(np.abs(mine[torch.from_numpy(feat_rows).cuda()].detach().cpu().numpy() - g["feats"]).max())
    assert err <= 2e-6 * float(g["feats_absmax"]), err
    grid.codebook.feats.grad = None
    mine.backward(go)
    gt = grid.codebook.feats.grad
    assert abs(float(gt.abs().max()) - float(g["grad_absmax"])) <= 2e-5 * float(g["grad_absmax"])
    gerr = float(np.abs(gt[torch.from_numpy(table_rows).cuda()].cpu().numpy() - g["grad_table"]).max())
    assert gerr <= 2e-5 * float(g["grad_absmax"]), gerr


def test_uniform_sampler_vs_reference_cuda(W):
    """OctreeAS._raymarch_uniform: wb_raymarch_uniform_{count,fill} vs the reference's uniform_sample_cuda kernel fed as
    octree_as.py:340-357 feeds it: ridx, depth samples and boundary bit-exact (a stored sample, then the digest of every entry)."""
    g = _golden("uniform_sample")
    mr, _, (_, _, insum) = G.uniform_case(W)
    total = int(g["total"])
    assert int(insum[-1]) == total == mr.ridx.shape[0] > 1000
    idx = torch.from_numpy(G.sample_index(total)).cuda()
    depth = mr.depth_samples[:, 0]
    assert np.array_equal(mr.ridx[idx].cpu().numpy(), g["ridx"])
    assert np.array_equal(depth[idx].cpu().numpy(), g["depth"])
    assert np.array_equal(mr.boundary[idx].cpu().numpy(), g["boundary"])
    assert mr.ridx.dtype == torch.int64 and mr.boundary.dtype == torch.bool
    assert G.digest(mr.ridx) == str(g["ridx_sha256"])
    assert G.digest(depth) == str(g["depth_sha256"])
    assert G.digest(mr.boundary) == str(g["boundary_sha256"])


def test_find_depth_bound_vs_reference_cuda(W):
    """wb_find_depth_bound vs find_depth_bound_cuda (cursor kernel of the SDF tracer), quirks included."""
    q, curr, depth = G.depth_bound_case()
    mine = W.ops.find_depth_bound(q[:, None], depth, curr_idxes=curr)
    assert np.array_equal(mine.cpu().numpy(), _golden("find_depth_bound")["out"])
