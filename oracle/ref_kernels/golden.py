"""Inputs and stored outputs of the original kaolin-wisp CUDA operators (TEST INFRASTRUCTURE).

    python -m oracle.ref_kernels.golden [OUT_DIR]       (needs a CUDA device and oracle/_ref/libwisp_ref_kernels.so)

tests/test_gpu_ref_kernels.py puts this repository's kernels beside the operators they replace:
    hashgrid_interpolate_cuda / _backward_cuda,  uniform_sample_cuda,  find_depth_bound_cuda
The original operators are built into oracle/_ref/ by oracle/ref_kernels/build_ref.py, which needs the original sources.  So that
every checkout can run the comparison, this script runs them once on the cases below and stores what they returned under
tests/golden/ref_*.npz; the tests rebuild the same inputs with the functions here and compare against those files.
Outputs compared with a tolerance are stored as a fixed, seeded sample of rows (each file stays well under 1 MB); outputs compared
bit for bit are stored as a sample plus the SHA-256 of the whole array, so the comparison stays exact."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libwisp_ref_kernels.so")
HASHGRID_FEATURE_DIMS = (2, 4)
SAMPLE = 4096            # entries kept of a bit-exact output besides its digest


def digest(t: torch.Tensor) -> str:
    return hashlib.sha256(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


def golden_path(name: str, out_dir: str = GOLDEN) -> str:
    return os.path.join(out_dir, f"ref_{name}.npz")


def hashgrid_case(W, F: int):
    """HashGrid with dense and hashed levels, 200k points (cell faces of the coarse levels and the +-1 borders included), a seeded
    table and output gradient.  Returns (grid, coords, grad_out, feature rows, table rows): the rows are the stored sample."""
    rng = np.random.default_rng(100 + F)
    blas = W.OctreeAS.make_dense(3, device="cuda")
    grid = W.HashGrid.from_geometric(blas, feature_dim=F, num_lods=12, multiscale_type='cat', feature_std=1.0, codebook_bitwidth=14,
                                     min_grid_res=8, max_grid_res=300).cuda()
    rows_table = grid.codebook.feats.shape[0]
    with torch.no_grad():
        grid.codebook.feats.copy_(torch.from_numpy(rng.standard_normal((rows_table, F), dtype=np.float32)))
    N = 200_000
    coords = rng.random((N, 3), dtype=np.float32) * 2 - 1
    coords[:1000] = np.round(coords[:1000] * 8) / 8                    # exact cell faces of the coarse levels
    coords[1000:1100] = np.sign(coords[1000:1100])                     # corners / borders of the unit cube
    go = rng.standard_normal((N, len(grid.resolutions) * F), dtype=np.float32)
    feat_rows = np.concatenate([np.arange(1100), np.sort(rng.choice(np.arange(1100, N), 1000, replace=False))])
    table_rows = np.sort(rng.choice(rows_table, 8192, replace=False))
    return grid, torch.from_numpy(coords).cuda(), torch.from_numpy(go).cuda(), feat_rows, table_rows


def uniform_case(W):
    """Lego-like level-6 octree, 96x96 rays, 256 uniform steps: the product's sampler and the nuggets that feed the original
    uniform_sample_cuda as octree_as.py:340-357 feeds it (zero-count nuggets filtered, inclusive sum)."""
    from oracle import oracle as O
    blas = W.OctreeAS.from_quantized_points(torch.from_numpy(O.lego_like_points(6)).cuda(), 6)
    o, d = O.look_at_rays([-3.0, 0.65, -3.0], [0, 0, 0], 96, 96, 30.0)
    rays = W.Rays(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), 0.0, 10.0)
    n = 256
    mr = blas.raymarch(rays, 'uniform', n, 6)
    rt = blas.raytrace(rays, 6, with_exit=True)
    scale = W.ops.uniform_scale(n)
    depth = rt.depth.contiguous()
    cnt = (torch.ceil(scale * depth[:, 1]) - torch.ceil(scale * depth[:, 0])).int()          # octree_as.py:343-345
    nz = cnt > 0
    nuggets = (rt.ridx[nz].contiguous(), depth[nz].contiguous(), torch.cumsum(cnt[nz], 0).int().contiguous())
    return mr, scale, nuggets


def depth_bound_case():
    """Cursor query of the SDF tracer: sorted nugget depths per ray, some cursors already retired (-1)."""
    rng = np.random.default_rng(3)
    P = 5000
    counts = rng.integers(1, 6, P); offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    Ng = int(offs[-1])
    en = np.sort(rng.random(Ng) * 5).astype(np.float32); depth = np.stack([en, en + 0.01 + rng.random(Ng).astype(np.float32) * 0.05], -1).astype(np.float32)
    curr = offs[:-1].copy(); curr[::13] = -1
    q = (rng.random(P) * 5).astype(np.float32)
    return torch.from_numpy(q).cuda(), torch.from_numpy(curr).cuda(), torch.from_numpy(depth).cuda()


def sample_index(n: int) -> np.ndarray:
    return np.sort(np.random.default_rng(7).choice(n, min(n, SAMPLE), replace=False))


def _p(t):
    return C.c_void_p(t.data_ptr())


def generate(out_dir: str = GOLDEN) -> None:
    import wisp_b200 as W
    assert torch.cuda.is_available(), "the original operators run on a CUDA device"
    L = C.CDLL(REF_LIB)
    L.ref_last_error.restype = C.c_char_p

    def chk(rc):
        assert rc == 0, L.ref_last_error().decode()
    os.makedirs(out_dir, exist_ok=True)
    for F in HASHGRID_FEATURE_DIMS:
        grid, coords, go, feat_rows, table_rows = hashgrid_case(W, F)
        table = grid.codebook.feats.detach().contiguous()
        nl, bw, N = len(grid.resolutions), grid.codebook_bitwidth, coords.shape[0]
        first = grid.codebook.begin_idxes.to("cuda").contiguous()
        res_host = (C.c_int64 * nl)(*grid.resolutions)
        feats = torch.empty(N, nl * F, device="cuda")
        chk(L.ref_hashgrid_fwd(0, _p(coords), C.c_int64(N), _p(table), C.c_int64(table.shape[0]), F, _p(first), nl, res_host, bw, _p(feats)))
        gt = torch.zeros_like(table)
        chk(L.ref_hashgrid_bwd(0, _p(coords), C.c_int64(N), _p(go), _p(table), C.c_int64(table.shape[0]), F, _p(first), nl, res_host, bw, _p(gt)))
        np.savez_compressed(golden_path(f"hashgrid_f{F}", out_dir), feat_rows=feat_rows, feats=feats[torch.from_numpy(feat_rows).cuda()].cpu().numpy(),
                            feats_absmax=np.float32(feats.abs().max().item()), table_rows=table_rows,
                            grad_table=gt[torch.from_numpy(table_rows).cuda()].cpu().numpy(), grad_absmax=np.float32(gt.abs().max().item()))
    mr, scale, (ridx_f, depth_f, insum) = uniform_case(W)
    V, total = int(ridx_f.shape[0]), int(insum[-1])
    r_ridx = torch.empty(total, dtype=torch.int64, device="cuda"); r_depth = torch.empty(total, device="cuda"); r_b = torch.empty(total, dtype=torch.bool, device="cuda")
    chk(L.ref_uniform_sample(0, scale, _p(ridx_f), _p(depth_f), _p(insum), C.c_int64(V), C.c_int64(total), _p(r_ridx), _p(r_depth), _p(r_b)))
    idx = torch.from_numpy(sample_index(total)).cuda()
    np.savez_compressed(golden_path("uniform_sample", out_dir), total=np.int64(total),
                        ridx=r_ridx[idx].cpu().numpy(), depth=r_depth[idx].cpu().numpy(), boundary=r_b[idx].cpu().numpy(),
                        ridx_sha256=np.array(digest(r_ridx)), depth_sha256=np.array(digest(r_depth)), boundary_sha256=np.array(digest(r_b)))
    q, curr, depth = depth_bound_case()
    out = torch.empty(q.shape[0], dtype=torch.int32, device="cuda")
    chk(L.ref_find_depth_bound(0, _p(q), _p(curr), _p(depth), C.c_int64(q.shape[0]), C.c_int64(depth.shape[0]), _p(out)))
    np.savez_compressed(golden_path("find_depth_bound", out_dir), out=out.cpu().numpy())


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    generate(sys.argv[1] if len(sys.argv) > 1 else GOLDEN)
