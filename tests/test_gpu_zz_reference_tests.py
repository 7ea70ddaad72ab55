"""GPU tests (-m gpu) that restate the reference's OWN test files on the host mirror (they run last: the file name sorts after
test_gpu_parity.py).  tests/core/test_packed_rf_tracer.py::test_extra_channels asks the tracer for a channel it does not
composite itself ("density") and checks that the render buffer carries it, one row per ray."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O


def test_extra_channels():
    import wisp_b200 as W
    torch.manual_seed(0)
    blas = W.OctreeAS.make_dense(3, device="cuda")
    grid = W.HashGrid.from_geometric(blas, feature_dim=2, num_lods=1, multiscale_type='cat', feature_std=0.3, codebook_bitwidth=8,
                                     min_grid_res=2, max_grid_res=4)                     # init_from_geometric(2, 4, 1) in the reference test
    # bias=True: with a single LOD the reference's 'cat' quirk (hash_grid.py:226-229) zeroes the only feature level, so the biases carry the field
    nef = W.NeuralRadianceField(grid, view_embedder='positional', view_multires=4, hidden_dim=128, num_layers=1, bias=True).cuda()
    tracer = W.PackedRFTracer()                                                          # reference defaults: 'ray', 1024 steps
    pipeline = W.Pipeline(nef, tracer)
    o, d = O.look_at_rays([-3.0, 0.65, -3.0], [0, 0, 0], 16, 8, 30.0)                     # 128 rays (RandomViewDataset(num_rays=128))
    rays = W.Rays(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), dist_min=0.0, dist_max=6.0)
    rb = pipeline(rays=rays, channels=["rgb", "density"])
    assert hasattr(rb, "density")
    assert rb.rgb.shape[0] == rb.density.shape[0] == 128
    # the extra channel is alpha * (front-to-back integral of the channel), zero for rays without samples (packed_rf_tracer.py:167-179)
    miss = ~rb.hit
    assert torch.isfinite(rb.density).all() and (rb.density >= 0).all()
    if bool(miss.any()):
        assert float(rb.density[miss].abs().max()) == 0.0
    assert float(rb.density[rb.hit].sum()) > 0.0 or not bool(rb.hit.any())
    rb.density.sum().backward()                                                          # differentiable like every other channel
    gb = nef.decoder_density.lout.bias.grad
    assert gb is not None and torch.isfinite(gb).all()


@pytest.mark.gpu
def test_native_adam_matches_torch():
    """wb_adam_step (all tensors in one launch, per-segment lr / weight decay, gradient cleared as consumed) vs torch.optim.Adam."""
    import wisp_b200 as W
    torch.manual_seed(0)
    shapes = [(1000003, 2), (64, 32), (64,), (3, 64), (7,)]
    ps = [torch.randn(s, device="cuda") for s in shapes]
    ref = [p.clone().requires_grad_(True) for p in ps]
    lrs, wds = [2e-3, 1e-3, 1e-3, 1e-3, 5e-4], [0.0, 1e-2, 1e-2, 0.0, 0.0]
    topt = torch.optim.Adam([{"params": [r], "lr": lr, "weight_decay": wd} for r, lr, wd in zip(ref, lrs, wds)], eps=1e-8, betas=(0.9, 0.99))
    nopt = W.NativeAdam([(p, lr, wd) for p, lr, wd in zip(ps, lrs, wds)], betas=(0.9, 0.99), eps=1e-8)
    for it in range(6):
        gs = [torch.randn_like(p) * (10.0 ** (it - 3)) for p in ps]
        for r, g in zip(ref, gs):
            r.grad = g.clone()
        topt.step()
        mine = [(g * 4.0).contiguous() for g in gs]                     # grad_scale undoes the factor (1/world after an all-reduce(sum))
        nopt.step(mine, grad_scale=0.25, zero_grad=True)
        assert all(float(g.abs().max()) == 0.0 for g in mine)
        for p, r in zip(ps, ref):
            assert float((p - r.detach()).abs().max()) <= 1e-6 * max(1.0, float(r.detach().abs().max())), it


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1])
def test_multiview_step_matches_autograd_step(precision):
    """MultiviewStep (march -> shade -> composite -> fused loss + composite backward -> decoder backward -> scatter -> one-launch
    Adam, no autograd) against the autograd route with torch's smooth_l1_loss and the same gradients: loss, every gradient, and the
    parameters after the update.  The premarch hand-over (next_rays) must not change anything."""
    import copy
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import wisp_b200 as W
    from oracle import oracle as O
    from gpu_util import nef_from_oracle, packed_grads
    onef = O.make_nef(num_lods=8, codebook_bitwidth=14, min_res=8, max_res=128, hidden_dim=64, feature_std=0.3, seed=1)
    spc = O.octree_to_spc(O.points_to_octree(O.lego_like_points(5), 5))
    o, d = O.look_at_rays([-3.0, 0.65, -3.0], [0, 0, 0], 48, 48, 30.0)
    o2, d2 = O.look_at_rays([3.0, 0.65, -3.0], [0, 0, 0], 48, 48, 30.0)
    tgt = torch.sigmoid(torch.randn(o.shape[0], 3, generator=torch.Generator().manual_seed(3))).cuda()
    rays = W.Rays(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), 0.0, 10.0)
    rays2 = W.Rays(torch.from_numpy(o2).cuda(), torch.from_numpy(d2).cuda(), 0.0, 10.0)
    # reference: autograd + torch loss
    nef_a, _ = nef_from_oracle(onef, spc)
    tr_a = W.PackedRFTracer('ray', 128, bg_color=(1.0, 1.0, 1.0)); tr_a.precision = precision; tr_a.seed = 21
    rb = W.Pipeline(nef_a, tr_a)(rays=rays, channels=["rgb"])
    loss_a = torch.nn.functional.smooth_l1_loss(rb.rgb, tgt, reduction='none').mean()
    loss_a.backward()
    gt, gd, gc = packed_grads(nef_a)
    # native step
    nef_b, _ = nef_from_oracle(onef, spc)
    tr_b = W.PackedRFTracer('ray', 128, bg_color=(1.0, 1.0, 1.0)); tr_b.precision = precision
    ms = W.MultiviewStep(W.Pipeline(nef_b, tr_b), lr=1e-3, eps=1e-8, rgb_loss_type="huber", rgb_loss_denom="rays")
    before = nef_b.grid.codebook.feats.detach().clone()
    loss_b = ms.step(rays, tgt, seed=21, next_rays=rays2, next_seed=22, zero_grad=False)
    assert tr_b.get_prev_num_samples() == tr_a.get_prev_num_samples() > 0
    tol = 1e-6 if precision == 0 else 1e-5
    assert abs(float(loss_b) - float(loss_a)) <= tol * max(1.0, abs(float(loss_a)))
    gtol = 2e-3 if precision == 0 else 3e-2
    for mine, ref in ((ms.g_grid[0].cpu().numpy(), gt), (ms.g_dens.cpu().numpy(), gd), (ms.g_col.cpu().numpy(), gc)):
        assert np.abs(mine.reshape(-1) - ref.reshape(-1)).max() <= gtol * np.abs(ref).max()
    # the update is Adam's: the same step of torch.optim.Adam on the autograd model lands on the same parameters (entries whose
    # gradient sits at the eps scale may differ by a fraction of lr), untouched table rows stay put
    topt = torch.optim.Adam([p_ for p_ in nef_a.parameters() if p_.requires_grad], lr=1e-3, eps=1e-8)
    topt.step()
    diff = (nef_b.grid.codebook.feats.detach() - nef_a.grid.codebook.feats.detach()).abs()
    assert float(diff.mean()) <= 0.02 * 1e-3 and float(diff.max()) <= 2.0e-3
    for pa, pb in zip(nef_a.decoder_color.parameters(), nef_b.decoder_color.parameters()):
        assert float((pa.detach() - pb.detach()).abs().mean()) <= 0.05 * 1e-3
    moved = (nef_b.grid.codebook.feats.detach() - before).abs()
    assert float(moved[~torch.from_numpy(gt != 0).cuda()].max()) == 0.0 and float(moved.max()) > 0.5e-3
    # second step consumes the pre-marched batch and keeps working (gradients cleared by the optimiser launch)
    loss_c = ms.step(rays2, tgt, seed=22)
    assert len(tr_b._pending) == 0 and torch.isfinite(loss_c) and float(ms.g_grid[0].abs().max()) == 0.0
    # decoder parameters are views of the flat buffers the optimiser updates
    assert nef_b.decoder_density.layers[0].weight.data_ptr() == ms.dens_flat.data_ptr()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [0, 1])
def test_multiview_step_on_triplanar_grid_channel_last(precision):
    """MultiviewStep over a TriplanarGrid(feature_dim=4): the kernels read channel-last copies of the planes and accumulate
    channel-last gradients (wb_nef_desc.grid_layout = 1); what the step leaves in g_grid is in the layout of the reference's
    plane parameters and equals the autograd route's .grad; two accumulating steps double it; the optimiser clears everything."""
    import wisp_b200 as W
    from oracle import oracle as O
    torch.manual_seed(4)
    o, d = O.look_at_rays([-3.0, 0.65, -3.0], [0, 0, 0], 32, 32, 30.0)
    rays = W.Rays(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), 0.0, 10.0)
    tgt = torch.sigmoid(torch.randn(o.shape[0], 3, generator=torch.Generator().manual_seed(3))).cuda()

    def make():
        torch.manual_seed(7)
        grid = W.TriplanarGrid(W.AxisAlignedBBoxAS(device="cuda"), feature_dim=4, log_base_resolution=4, num_lods=3, multiscale_type='sum', feature_std=0.3)
        nef = W.NeuralRadianceField(grid, view_embedder='positional', view_multires=4, hidden_dim=64, num_layers=1, bias=True).cuda()
        tr = W.PackedRFTracer('voxel', 32, bg_color=(1.0, 1.0, 1.0)); tr.precision = precision
        return nef, tr
    nef_a, tr_a = make(); tr_a.seed = 5
    rb = W.Pipeline(nef_a, tr_a)(rays=rays, channels=["rgb"])
    loss_a = torch.nn.functional.smooth_l1_loss(rb.rgb, tgt, reduction='none').mean()
    loss_a.backward()
    ga = [p.grad.detach().clone() for p in W.ops.grid_tensors(nef_a, W.ops.nef_spec(nef_a, None))]
    nef_b, tr_b = make()
    ms = W.MultiviewStep(W.Pipeline(nef_b, tr_b), lr=1e-3, eps=1e-8)
    assert W.ops.triplane_wants_channel_last(ms.spec)
    loss_b = ms.step(rays, tgt, seed=5, zero_grad=False, update=False)
    assert abs(float(loss_b) - float(loss_a)) <= (1e-6 if precision == 0 else 1e-5) * max(1.0, abs(float(loss_a)))
    gtol = 2e-3 if precision == 0 else 0.2          # fp16 'sum' grids: see test_fused_triplanar_octree_nerf
    for mine, ref in zip(ms.g_grid, ga):
        assert mine.shape == ref.shape
        assert float((mine - ref).abs().max()) <= gtol * float(ref.abs().max())
    first = [g.clone() for g in ms.g_grid]
    ms.step(rays, tgt, seed=5, zero_grad=False, update=False)                # accumulates: exactly twice the first gradient at precision 0
    if precision == 0:
        for g2, g1 in zip(ms.g_grid, first):
            assert float((g2 - 2 * g1).abs().max()) <= 1e-4 * float(g1.abs().max())
    ms.zero_grads()
    before = [p.detach().clone() for p in ms.grid]
    ms.step(rays, tgt, seed=5)                                               # a real update: planes move, every accumulator is cleared
    assert all(float((p.detach() - b).abs().max()) > 0 for p, b in zip(ms.grid, before))
    assert all(float(g.abs().max()) == 0.0 for g in ms.g_grid + ms._cl[1])
