"""GPU test (-m gpu) of the sample-count dependent schedule of the tensor-core decoder backward (csrc/wb_shade_tc.cu,
wb_tc_shade_bwd): with hidden_dim = 128 (one 128-wide group per SM) and at least 2^20 samples, the decoder backward of sample chunk
c+1 runs beside the table scatter of chunk c on a side stream."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import oracle as O


def _trace_step(W, onef, spc, o, d, tgt):
    from gpu_util import nef_from_oracle, packed_grads
    nef, _ = nef_from_oracle(onef, spc)
    tracer = W.PackedRFTracer('ray', 2048, bg_color=(0.0, 0.0, 0.0)); tracer.seed = 9; tracer.precision = 1
    rb = W.Pipeline(nef, tracer)(rays=W.Rays(torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda(), 0.0, 10.0), channels=["rgb"])
    torch.nn.functional.smooth_l1_loss(rb.rgb, tgt).backward()
    return tracer.get_prev_num_samples(), rb.rgb.detach().cpu().numpy(), packed_grads(nef)


def test_wide_decoder_chunked_backward_matches_single_pass(monkeypatch):
    """The chunked schedule (wb_rf_shade_bwd) against the decoder backward and the table scatter over all samples at once
    (wb_rf_decoder_bwd + wb_rf_table_scatter, ops.SPLIT_BWD) on the same rays, seed and weights: same samples, rgb within fp16
    round-off, gradients within the precision-1 tolerance (the two differ in the order of the atomic sums only)."""
    import wisp_b200 as W
    onef = O.make_nef(feature_std=0.2, seed=3, hidden_dim=128)
    spc = O.octree_to_spc(O.points_to_octree(O.lego_like_points(6), 6))
    o, d = O.look_at_rays([-3.0, 0.65, -3.0], [0, 0, 0], 256, 256, 30.0)
    tgt = torch.sigmoid(torch.randn(o.shape[0], 3, generator=torch.Generator().manual_seed(2))).cuda()
    n_a, rgb_a, grads_a = _trace_step(W, onef, spc, o, d, tgt)
    monkeypatch.setattr(W.ops, "SPLIT_BWD", True)
    n_b, rgb_b, grads_b = _trace_step(W, onef, spc, o, d, tgt)
    assert n_a == n_b >= 1 << 20                     # the chunked schedule only runs from 2^20 samples on
    print("samples", n_a, "max |rgb diff|", float(np.abs(rgb_b - rgb_a).max()))
    np.testing.assert_allclose(rgb_b, rgb_a, atol=2e-3)
    for a, b, name in zip(grads_a, grads_b, ("table", "dens", "col")):
        diff, scale = np.abs(a - b).max(), np.abs(a).max()
        print(name, "max |grad diff| / max |grad|", float(diff / scale))
        assert diff <= 3e-2 * scale, name
