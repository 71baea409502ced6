"""RenderCNN + tanh on the tensor cores (sdb_cnn_forward) against (a) the oracle's restatement evaluated in float64 on the
GPU and (b) what the reference's own `RenderCNN` module computed in fp32 with TF32 off on a B200 for the same inputs
(tests/golden/ref_cuda_ops.npz, tests/golden/make_golden_cuda.py)."""
import pytest
import torch

import oracle
from scenedreamer_b200 import rendercnn

import _golden

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
DEV = 'cuda:0'


def _inputs(H, W, seed=0):
    g = torch.Generator().manual_seed(seed)
    net_out = (torch.rand(1, H, W, 64, generator=g) * 2 - 1).to(DEV)
    z = torch.randn(1, 256, generator=g).to(DEV)
    P = {k: v.to(DEV) for k, v in oracle.make_cnn_params(seed + 1).items()}
    return net_out, z, P


@pytest.mark.parametrize('H,W', [(37, 150), (8, 128), (2, 5)])
def test_cnn_matches_float64_restatement(H, W):
    """Odd sizes: partial tiles in x (150 = 128 + 22) and y (37 rows = 18 tiles of 2 + 1), tiny frames."""
    net_out, z, P = _inputs(H, W)
    eng = rendercnn.RenderCNNEngine(P, rendercnn.PRECISION_FP16X3)
    rgb, raw = eng.forward(net_out, z)
    torch.cuda.synchronize()
    ref, ref_raw = oracle.render_cnn(net_out, z, P, dtype=torch.float64)
    e_raw = float((raw.double() - ref_raw).abs().max())
    e_rgb = float((rgb.double() - ref).abs().max())
    print('RenderCNN fp16x3 %dx%d: max|raw - f64| %.3e (|raw| max %.2f)   max|tanh - f64| %.3e' % (H, W, e_raw, float(ref_raw.abs().max()), e_rgb))
    assert e_rgb <= 1e-4 and e_raw <= 1e-3 * max(1.0, float(ref_raw.abs().max()))
    # second call re-uses pack and workspace (borders stay zero), different input
    net2 = net_out.flip(1).contiguous()
    rgb2, _ = eng.forward(net2, z)
    ref2, _ = oracle.render_cnn(net2, z, P, dtype=torch.float64)
    assert float((rgb2.double() - ref2).abs().max()) <= 1e-4
    # single-pass fp16: the accuracy class of the reference's default (cuDNN TF32)
    eng1 = rendercnn.RenderCNNEngine(P, rendercnn.PRECISION_FP16)
    rgb1, _ = eng1.forward(net_out, z)
    e1 = float((rgb1.double() - ref).abs().max())
    print('RenderCNN fp16x1 %dx%d: max|tanh - f64| %.3e' % (H, W, e1))
    assert e1 <= 2e-2


FULL_FRAME = (570, 990, 3)      # H, W, input seed


def test_cnn_matches_reference_module_full_frame():
    """The reference's own RenderCNN (fp32, TF32 off) on a C2-sized padded frame: 570 x 990."""
    H, W, seed = FULL_FRAME
    net_out, z, P = _inputs(H, W, seed=seed)
    eng = rendercnn.RenderCNNEngine(P)
    rgb, raw = eng.forward(net_out, z)
    g = _golden.load()
    _golden.check_close(g, 'cnn_rgb', rgb, rtol=0.0, atol=1e-3)
    print('RenderCNN 570x990: |ours - reference fp32| <= 1e-3 on %d sampled outputs ; reference TF32 (its default) vs its fp32 %.3e'
          % (g['cnn_rgb.idx'].size, float(g['cnn_rgb_tf32_err'])))
    t = []
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.forward(net_out, z, want_raw=False)
        b.record()
        torch.cuda.synchronize()
        t.append(a.elapsed_time(b))
    print('RenderCNN 570x990 fp16x3: %.2f ms per frame (%.0f TFLOP/s algorithmic)' % (min(t), 570 * 990 * 5.0246e6 / (min(t) * 1e-3) / 1e12))
