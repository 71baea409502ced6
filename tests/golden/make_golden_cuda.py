"""Writes tests/golden/ref_cuda_ops.npz: what the reference's own CUDA extensions (voxlib, gridencoder) and its RenderCNN
module compute for the inputs of the GPU tests that compare with them (tests/test_gpu_ops.py, tests/test_gpu_cnn.py).

Needs a CUDA device and the reference built by oracle/build_ref.py into oracle/_ref/ (extensions and staged Python):

    python tests/golden/make_golden_cuda.py

The inputs come from the same helpers the tests call; tests/_golden.py says what is kept of each output."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS):
    if p not in sys.path:
        sys.path.insert(0, p)

import _golden                      # noqa: E402
import test_gpu_cnn as tc           # noqa: E402
import test_gpu_ops as to           # noqa: E402
from _ref_ext import load as load_ref   # noqa: E402

DEV = 'cuda:0'


def dda(out, rv):
    world = to.make_world()
    vox = world.voxel_t.to(DEV)
    for k, pattern in to.REF_DDA_FRAMES:
        o, d, u, f, c, res = to._frame(world, k, hw=(135, 240), pad=30, pattern=pattern)
        vid, dep, rd = rv.ray_voxel_intersection_perspective(vox, o, d, u, float(f), [float(c[0]), float(c[1])],
                                                             [int(res[0]), int(res[1])], 6)
        key = 'dda_%d_%d' % (k, pattern)
        _golden.record(out, key + '_vid', vid, seed=1, exact=True)
        _golden.record(out, key + '_rd', rd, seed=2, exact=True)
        _golden.record(out, key + '_dep', torch.nan_to_num(dep, nan=-1.0), seed=3, exact=True)


def table_sample(t, seed, n=_golden.SAMPLE):
    """Half of the sample from the entries the scatter touched, half from the whole table."""
    a = t.detach().contiguous().cpu().numpy().reshape(-1)
    rng = np.random.default_rng(seed)
    nz = np.flatnonzero(a)
    hit = rng.choice(nz, size=min(n // 2, nz.size), replace=False)
    anywhere = rng.choice(a.size, size=min(n // 2, a.size), replace=False)
    return np.unique(np.concatenate([hit, anywhere]))


def grid_encode(out, rg):
    for i, case in enumerate(to.GE_CASES[:3]):
        o, dd, ge, gi = to.grid_encode_fp32_case(rg, case)
        key = 'ge32_%d' % i
        _golden.record(out, key + '_out', o, seed=10 + i)
        _golden.record(out, key + '_dydx', dd, seed=20 + i)
        _golden.record(out, key + '_gemb', ge, seed=0, idx=table_sample(ge, 30 + i))
        _golden.record(out, key + '_gin', gi, seed=40 + i)
    for i, case in enumerate(to.GE16_CASES):
        o, dd, ge, gi, g32 = to.grid_encode_fp16_case(rg, case)
        key = 'ge16_%d' % i
        _golden.record(out, key + '_out', o, seed=50 + i, exact=True)
        _golden.record(out, key + '_dydx', dd, seed=60 + i, exact=True)
        _golden.record(out, key + '_gin', gi, seed=70 + i, exact=True)
        out[key + '_gemb_err'] = np.float64((ge.float() - g32).abs().max().item())


def positional_encoding(out, rv):
    x, _, gy = to.positional_encoding_inputs()
    y = rv.positional_encoding(x.to(DEV), 5, -1, True)
    gx = rv.positional_encoding_backward(gy.to(DEV), y, 5, -1, True)
    _golden.record(out, 'pe_y', y, seed=80)
    _golden.record(out, 'pe_gx', gx, seed=81)


def sp_trilinear(out, rv):
    for ign_zero, strided, C in to.SP_CASES:
        lut, feat, wc = to._sp_case(3, ign_zero, strided, C)
        key = 'sp_%d_%d_%d' % (ign_zero, strided, C)
        r = rv.sp_trilinear_worldcoord(feat.to(DEV), lut.to(DEV), wc.to(DEV), ign_zero, -1)
        r_cf = rv.sp_trilinear_worldcoord(feat.to(DEV), lut.to(DEV), wc.to(DEV), ign_zero, -3)
        go = torch.randn(r.shape, generator=torch.Generator().manual_seed(5))
        r_g, = rv.sp_trilinear_worldcoord_backward(go.to(DEV), feat.to(DEV), lut.to(DEV), wc.to(DEV), ign_zero, False)
        _golden.record(out, key + '_out', r, seed=90, exact=True, values=True)
        _golden.record(out, key + '_out_cf', r_cf, seed=90, exact=True, values=True)
        out[key + '_cf_stride'] = np.array(r_cf.stride(), dtype=np.int64)
        _golden.record(out, key + '_gfeat', r_g, seed=91)


def render_cnn(out):
    from oracle import refgen
    ref_root = refgen.reference_python_root()
    for pth in (ref_root, os.path.join(ROOT, 'dropin'), refgen.STUBS):
        if pth not in sys.path:
            sys.path.append(pth)
    from imaginaire.generators.gancraft_base import RenderCNN
    H, W, seed = tc.FULL_FRAME
    net_out, z, P = tc._inputs(H, W, seed=seed)
    mod = RenderCNN(64, style_dim=256).to(DEV)
    mod.load_state_dict({k[len('denoiser.'):]: v for k, v in P.items()})
    old = torch.backends.cudnn.allow_tf32
    try:
        with torch.no_grad():
            torch.backends.cudnn.allow_tf32 = False
            rgb = torch.tanh(mod(net_out.permute(0, 3, 1, 2).contiguous(), z))
            torch.backends.cudnn.allow_tf32 = True
            rgb_tf32 = torch.tanh(mod(net_out.permute(0, 3, 1, 2).contiguous(), z))
    finally:
        torch.backends.cudnn.allow_tf32 = old
    _golden.record(out, 'cnn_rgb', rgb, seed=100, n=16384)
    out['cnn_rgb_tf32_err'] = np.float64((rgb_tf32 - rgb).abs().max().item())


def main():
    rv, rg = load_ref('ref_voxlib'), load_ref('ref_gridencoder')
    if rv is None or rg is None:
        raise SystemExit('the reference extensions are not built into oracle/_ref/ (oracle/build_ref.py)')
    torch.backends.cuda.matmul.allow_tf32 = False
    out = {}
    dda(out, rv)
    grid_encode(out, rg)
    positional_encoding(out, rv)
    sp_trilinear(out, rv)
    render_cnn(out)
    dst = sys.argv[1] if len(sys.argv) > 1 else _golden.PATH
    os.makedirs(os.path.dirname(os.path.abspath(dst)), exist_ok=True)
    np.savez_compressed(dst, **out)
    print(dst, os.path.getsize(dst) // 1024, 'KiB,', len(out), 'arrays')


if __name__ == '__main__':
    main()
