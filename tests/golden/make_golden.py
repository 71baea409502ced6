"""Generate tests/golden/*.npz by running the REFERENCE's own pure-PyTorch code on CPU.

Run in the build container only (needs /root/reference, which does not exist on the GPU box):

    python tests/golden/make_golden.py

The reference cannot travel, so the vectors are committed as small fixtures together with this
script (task section 3).  Native-only reference ops (voxlib / gridencoder CUDA extensions) are
not runnable on CPU; where the reference's Python calls them, this script plugs in
  * the reference's own pure-PyTorch positional_encoding_pt for voxlib.positional_encoding, and
  * the oracle's hash-grid encoder (itself checked against the reference CUDA extension on the
    GPU box by tests/test_vs_reference_gpu.py)
so that `_forward_perpix` (imaginaire/generators/scenedreamer.py:313-428) runs unmodified.
"""
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, '..', '..'))
REF = os.environ.get('SD_REFERENCE_ROOT', '/root/reference')
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)

import oracle  # noqa: E402
from scenedreamer_b200 import synth  # noqa: E402


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install_stubs():
    # import-time dependencies that are absent offline and never executed on this path (SURVEY 8b)
    _stub('upfirdn2d_cuda')
    _stub('bias_act_cuda')
    _stub('imageio')
    mpl = _stub('matplotlib')
    mpl.use = lambda *a, **k: None
    _stub('matplotlib.pyplot')
    _stub('matplotlib.colors')
    mpl.pyplot = sys.modules['matplotlib.pyplot']
    # top-level `voxlib` extension: only positional_encoding is reachable on CPU
    vox = _stub('voxlib')
    vox.ray_voxel_intersection_perspective = oracle.ray_voxel_intersection_perspective
    vox.sp_trilinear_worldcoord = vox.sp_trilinear_worldcoord_backward = None
    vox.positional_encoding_backward = None

    def _pe(x, ndeg, dim, incl_orig):
        from imaginaire.model_utils.gancraft.voxlib.positional_encoding import positional_encoding_pt
        return positional_encoding_pt(x, ndeg, dim, incl_orig)
    vox.positional_encoding = _pe
    _stub('_gridencoder')


def golden_sampling(out):
    from imaginaire.model_utils.gancraft import mc_utils
    g = torch.Generator().manual_seed(11)
    N, H, W, M = 1, 6, 7, 6
    # entries/exits along a ray: increasing t with gaps, NaN tail on some rays, all-NaN (sky) on others
    seg = torch.rand(N, H, W, M, 2, generator=g) * torch.tensor([1.5, 1.2]) + 0.01
    t = torch.cumsum(seg.reshape(N, H, W, 2 * M), -1) + 20
    entry, exit_ = t[..., 0::2], t[..., 1::2]
    nhit = torch.randint(0, M + 1, (N, H, W), generator=g)
    k = torch.arange(M).view(1, 1, 1, M)
    miss = k >= nhit[..., None]
    entry = entry.masked_fill(miss, float('nan'))
    exit_ = exit_.masked_fill(miss, float('nan'))
    depth2 = torch.stack([entry, exit_], 1).unsqueeze(-1)          # [N,2,H,W,M,1]
    for nsamples in (25, 5):
        rd, nd, idx = mc_utils.sample_depth_batched(depth2.clone(), nsamples, deterministic=True,
                                                    use_box_boundaries=False, sample_depth=3)
        out['samp_det%d_rand_depth' % nsamples] = rd.numpy()
        out['samp_det%d_new_dists' % nsamples] = nd.numpy()
        out['samp_det%d_idx' % nsamples] = idx.numpy()
    # stratified branch: make torch.rand return known uniforms
    u = torch.rand(N, H, W, 25, 1, generator=g)
    real_rand = torch.rand
    mc_utils.torch.rand = lambda *a, **kw: u.clone()
    try:
        rd, nd, idx = mc_utils.sample_depth_batched(depth2.clone(), 25, deterministic=False,
                                                    use_box_boundaries=False, sample_depth=3)
    finally:
        mc_utils.torch.rand = real_rand
    out['samp_depth2'] = depth2.numpy()
    out['samp_uniforms'] = u.numpy()
    out['samp_rnd_rand_depth'] = rd.numpy()
    out['samp_rnd_new_dists'] = nd.numpy()
    out['samp_rnd_idx'] = idx.numpy()
    # volum_rendering_relu
    sigma = torch.randn(N, H, W, 24, 1, generator=g) * 30
    dists = torch.rand(N, H, W, 24, 1, generator=g) * 0.05
    out['vr_sigma'] = sigma.numpy()
    out['vr_dists'] = dists.numpy()
    out['vr_weights'] = mc_utils.volum_rendering_relu(sigma, dists, dim=-2).numpy()


def golden_label_lut(out):
    from imaginaire.model_utils.gancraft import mc_utils
    lt = mc_utils.MCLabelTranslator()
    out['mc2reduced_lut'] = lt.mcid2rdid_lut.numpy().astype(np.int32)
    out['label_meta'] = np.array([lt.get_num_reduced_lbls(), lt.ignore_id, lt.dirt_id, lt.water_id], dtype=np.int32)
    ids = torch.tensor([0, 1, 8, 9, 17, 18, 26, 28, 30, 679], dtype=torch.int32)
    out['mc2reduced_probe_in'] = ids.numpy()
    out['mc2reduced_probe_out'] = lt.mc2reduced(ids, ign2dirt=True).numpy().astype(np.int32)
    return lt


def load_into(module, P, prefix):
    sd = {k[len(prefix) + 1:]: v for k, v in P.items() if k.startswith(prefix + '.')}
    missing = module.load_state_dict(sd, strict=True)
    return missing


def golden_mlps(out):
    from imaginaire.model_utils.layers import LightningMLP
    from imaginaire.generators.gancraft_base import SKYMLP, StyleMLP
    g = torch.Generator().manual_seed(5)
    for tag, stress in (('spec', False), ('stress', True)):
        P = oracle.make_params(seed=3, stress=stress, table_entries=8)
        net = LightningMLP(128, style_dim=256, viewdir_dim=0, mask_dim=12, out_channels_s=1, out_channels_c=64,
                           use_seg=True)
        load_into(net, P, 'render_net')
        sky = SKYMLP(33, style_dim=256, out_channels_c=64)
        load_into(sky, P, 'sky_net')
        sty = StyleMLP(128, 256, num_layers=5, normalize_input=True)
        load_into(sty, P, 'style_net')
        zin = torch.randn(2, 128, generator=g)
        x = torch.randn(2, 3, 4, 5, 128, generator=g) * (0.5 if stress else 0.05)
        lab = torch.randint(0, 12, (2, 3, 4, 5), generator=g)
        m = torch.nn.functional.one_hot(lab, 12).float()
        pe = torch.randn(2, 3, 4, 1, 33, generator=g)
        with torch.no_grad():
            z = sty(zin)
            s, c = net(x, None, z, m)
            skyc = sky(pe, z)
        for k, v in dict(zin=zin, z=z, x=x, lab=lab, sigma=s, c=c, pe=pe, sky=skyc).items():
            out['mlp_%s_%s' % (tag, k)] = v.numpy()


def golden_pe(out):
    from imaginaire.model_utils.gancraft.voxlib.positional_encoding import positional_encoding_pt
    g = torch.Generator().manual_seed(2)
    x = torch.rand(5, 7, 3, generator=g) * 2 - 1
    out['pe_in'] = x.numpy()
    out['pe_out_5_orig'] = positional_encoding_pt(x, 5, -1, True).numpy()
    out['pe_out_4_dim1'] = positional_encoding_pt(x, 4, 1, False).numpy()


def golden_grid_offsets(out):
    sys.path.insert(0, REF)
    from gridencoder.grid import GridEncoder
    ge = GridEncoder(input_dim=5, num_levels=16, level_dim=8, base_resolution=16, log2_hashmap_size=19,
                     desired_resolution=2048, gridtype='hash', align_corners=False)
    out['ge5_offsets'] = ge.offsets.numpy()
    out['ge5_per_level_scale'] = np.array([ge.per_level_scale], dtype=np.float64)
    ge3 = GridEncoder(input_dim=3, num_levels=8, level_dim=2, base_resolution=4, log2_hashmap_size=12,
                      desired_resolution=64)
    out['ge3_offsets'] = ge3.offsets.numpy()
    out['ge3_per_level_scale'] = np.array([ge3.per_level_scale], dtype=np.float64)


def golden_forward_perpix(out, lt):
    """Run the reference Generator._forward_perpix itself on a tiny frame."""
    from imaginaire.generators import scenedreamer as sd
    world = synth.SyntheticVoxelWorld(size=128, seed=7)
    pose = synth.eval_camera_poses(world, maxstep=8, pattern=0)[1]
    o, d, u, f, c, res = synth.frame_camera(world, pose, resolution_hw=(20, 28), pad=4)
    vid, dep, rdirs = oracle.ray_voxel_intersection_perspective(world.voxel_t, o, d, u, f, c, res, 6)
    offsets, pls = oracle.grid_offsets()
    for tag, stress in (('spec', False), ('stress', True)):
        P = oracle.make_params(seed=9, stress=stress)
        self = types.SimpleNamespace()
        self.pe_params = [0, 0, 0, False]            # feat PE unused, viewdir disabled (gancraft_base.py:331-347)
        self.pe_params_sky = [5, True]
        self.num_samples = 24
        self.sample_use_box_boundaries = False
        self.num_blocks_early_stop = 6
        self.coarse_deterministic_sampling = True
        self.sample_depth = 3
        self.label_trans = lt
        self.num_reduced_labels = lt.get_num_reduced_lbls()
        self.raw_noise_std = 0.0
        self.dists_scale = 0.25
        self.keep_sky_out = True
        self.keep_sky_out_avgpool = True
        self.sky_global_avgpool = True
        self.sky_replace_color = None
        self.clip_feat_map = True
        self.voxel = world

        def hash_encoder(x):
            return oracle.grid_encoder_module_forward(x, P['hash_encoder.embeddings'], offsets, pls)

        def render_net(x, raydir, z, m):
            lab = m.argmax(-1)
            s, cc = oracle.render_mlp(x.reshape(1, -1, 128), z, lab.reshape(1, -1), P)
            return s.reshape(*x.shape[:-1], 1), cc.reshape(*x.shape[:-1], 64)

        def sky_net(x, z):
            return oracle.sky_mlp(x.reshape(1, -1, 33), z, P).reshape(*x.shape[:-1], 64)
        self.hash_encoder, self.render_net, self.sky_net = hash_encoder, render_net, sky_net
        self._forward_perpix_sub = types.MethodType(sd.Generator._forward_perpix_sub, self)
        g = torch.Generator().manual_seed(8888)
        z = oracle.style_mlp(torch.randn(1, 128, generator=g), P)
        genc = torch.tanh(torch.randn(1, 2, generator=g))
        with torch.no_grad():
            ret = sd.Generator._forward_perpix(self, None, vid.unsqueeze(0), dep.unsqueeze(0), rdirs.unsqueeze(0),
                                               o.unsqueeze(0), z, genc)
        names = ['net_out', 'new_dists', 'weights', 'total_weights_raw', 'rand_depth', 'net_out_s', 'net_out_c',
                 'skynet_out_c', 'nosky_mask', 'sky_mask', 'sky_only_mask', 'new_idx']
        for n, v in zip(names, ret):
            if n == 'net_out_c':           # 4.7 MB in full: keep two image rows only
                v = v[:, 10:12]
            out['fpp_%s_%s' % (tag, n)] = v.numpy()
        out['fpp_%s_z' % tag] = z.numpy()
        out['fpp_%s_genc' % tag] = genc.numpy()
    out['fpp_voxel_id'] = vid.numpy()
    out['fpp_depth2'] = dep.numpy()
    out['fpp_raydirs'] = rdirs.numpy()
    out['fpp_cam'] = np.concatenate([o.numpy(), d.numpy(), u.numpy(), [f], c, res]).astype(np.float64)
    out['fpp_voxel_dims'] = np.array(world.voxel_t.shape, dtype=np.int64)


def main():
    install_stubs()
    torch.manual_seed(0)
    a, b = {}, {}
    golden_sampling(a)
    lt = golden_label_lut(a)
    golden_mlps(a)
    golden_pe(a)
    golden_grid_offsets(a)
    np.savez_compressed(os.path.join(HERE, 'ref_python_ops.npz'), **a)
    golden_forward_perpix(b, lt)
    b = {k: (v.astype(np.float32) if v.dtype == np.float64 and not k.endswith('cam') else v) for k, v in b.items()}
    stress = {k: v for k, v in b.items() if k.startswith('fpp_stress_')}           # two files, each under 1 MB
    np.savez_compressed(os.path.join(HERE, 'ref_forward_perpix.npz'), **{k: v for k, v in b.items() if k not in stress})
    np.savez_compressed(os.path.join(HERE, 'ref_forward_perpix_stress.npz'), **stress)
    for f in ('ref_python_ops.npz', 'ref_forward_perpix.npz', 'ref_forward_perpix_stress.npz'):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, 'KiB')


if __name__ == '__main__':
    main()
