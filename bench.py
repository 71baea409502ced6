#!/usr/bin/env python
"""Benchmark of the SceneDreamer per-pixel render hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, libsdb200)
    python bench.py --impl reference --steps K --warmup W    # reference arm: CPU path on host cores

A "step" is ONE frame of the C2 workload (BASELINE.md): 540x960 output pixels, 24 samples/ray,
scene_size 1024, cam_mode 0, pad 30 -> 570x990 rays raycast + shaded:
    a1  ray/voxel DDA                        (sdb_ray_voxel_intersection_perspective_ex, exact empty-space flight)
    a9  sky branch: PE + SKYMLP + frame mean  (sdb_sky_forward: same tcgen05 engine, per ray)
    a2-a8, a10-a12 fused per-pixel kernel    (sdb_render_rays_forward: tcgen05 MLP, hash gather, compositing)
    f1  RenderCNN + tanh (e2e only)          (sdb_cnn_forward: tcgen05 implicit-GEMM convolution over the whole padded frame)
Credit = OUTPUT samples: 518,400 px x 24 = 12,441,600 samples per frame (padding rays are overhead).
`value` is the per-pixel path a1-a12 with inputs resident (SURVEY.md 8(d)); `e2e` goes from a host pose to the RGB image on
the host (RenderCNN included).  Both are the product default: the fused kernel runs its rows as RAY SLOTS -- a ray leaves its
row once its transmittance is < 1e-7 and the next live ray of the frame takes the row; `value_exact_march` is the same
measurement with that early termination off (every sample of every live ray shaded) -- the two differ by less than 2e-7 in the
rendered features.  `samples_shaded_per_frame` says how many of the credited samples were actually evaluated.
Each step renders a different pose of the 40-frame trajectory and L2 is flushed between steps (256 MiB memset outside the
per-step CUDA events).
Multi-GPU: weak scaling by default (every rank renders its own frames, frame f -> rank f mod N; the finished frames are
all-gathered once per step over NCCL); `--mode strong` splits ONE frame into 16-row bands dealt round-robin
to the ranks (one banded raycast and one render launch per rank).
Extra keys at N=1: `c4` (2160x3840x40), `c5_train_step` (bench_train.py), `reference_cuda_b200` (the reference renderer itself
on this GPU, and the same Python with dropin/ on the path), `cpu_baseline`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# The CPU arm runs two OpenMP pools (torch's and the oracle's libgomp); with active spinning and 100+
# threads they fight each other, so: passive waiting and a bounded thread count (set before torch loads).
CPU_THREADS = min(os.cpu_count() or 1, int(os.environ.get('SDB_CPU_THREADS', '32')))
if '--impl' in sys.argv and 'reference' in sys.argv:
    os.environ.setdefault('OMP_NUM_THREADS', str(CPU_THREADS))
    os.environ.setdefault('OMP_WAIT_POLICY', 'PASSIVE')
    os.environ.setdefault('GOMP_SPINCOUNT', '0')

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OUT_HW = (540, 960)
PAD = 30
SPP = 24
SCENE = 1024
BYTES_PER_SAMPLE = 16384 + 344.0 / SPP     # SURVEY.md 8(d): table gather + per-ray I/O
SAMPLES_PER_FRAME = OUT_HW[0] * OUT_HW[1] * SPP
PIX_PER_FRAME = OUT_HW[0] * OUT_HW[1]


DUMP_CAP_BYTES = 64 * 10**6


def write_dump(dirname, arrays):
    """--dump-outputs: every array as DIR/<name>.npy in float32.  Over DUMP_CAP_BYTES in all, each array is replaced by the
    same seeded sample of its flattened elements on every run (DIR/<name>.npy) and their flat indices (DIR/<name>_index.npy,
    float64), the two together kept within the cap."""
    os.makedirs(dirname, exist_ok=True)
    total = sum(a.size * 4 for a in arrays.values())
    budget = DUMP_CAP_BYTES - 2 * 4096 * len(arrays)                     # room for the .npy headers
    for seed, (name, a) in enumerate(sorted(arrays.items())):
        flat = np.ascontiguousarray(a, dtype=np.float32).reshape(-1)
        if total <= budget:
            np.save(os.path.join(dirname, name + '.npy'), flat.reshape(a.shape))
            continue
        n = int(flat.size * budget // (3 * total))                        # 4 B of value + 8 B of index per kept element
        idx = np.sort(np.random.default_rng(seed).choice(flat.size, size=n, replace=False))
        np.save(os.path.join(dirname, name + '.npy'), flat[idx])
        np.save(os.path.join(dirname, name + '_index.npy'), idx.astype(np.float64))


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1430.0))), 'measured'
    return 6650.0, 1400.0, 'fallback'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md): one streaming
    `nvidia-smi -lms 100` process, lines collected by this thread."""

    QUERY = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.QUERY,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), [c.strip() for c in line.split(',')]))
        except Exception:       # noqa: BLE001  (no nvidia-smi: clocks stay None)
            pass

    def stop(self, t0=None, t1=None):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=5)
        rows = [r for (t, r) in self.rows if (t0 is None or t >= t0) and (t1 is None or t <= t1)] or [r for _, r in self.rows]

        def num(x):
            try:
                return float(x)
            except ValueError:
                return None
        sm = [num(r[0]) for r in rows if r and num(r[0]) is not None]
        mx = [num(r[1]) for r in rows if len(r) > 1 and num(r[1]) is not None]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


def build_workload(device, seed=3407, scene=SCENE, pattern=0):
    import oracle
    from scenedreamer_b200 import synth
    world = synth.SyntheticVoxelWorld(scene, seed)
    poses = synth.eval_camera_poses(world, maxstep=40, pattern=pattern)
    P = oracle.make_params(seed=0, stress=True)
    g = torch.Generator().manual_seed(8888)
    z = oracle.style_mlp(torch.randn(1, 128, generator=g), P)
    genc = torch.tanh(torch.randn(1, 2, generator=g))
    lut = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_python_ops.npz'))['mc2reduced_lut']
    P.update(oracle.make_cnn_params(seed=1))                       # denoiser.* (RenderCNN), reference state-dict names
    return world, poses, P, z, genc, lut


# ----------------------------------------------------------------------------------------------------
# CPU arm: the reference's path restated for the CPU (oracle/), all host threads, bounded sample
# ----------------------------------------------------------------------------------------------------
def cpu_frame_sample(world, pose, P, z, genc, lut, crop=64):
    """One bounded sample of the C2 frame on the CPU: a crop x crop ray window in the image centre.
    Returns (seconds, samples credited)."""
    import oracle
    from scenedreamer_b200 import synth
    o, d, u, f, c, res = synth.frame_camera(world, pose, OUT_HW, PAD)
    # shift the principal point so that the crop window is the centre of the full frame
    i0, j0 = (res[0] - crop) // 2, (res[1] - crop) // 2
    cc = [c[0] - i0, c[1] - j0]
    offsets, pls = oracle.grid_offsets()
    t0 = time.perf_counter()
    vid, dep, rd = oracle.ray_voxel_intersection_perspective(world.voxel_t, o, d, u, f, cc, [crop, crop], 6)
    r = oracle.forward_perpix(P, vid.unsqueeze(0), dep.unsqueeze(0), rd.unsqueeze(0), o.unsqueeze(0), z, genc,
                              list(world.voxel_t.shape), torch.from_numpy(lut), offsets, pls, num_samples=SPP)
    oracle.render_cnn(r['net_out'], z, P)                          # RenderCNN + tanh on the same crop (gancraft_base.py:588-603)
    return time.perf_counter() - t0, crop * crop * SPP


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import oracle
    torch.set_num_threads(CPU_THREADS)
    world, poses, P, z, genc, lut = build_workload('cpu')
    crop = 64
    for w in range(args.warmup):
        cpu_frame_sample(world, poses[w % 40], P, z, genc, lut, crop)
    ts, ns = [], 0
    for k in range(args.steps):
        dt, n = cpu_frame_sample(world, poses[k % 40], P, z, genc, lut, crop)
        ts.append(dt)
        ns += n
    total = sum(ts)
    val = ns / total / 1e6
    line = {
        'impl': 'reference', 'metric': 'rendered Msamples/sec at 960x540x24spp', 'value': val, 'unit': 'Msamples/s',
        'mpix_per_s': val / SPP, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * total / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'C2: single 540x960 frame, scene_size=1024, num_samples=24, cam_mode=0 (CPU: %dx%d-ray '
                               'centre crop per step)' % (crop, crop)},
        'cpu_baseline': {'value': val, 'unit': 'Msamples/s', 'cores': CPU_THREADS, 'host_cpus': os.cpu_count(), 'kind': 'port',
                         'sample': '%dx%d-ray centre crop of the C2 frame per step: raycast + per-pixel path + RenderCNN (oracle/: C DDA + '
                                   'hash encode with OpenMP, torch fp32 MLP / conv2d), %d steps' % (crop, crop, args.steps),
                         'omp_threads': oracle.num_threads()},
        'e2e': {'value': val, 'unit': 'Msamples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
WORKLOADS = {
    # name: (output H x W, samples per ray, scene_size, camera pattern, description)
    'c2': ((540, 960), 24, 1024, 0, 'C2: single 540x960 frame, scene_size=1024, num_samples=24, cam_mode=0'),
    'c3': ((540, 960), 24, 1024, 4, 'C3: 40-frame trajectory cam_mode=4, 540x960, num_samples=24, scene_size=1024, frames sharded over the ranks'),
    'c4': ((2160, 3840), 40, 2048, 0, 'C4: single 2160x3840 frame, num_samples=40, scene_size=2048'),
}
FLOP_PER_SAMPLE = 754176          # LightningMLP, SURVEY.md 8(a8)


def pin_rank_to_gpu_numa(local):
    """One process per GPU: keep each rank's host thread on the CPUs of its GPU's NUMA node (what the reference's
    imaginaire/utils/gpu_affinity.py does through NVML) -- torchrun does not pin, and with 8 ranks the frame loop of the
    ranks driving GPUs 4-7 otherwise runs across the socket.  Returns the number of CPUs in the mask (None: unchanged)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        idx = local
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        if vis:
            ids = [v.strip() for v in vis.split(',') if v.strip()]
            if local < len(ids) and ids[local].isdigit():
                idx = int(ids[local])
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n64 = (os.cpu_count() + 63) // 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, n64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:       # noqa: BLE001  (no NVML / no permission: leave the affinity alone)
        pass
    return None


class FrameRenderer:
    """The public-API call a user makes per frame: pose (host) -> DDA -> sky -> fused render."""

    def __init__(self, world, P, z, genc, lut, device, precision, spp):
        from scenedreamer_b200 import ops, render
        import oracle
        self.ops, self.render, self.dev, self.spp = ops, render, device, spp
        self.P = {k: v.to(device) for k, v in P.items()}
        self.voxel = world.voxel_t.to(device)
        _, pls = oracle.grid_offsets()
        self.r = render.FusedPerPixelRenderer(self.P, world.voxel_t.shape, render.reduced_label_lut(lut), pls,
                                              precision=precision, preblend=True)
        self.z, self.genc = z.to(device), genc.to(device)
        from scenedreamer_b200 import rendercnn
        self.cnn = rendercnn.RenderCNNEngine(self.P)

    def image(self, out, pad):
        """f1: per-pixel features of the padded frame -> RGB [3, H - pad, W - pad] (RenderCNN + tanh on the whole frame, then
        the crop of pad/2 the reference applies to every tile, scenedreamer.py:621-622)."""
        rgb, _ = self.cnn.forward(out['net_out'], self.z, want_raw=False)
        c = pad // 2
        return rgb[0, :, c:rgb.shape[2] - c, c:rgb.shape[3] - c] if c else rgb[0]

    def set_early_stop(self, T):
        self.r.early_stop = T

    def cast(self, cam, rows=None):
        """a1 + a9 for the frame or for a band of rows (y0, y1) of it: -> (voxel_id, depth2, raydirs, sky, band sky mean, n rays)."""
        o, d, u, f, c, res = cam
        if rows is not None:
            y0, y1 = rows
            c, res = [c[0] - y0, c[1]], [y1 - y0, res[1]]          # same rays: the principal point moves with the window
        vid, dep, rd = self.ops.ray_voxel_intersection_perspective(self.voxel, o, d, u, f, c, res, 6)
        vid, dep, rd = vid.unsqueeze(0), dep.unsqueeze(0), rd.unsqueeze(0)
        sky, sky_avg = self.render.sky_forward(rd, self.r.sky_pack_for(self.z), self.r.precision)
        return vid, dep, rd, sky, sky_avg, res[0] * res[1]

    def cast_bands(self, cam, bands):
        """Several equally spaced row bands of one frame as ONE virtual image (rays are independent: the fused kernel only sees a
        list of them): one banded raycast, one sky launch -- and later one render launch -- over all of them."""
        from scenedreamer_b200 import sharding
        o, d, u, f, c, res = cam
        first, bh, stride, rows = sharding.band_spec(bands)
        vid, dep, rd = self.ops.ray_voxel_intersection_perspective(self.voxel, o, d, u, f, c, [rows, res[1]], 6, band=(first, bh, stride))
        vid, dep, rd = vid.unsqueeze(0), dep.unsqueeze(0), rd.unsqueeze(0)
        sky, sky_avg = self.render.sky_forward(rd, self.r.sky_pack_for(self.z), self.r.precision)
        return vid, dep, rd, sky, sky_avg, rows * res[1]

    def shade(self, cam, rays, sky_avg, events=None):
        vid, dep, rd, sky = rays[:4]
        if events is not None:
            events[0].record()
        out = self.r.forward(vid, dep, rd, cam[0].unsqueeze(0), self.z, self.genc, num_samples=self.spp, sky=sky, sky_avg=sky_avg)
        if events is not None:
            events[1].record()
        return out

    def frame(self, cam, events=None, rows=None):
        """cam = (ori, dir, up, f, c, res) with HOST tensors: the reference API takes the pose from the CPU
        (scenedreamer.py:569-586); it rides in the kernel arguments of the DDA and of the fused kernel, nothing is
        copied to the device per frame.  rows = (y0, y1): only that band of the padded frame."""
        rays = self.cast(cam, rows)
        return self.shade(cam, rays, rays[4], events)


def run_gpu_arm(args):
    import torch.distributed as dist
    from scenedreamer_b200 import synth, render, sharding, _lib
    world_size = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    # one process per GPU: pin each rank to its GPU's NUMA node (8 unpinned ranks migrate across sockets: round 1's straggler).  A
    # single process is left to the OS scheduler -- on a shared host the node-local cores may be the busy ones, and the host-bound
    # legs measured 3-5x slower when confined to them.
    pinned_cpus = pin_rank_to_gpu_numa(local) if world_size > 1 else None
    torch.set_num_threads(max(1, min(8, (pinned_cpus or os.cpu_count() or 8) // max(1, world_size))))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world_size > 1:
        dist.init_process_group('nccl', device_id=dev)
    precision = {'fp16': render.PRECISION_FP16, 'bf16x3': render.PRECISION_BF16X3, 'fp16x3': render.PRECISION_FP16X3}[args.precision]
    out_hw, spp, scene, pattern, wl_name = WORKLOADS[args.workload]
    strong = args.mode == 'strong'
    samples_per_frame = out_hw[0] * out_hw[1] * spp
    world, poses, P, z, genc, lut = build_workload(dev, scene=scene, pattern=pattern)
    fr = FrameRenderer(world, P, z, genc, lut, dev, precision, spp)
    fr.set_early_stop(0.0 if args.no_early_stop else None)
    cams = [synth.frame_camera(world, p, out_hw, PAD) for p in poses]
    # pinned host copies of the per-frame inputs (camera pose) and of the per-frame result
    pose_pinned = [torch.stack([c[0], c[1], c[2]]).pin_memory() for c in cams]
    res = cams[0][5]
    bands = sharding.cyclic_bands(res[0], rank, world_size) if strong else None      # thin bands, band b -> rank b mod N
    rows = bands[0] if strong else None
    band_h = sum(b[1] - b[0] for b in bands) if strong else res[0]
    band_cap = (16 if world_size > 1 else res[0]) if strong else res[0]              # rows of one band slot (2 tile rows; N=1: the frame)
    n_slots = len(bands) if strong else 1
    host_out = torch.empty(2, (n_slots * band_cap * world_size) if strong else res[0], res[1], dtype=torch.float32).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    L = _lib.lib()

    global_sky_mean = sharding.global_mean          # frame-global sky mean from band means: one 65-float all-gather

    def strong_step(cam, kev):
        """ONE frame over all ranks: this rank's bands -> [2, n_slots * band_cap, W] maps (every slot padded to band_cap rows)."""
        rays = fr.cast_bands(cam, bands)
        avg = global_sky_mean([(rays[4], rays[5])])
        out = fr.shade(cam, rays, avg, kev)
        got = torch.stack([out['depth'][0], out['total_weight'][0]])          # [2, rows of this rank's bands, W], band after band
        if got.shape[1] == n_slots * band_cap:
            return got, out
        m = torch.zeros(2, n_slots * band_cap, res[1], device=dev)            # only a rank's LAST band can be short or missing
        m[:, :got.shape[1]] = got
        return m, out

    host_rgb = torch.empty(3, out_hw[0], out_hw[1], dtype=torch.float32).pin_memory()
    e2e_image = not strong                    # the user-facing result of a frame is the IMAGE: RenderCNN + tanh (f1) on top of the path

    def one_step(k, ev=None, kev=None, cev=None, want_host=True, to_image=False):
        idx = (k if strong else (k * world_size + rank)) % len(cams)
        cam = cams[idx]
        if ev is not None:
            ev[0].record()
        pose = pose_pinned[idx]                                      # this step's inputs, pinned host memory, passed by value
        camk = (pose[0], pose[1], pose[2], cam[3], cam[4], cam[5])
        if strong:
            maps, out = strong_step(camk, kev)
        else:
            out = fr.frame(camk, kev)
            maps = fr.image(out, PAD) if to_image else torch.stack([out['depth'][0], out['total_weight'][0]])
        if world_size > 1:
            if cev is not None:
                cev[0].record()
            allm = sharding.gather_frames(maps.unsqueeze(0))         # THE collective of the path: finished frames / bands of every rank
            if cev is not None:
                cev[1].record()
            if strong:                                               # slot j of rank r is band j * N + r: back into frame order
                maps = sharding.assemble_bands(allm, world_size, n_slots, band_cap)
        if want_host:                                                # D2H of the step's result
            if to_image:
                host_rgb.copy_(maps, non_blocking=True)
            else:
                host_out[:, :maps.shape[1]].copy_(maps, non_blocking=True)
        if ev is not None:
            ev[1].record()
        return out

    for w in range(max(args.warmup, 3)):
        one_step(w, to_image=e2e_image)
        flush.zero_()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    mk = lambda: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    evs, kevs, cevs = mk(), mk(), mk()
    torch.cuda.synchronize()
    if world_size > 1:
        dist.barrier()           # AFTER rank 0 has started its clock sampler: every rank enters the timed region together
        torch.cuda.synchronize()
    launches0 = int(L.sdb_launch_count())
    t_begin = time.perf_counter()
    for k in range(args.steps):
        one_step(k, evs[k], kevs[k], cevs[k], to_image=e2e_image)
        torch.cuda.synchronize()                                     # the caller READS the step's result on the host
        flush.zero_()                                                # L2 flush between timed iterations
    torch.cuda.synchronize()
    t_wall = time.perf_counter() - t_begin
    launches = int(L.sdb_launch_count()) - launches0
    if args.dump_outputs and rank == 0:                              # the host result of the last timed step, before anything reuses it
        if e2e_image:
            dump = {'rgb': host_rgb.numpy().copy()}
        else:
            dump = {'depth': host_out[0, :res[0]].numpy().copy(), 'opacity': host_out[1, :res[0]].numpy().copy()}
    if world_size > 1:
        dist.barrier()
    step_ms = [a.elapsed_time(b) for a, b in evs]
    kern_ms = [a.elapsed_time(b) for a, b in kevs]
    pre_ms = [evs[i][0].elapsed_time(kevs[i][0]) for i in range(args.steps)]
    coll_ms = [a.elapsed_time(b) for a, b in cevs] if world_size > 1 else [0.0] * args.steps
    tot = torch.tensor([sum(step_ms), sum(kern_ms)], dtype=torch.float64, device=dev)
    if world_size > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    tot_ms, tot_kern_ms = float(tot[0]), float(tot[1])
    # per-rank table (mean ms per step): e2e step, DDA+sky before the fused kernel, fused kernel window, collective incl. wait
    mine = torch.tensor([[float(np.mean(step_ms)), float(np.mean(pre_ms)), float(np.mean(kern_ms)), float(np.mean(coll_ms)),
                          float(np.max(step_ms)), float(pinned_cpus or 0)]], dtype=torch.float64, device=dev)
    table = mine
    if world_size > 1:
        table = torch.empty(world_size, mine.shape[1], dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(table, mine)
    table = table.cpu().tolist()

    def device_only(early, steps, lead=0):
        """inputs resident, nothing copied to the host; the collective stays inside"""
        fr.set_early_stop(early)
        ms = []
        for k in range(-lead, steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            flush.zero_()
            a.record()
            one_step(max(k, 0), want_host=False)
            b.record()
            torch.cuda.synchronize()
            if k >= 0:
                ms.append(a.elapsed_time(b))
        t = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
        if world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]) / max(1, len(ms))
    dev_ms = device_only(0.0 if args.no_early_stop else None, args.steps)
    exact_ms = dev_ms if args.no_early_stop else device_only(0.0, min(args.steps, 10), lead=2)
    fr.set_early_stop(0.0 if args.no_early_stop else None)
    # clocks are sampled over BOTH timed loops (host-inclusive and device-only)
    clocks = sampler.stop(t_begin, time.perf_counter()) if rank == 0 else None

    if rank == 0:
        hbm, tf, which = measured_peaks()
        frames_per_step = 1 if strong else world_size
        value = frames_per_step * samples_per_frame / (dev_ms * 1e-3) / 1e6
        e2e = frames_per_step * samples_per_frame / (tot_ms / args.steps * 1e-3) / 1e6
        kern_s = tot_kern_ms * 1e-3 / args.steps
        # executed tensor work: live 16x8 ray tiles x steps x 128 rows, MMAs as issued (x3 split: 3 per product)
        # (rank 0 alone: no collective in here)
        wss = [fr.frame(cams[(k if strong else k * world_size) % len(cams)], rows=rows)['workspace'][:16].view(torch.int32).cpu()   # (strong: first band only)
               for k in range(min(args.steps, 8))]
        live_tiles = float(np.mean([int(w[0]) for w in wss]))         # live 16x8 tiles (tile kernel) or live RAYS (ray-slot kernel)
        steps_exec = float(np.mean([int(w[1]) for w in wss]))         # steps of 128 rows executed (after early termination)
        ray_slots = bool(int(wss[0][3]) == 1)
        mma_eq = {'fp16': (9 + 5 * 17 + 17 * 0.25), 'bf16x3': (27 + 5 * 50 + 50 * 0.25), 'fp16x3': (27 + 5 * 50 + 50 * 0.25)}[args.precision]
        exec_tflops = steps_exec * mma_eq * (2.0 * 128 * 256 * 16) / kern_s / 1e12
        cnn_ms = None
        if e2e_image:
            o_ = fr.frame(cams[0])
            ts_ = []
            for _ in range(5):
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record()
                fr.image(o_, PAD)
                b_.record()
                torch.cuda.synchronize()
                ts_.append(a_.elapsed_time(b_))
            cnn_ms = float(np.median(ts_))
        band_frac = band_h / float(res[0])
        alg_tflops = samples_per_frame * band_frac * FLOP_PER_SAMPLE / kern_s / 1e12
        traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(args.precision)
        extras = {}
        cpu = getattr(args, 'cpu_result', None)
        extras = getattr(args, 'extras_result', None) or {}
        line = {
            'metric': 'rendered Msamples/sec at 960x540x24spp', 'value': value, 'unit': 'Msamples/s',
            'mpix_per_s': value / spp, 'n_gpus': world_size, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': dev_ms, 'higher_is_better': True, 'scaling': 'strong' if strong else 'weak', 'vs_baseline': None,
            'value_exact_march': frames_per_step * samples_per_frame / (exact_ms * 1e-3) / 1e6,
            'value_exact_march_note': 'same measurement with early termination off (every sample of every live ray shaded)',
            'samples_credited_per_frame': samples_per_frame,
            'samples_shaded_per_frame': steps_exec * 128 / band_frac,
            'samples_shaded_note': 'steps executed x 128 rows (rank 0, mean over frames).  Ray-slot kernel: only live rays occupy rows, a ray '
                                   'leaves its row once it is opaque (one sample later) -- rows idle at the tail of a CTA are counted; tile kernel: '
                                   'sky-only tiles are skipped, a tile stops once every live ray is opaque',
            'dtype': {'fp16': 'f16 (f32 accumulate)', 'bf16x3': 'bf16x3 split (f32-grade), f32 accumulate',
                      'fp16x3': 'f16x3 split (f32-grade), f32 accumulate'}[args.precision] + '; table/compositing f32',
            'data': 'synthetic',
            'config': {'workload': wl_name + ', pad %d (%dx%d rays cast+shaded, %d px credited); ' % (PAD, res[0], res[1], out_hw[0] * out_hw[1]) +
                                   ('ONE frame per step in 16-row bands dealt round-robin to the GPUs' if strong else 'one frame per GPU per step'),
                       'precision': args.precision, 'l2': 'flushed between steps (256 MiB memset) + a different pose each step',
                       'table': 'per-scene pre-blended 3-D table (8 corners/level)', 'sky_mlp': 'tcgen05 engine (sdb_sky_forward)',
                       'early_termination': ('off' if args.no_early_stop else
                                             'a ray leaves its MMA row once its transmittance is < %g (skipped samples carry less than '
                                             'that compositing weight; credited like sky-only rays); --no-early-stop marches everything'
                                             % render.EARLY_STOP_T),
                       'host_affinity': ('each rank pinned to the CPUs of its GPU (NVML affinity), %s CPUs for rank 0' % pinned_cpus) if world_size > 1 else 'not pinned (single process)'},
            'e2e': {'value': e2e, 'unit': 'Msamples/s', 'h2d_bytes_per_step': int(pose_pinned[0].numel() * 4),
                    'd2h_bytes_per_step': int((host_rgb if e2e_image else host_out).numel() * 4), 'ms_per_step': tot_ms / args.steps,
                    'result': 'RGB image [3,%d,%d] fp32' % out_hw if e2e_image else 'depth + opacity maps',
                    'note': ('per step: pose from pinned host memory (by value in the launch arguments) -> DDA -> sky -> fused render -> '
                             'RenderCNN + tanh on the whole padded frame (tcgen05 implicit GEMM, fp16x3) -> crop -> RGB to pinned host, host '
                             'waits for it.  `value` is the per-pixel path alone (SURVEY 8(d): a1-a12), e2e goes on to the image, so the two '
                             'differ by the RenderCNN time (`rendercnn_ms`)') if e2e_image else
                            'per step: pose (by value) -> DDA -> sky -> fused render of this rank\'s row band -> band maps gathered -> host'},
            'gpu_launches': launches,
            'gpu_launches_note': 'counted by the library (sdb_launch_count) over the timed (e2e) region on rank 0: per step dda_perspective, '
                                 'mlp_kernel<sky>, sky_mean, set_cam, prepass_rays, mlp_kernel<render, ray slots>, set_flag, pack_input, '
                                 '7 x conv_kernel (all ours; torch adds a few slicing / copy kernels for the crop and the gather)',
            'roofline': {'bound': 'tensor', 'achieved': alg_tflops, 'peak': tf, 'unit': 'TFLOP/s', 'frac': alg_tflops / tf,
                         'traffic': (traffic or {}).get('dram_bytes_per_launch'), 'traffic_unit': 'B of DRAM per launch (ncu dram__bytes)',
                         'traffic_source': (traffic or {}).get('source'),
                         'kernel': 'rf::mlp_kernel<render> (+prepass)', 'kernel_ms': tot_kern_ms / args.steps,
                         'peak_source': which + ' (MEASURED_PEAKS.json bf16_tflops_sustained: the kernel is timed inside a long step)',
                         'what': 'ALGORITHMIC flops: credited samples x 754,176 FLOP (LightningMLP at 1 MMA per product) / kernel time',
                         'executed_tflops': exec_tflops, 'executed_frac': exec_tflops / tf,
                         'executed_what': '16-bit MMA flops as issued: tile-steps executed x MMAs per step (the parity modes issue 3 MMAs '
                                          'per product) -- the tensor-pipe occupancy; one third of it is algorithmic work',
                         'kernel_variant': 'ray slots: every MMA row is a ray with its own cursor, refilled from a queue of live rays' if ray_slots
                                           else '16x8 ray tiles marched in lock step',
                         ('live_rays_per_frame' if ray_slots else 'live_tiles_per_frame'): live_tiles, 'tile_steps_executed_per_frame': steps_exec,
                         'tile_steps_without_early_termination': (np.ceil(live_tiles / 128.0) if ray_slots else live_tiles) * spp,
                         'hbm': {'algorithmic_bytes_per_launch': samples_per_frame * BYTES_PER_SAMPLE,
                                 'algorithmic_GBps': samples_per_frame * band_frac * BYTES_PER_SAMPLE / kern_s / 1e9, 'peak_GBps': hbm,
                                 'note': 'SURVEY 8(d) prescribes 16,398 B/sample; the kernel does NOT move them (pre-blended table: 4x fewer '
                                         'corners, L2-resident gathers): measured DRAM traffic is `traffic`, ~600x lower, so HBM is not the bound'}},
            'cpu_baseline': cpu, 'clocks': clocks, 'wall_s': t_wall,
            'per_rank_ms': {'columns': ['e2e_step', 'dda_sky', 'fused_kernel_window', 'collective_incl_wait', 'e2e_step_max', 'cpus_in_affinity'],
                            'rows': table},
            'rendercnn_ms': cnn_ms,
            'collective': {'op': 'all_gather_into_tensor(%s)' % ('RGB frames in the e2e loop, depth+opacity maps in the device-only loops' if e2e_image else 'row bands of depth+opacity maps'), 'bytes_per_rank': int(2 * n_slots * band_cap * res[1] * 4) if strong else int(host_out.numel() * 4),
                           'ms_per_step_incl_wait_for_slowest_rank': float(np.mean(coll_ms))} if world_size > 1 else None,
        }
        line.update(extras)
        if args.dump_outputs:
            write_dump(args.dump_outputs, dump)
        print(json.dumps(line))
    if world_size > 1:
        dist.destroy_process_group()


def extra_legs(args):
    """Reported next to the headline at N=1 (each in a subprocess, bounded): C4 throughput, the C5 train step, and the
    reference renderer itself on this B200 (its own CUDA extensions + PyTorch, through the real Generator)."""
    ex = {}

    def run(cmd, timeout):
        def unpin():                                   # children must not inherit a CPU mask
            try:
                os.sched_setaffinity(0, range(os.cpu_count() or 1))
            except OSError:
                pass
        o = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT, preexec_fn=unpin)
        if o.returncode != 0:
            raise RuntimeError((o.stderr or o.stdout)[-300:])
        return o

    try:
        o = run([sys.executable, os.path.abspath(__file__), '--workload', 'c4', '--steps', '3', '--warmup', '3', '--no-cpu', '--no-extras'], 900)
        c4 = json.loads(o.stdout.strip().splitlines()[-1])
        ex['c4'] = {k: c4[k] for k in ('value', 'unit', 'ms_per_step', 'value_exact_march', 'samples_credited_per_frame', 'samples_shaded_per_frame')}
        ex['c4']['config'] = c4['config']['workload']
        ex['c4']['e2e'] = c4['e2e']['value']
        ex['c4']['roofline_frac'] = c4['roofline']['frac']
    except Exception as e:          # noqa: BLE001
        ex['c4'] = {'error': repr(e)[:300]}
    try:
        o = run([sys.executable, os.path.join(ROOT, 'bench_train.py'), '--steps', '8', '--warmup', '3', '--no-composition'], 900)
        ex['c5_train_step'] = json.loads(o.stdout.strip().splitlines()[-1])
    except Exception as e:          # noqa: BLE001
        ex['c5_train_step'] = {'error': repr(e)[:300]}
    try:
        import numpy as _np
        res = {}
        for backend in ('ref', 'dropin'):
            out = '/tmp/sdb_bench_%s.npz' % backend
            run([sys.executable, '-m', 'oracle.refgen', '--backend', backend, '--frames', '4', '--warm', '1', '--out', out,
                 '--workdir', '/tmp/sdb_bench_refgen'], 900)
            d = _np.load(out)
            res[backend] = (float(_np.mean(d['perpix_ms'])), float(_np.mean(d['cnn_ms'])))
        spf = SAMPLES_PER_FRAME
        ex['reference_cuda_b200'] = {
            'what': "the reference's own Generator.inference_givenstyle (unmodified Python staged in oracle/_ref/py) on this GPU: "
                    "'reference' = its own CUDA extensions compiled for sm_100a + cuBLAS/ATen, unfused 40-tile loop; 'dropin_zero_edit' = the "
                    'same Python with dropin/ on the path (class-level fused hook, one launch per frame). GPU-timeline ms per C2 frame, '
                    'per-pixel path (raycast + sky pre-pass + _forward_perpix) and RenderCNN (_forward_global) separately',
            'reference': {'perpix_ms': res['ref'][0], 'cnn_ms': res['ref'][1], 'msamples_per_s': spf / (res['ref'][0] * 1e-3) / 1e6},
            'dropin_zero_edit': {'perpix_ms': res['dropin'][0], 'cnn_ms': res['dropin'][1], 'msamples_per_s': spf / (res['dropin'][0] * 1e-3) / 1e6},
            'perpix_speedup': res['ref'][0] / res['dropin'][0]}
    except Exception as e:          # noqa: BLE001
        ex['reference_cuda_b200'] = {'error': repr(e)[:300]}
    return ex


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--precision', default='fp16x3', choices=['fp16', 'bf16x3', 'fp16x3'])
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS), help='BASELINE.json config (default: the headline, C2)')
    ap.add_argument('--mode', default='weak', choices=['weak', 'strong'],
                    help='weak: one frame per GPU per step (frames sharded); strong: ONE frame per step split into row bands')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-extras', action='store_true', help='skip the C4 / C5 / reference-CUDA legs reported next to the headline at N=1')
    ap.add_argument('--no-early-stop', action='store_true',
                    help='march every sample of every live tile (early termination off; the reference arithmetic sample for sample)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the host result of the last timed step (rank 0: in weak mode with several GPUs, its own frame) to '
                         'DIR/<name>.npy in float32: rgb [3,H,W], or in strong mode depth and opacity [rows,W].  Over 64 MB in all, '
                         'a fixed seeded sample of the flattened elements is written instead, with its flat indices in '
                         'DIR/<name>_index.npy (float64).  The inputs depend on the arguments alone')
    args = ap.parse_args()
    if args.impl == 'reference' and args.dump_outputs:
        ap.error('--dump-outputs writes what the CUDA path computed; the reference arm has nothing to dump')
    if args.impl == 'reference':
        run_reference_arm(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the product path has no CPU fallback '
                         '(use --impl reference for the CPU baseline)')
    # The legs reported NEXT TO the headline at N=1 run first, each in its own process, before this process creates its CUDA
    # context: they are host-bound in places (the reference's tile loop, autograd) and measured 3-5x slower as children of a
    # process that already held the GPU and a CPU mask.
    if int(os.environ.get('WORLD_SIZE', '1')) == 1:
        if not args.no_cpu:
            try:
                o = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '12', '--warmup', '1'],
                                   capture_output=True, text=True, timeout=600)
                args.cpu_result = json.loads(o.stdout.strip().splitlines()[-1])['cpu_baseline']
            except Exception as e:          # noqa: BLE001
                args.cpu_result = {'error': repr(e)[:200]}
        if not args.no_extras and args.workload == 'c2':
            args.extras_result = extra_legs(args)
    run_gpu_arm(args)


if __name__ == '__main__':
    main()
