#!/usr/bin/env python
"""bench.py - crops/s of the MeTRAbs crop-model hot path (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port, torch-cpu)
  python bench.py --steps K --warmup W --dump-outputs DIR  # also writes the last timed step's joints as DIR/coords3d_abs.npy

One JSON line on rank 0.  `value`: whole-job crops/s with the crops already resident in HBM.  `e2e`: the same metric
through the reference-facing host-buffer call (mtb_forward_host: pinned host crops -> H2D -> forward -> D2H joints).
`roofline`: the dominant kernel class, timed live with CUDA events on the launching stream inside the timed region.
`cpu_baseline`: the oracle port on the box's host cores on a bounded sample (rank 0, N=1 only)."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = 'crops/sec'
DUMP_LIMIT_BYTES = 64e6  # --dump-outputs writes at most this much
NAMES = {'s': 'efficientnetv2-s', 'm': 'efficientnetv2-m', 'l': 'efficientnetv2-l', 'tiny': 'efficientnetv2-tiny',
         'resnet50': 'resnet50', 'mobilenetv3-small': 'mobilenetv3-small'}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10,
                    help='timed steps of `value`, `e2e`, the graph replay and --impl reference (the tf32x3 sibling line runs '
                         'min(steps, 5); the frames leg and the CPU baseline run fixed counts)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--size', default='l', choices=list(NAMES))
    ap.add_argument('--side', type=int, default=256)
    ap.add_argument('--stride', type=int, default=32, help='stride_test (ResNet-50 config c2: 8)')
    ap.add_argument('--depth', type=int, default=8, help='heatmap depth D (config c2: 32)')
    ap.add_argument('--joints', type=int, default=24)
    ap.add_argument('--batch', type=int, default=256, help='crops per GPU per step (weak scaling) / per step in total (strong)')
    ap.add_argument('--scaling', default=os.environ.get('MTB_BENCH_SCALING', 'weak'), choices=['weak', 'strong'],
                    help='weak: --batch crops per GPU; strong: --batch crops in total, split over the GPUs (BASELINE config c3)')
    ap.add_argument('--no-frames', action='store_true', help='skip the frames -> poses leg (crop generation + TTA merge around the model)')
    ap.add_argument('--no-parity', action='store_true', help='skip the device-vs-oracle joint error of the benchmarked mode')
    ap.add_argument('--no-parity-line', action='store_true', help='skip the tf32x3 (parity mode) sibling measurement')
    ap.add_argument('--precision', default=os.environ.get('MTB_BENCH_PRECISION', 'bf16'), choices=['fp32', 'bf16', 'tf32x3'])
    ap.add_argument('--cpu-sample', type=int, default=16, help='crops per CPU-baseline iteration')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--graph', type=int, default=int(os.environ.get('MTB_BENCH_GRAPH', '0')),
                    help='1: replay the forward from a CUDA graph in the `value` region (mtb_forward never syncs or allocates)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the joints of the last timed step to DIR/coords3d_abs.npy (float32), to compare two builds '
                         'output for output (the inputs and weights are seeded, so the same arguments give the same inputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes what the CUDA path computed: use it with --impl b200')
    return args


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p['hbm_gbs'], tflops=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    tflops_burst=p['bf16_tflops'], source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, tflops=1400.0, tflops_burst=1590.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index), '-lms', '100'], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        window = [ln for (t, ln) in self.lines if t0 is None or (t0 <= t <= t1 + 0.15)]
        if not window:  # timed region shorter than the sampling period: use the samples taken under warm-up load
            window = [ln for (_, ln) in self.lines[-3:]]
        for ln in window:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], f[5:9]):
                if v.lower() == 'active':
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def build_model(args, device):
    import metrabs_b200
    from metrabs_b200.backbones import efficientnet as E
    from metrabs_b200.init import conditioned_random_init_
    from metrabs_b200.models.metrabs import Metrabs
    import types
    metrabs_b200.set_config(metrabs_b200.Config(proc_side=args.side, precision=args.precision,
                                                stride_test=getattr(args, 'stride', 32), depth=getattr(args, 'depth', 8)))
    ji = types.SimpleNamespace(names=[f'j{i}' for i in range(args.joints)], stick_figure_edges=[(0, 1)],
                               n_joints=args.joints)
    if args.size == 'resnet50':
        from metrabs_b200.backbones import resnet
        backbone = resnet.resnet50()
    elif args.size == 'mobilenetv3-small':
        from metrabs_b200.backbones import mobilenet_v3
        backbone = mobilenet_v3.mobilenet_v3_small()
    else:
        backbone = torch.nn.Sequential(E.PreprocLayer(), E.EfficientNet(args.size).features)
    model = Metrabs(backbone, ji).eval()
    conditioned_random_init_(model, seed=0)
    return model.to(device) if device is not None else model


def synthetic(batch, side, seed):
    g = torch.Generator().manual_seed(seed)
    crops = torch.rand(batch, 3, side, side, generator=g)
    f = 1000 + 500 * torch.rand(batch, generator=g)
    k = torch.zeros(batch, 3, 3)
    k[:, 0, 0] = f
    k[:, 1, 1] = f
    k[:, 0, 2] = side / 2
    k[:, 1, 2] = side / 2
    k[:, 2, 2] = 1
    return crops, k


def cpu_topology():
    """What the host offers this process: logical CPUs, affinity mask, cgroup CPU quota (printed with the baseline)."""
    info = {'cpu_count': os.cpu_count(), 'affinity': None, 'cgroup_quota_cpus': None}
    if hasattr(os, 'sched_getaffinity'):
        info['affinity'] = len(os.sched_getaffinity(0))
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            quota, period = f.read().split()
        if quota != 'max':
            info['cgroup_quota_cpus'] = float(quota) / float(period)
    except Exception:
        try:
            with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f:
                quota = int(f.read())
            with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as f:
                period = int(f.read())
            if quota > 0:
                info['cgroup_quota_cpus'] = quota / period
        except Exception:
            pass
    return info


def effective_cores():
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota (a container that
    reports 128 logical CPUs but is throttled to a few makes torch-cpu oversubscribe badly)."""
    t = cpu_topology()
    n = t['affinity'] or t['cpu_count'] or 1
    if t['cgroup_quota_cpus']:
        n = max(1, min(n, int(t['cgroup_quota_cpus'] + 0.5)))
    return n


def oracle_setup(args):
    """(state_dict, spec, PathConfig) of the oracle port for the bench workload: the device model's own weights."""
    from oracle import port
    model = build_model(args, None)
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    pcfg = port.PathConfig(proc_side=args.side, stride_test=getattr(args, 'stride', 32), depth=getattr(args, 'depth', 8))
    if args.size in ('resnet50', 'mobilenetv3-small'):
        from oracle import port_tf_backbones as tfb
        spec = tfb.ResNet50Spec(pcfg) if args.size == 'resnet50' else tfb.MobileNetV3SmallSpec(pcfg)
    else:
        spec = port.effnet_spec(NAMES[args.size])
    return sd, spec, pcfg


def best_thread_count(args, sd, spec, pcfg, probe_crops=4):
    """All the host threads torch-cpu can actually USE, probed ON THE REAL WORKLOAD (BASELINE.md section 2): one forward of
    `probe_crops` crops of the bench model per candidate count, fastest wins (on shared hosts 'all logical CPUs' can be far
    slower than a moderate count).  Returns (threads, {count: seconds})."""
    from oracle import port
    eff = effective_cores()
    cands = sorted({eff, min(eff, 96), min(eff, 64), min(eff, 32), min(eff, 16), min(eff, 8)}, reverse=True)
    crops, k = synthetic(probe_crops, args.side, 0)
    best, best_t, seen = cands[-1], float('inf'), {}
    with torch.inference_mode():
        for n in cands:
            torch.set_num_threads(n)
            t0 = time.perf_counter()
            port.metrabs_forward(sd, spec, pcfg, args.joints, crops, k)
            dt = time.perf_counter() - t0
            seen[n] = round(dt, 3)
            if dt < best_t:
                best, best_t = n, dt
            if dt > 20:  # a badly oversubscribed count: do not spend the budget probing smaller ones at the same size
                break
    return best, seen


def cpu_reference_forward(args, n_crops, iters, warmup, setup=None):
    """The reference's CPU path (oracle port of metrabs_pytorch Metrabs.forward, torch-cpu fp32, all usable host threads) on
    `n_crops` synthetic crops per iteration, in chunks of <= 32 crops; `warmup` warm-ups + `iters` timed iterations, median
    (BASELINE.md section 2).  -> (crops/s, threads, median seconds per iteration, description dict)."""
    from oracle import port
    sd, spec, pcfg = setup or oracle_setup(args)
    threads, probe = best_thread_count(args, sd, spec, pcfg)
    torch.set_num_threads(threads)
    crops, k = synthetic(n_crops, args.side, 0)
    times = []
    with torch.inference_mode():
        for i in range(warmup + iters):
            t0 = time.perf_counter()
            for c0 in range(0, n_crops, 32):
                port.metrabs_forward(sd, spec, pcfg, args.joints, crops[c0:c0 + 32], k[c0:c0 + 32])
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    times.sort()
    med = times[len(times) // 2]
    desc = dict(cpu_topology(), threads_used=threads, thread_probe_seconds=probe, iterations=len(times), warmup=warmup)
    return n_crops / med, threads, med, desc


def workload_name(args):
    return (f'{NAMES[args.size]} {args.side}x{args.side} J={args.joints} D={args.depth} stride={args.stride}, {args.batch} crops'
            f'{"/GPU" if args.scaling == "weak" else " total"}/step '
            f'(BASELINE.json metric: crops/sec, 256x256, EffNetV2-L, 24 joints)')


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n = args.cpu_sample
    v, cores, sec, desc = cpu_reference_forward(args, n, args.steps, args.warmup)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'crops/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
        'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_name(args), 'note': 'reference arm = oracle port of the reference forward on '
                   'torch-cpu (the reference is pure Python; /root/reference is absent on the GPU box)'},
        'cpu_baseline': {'value': v, 'unit': 'crops/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{n} crops per step (chunks <= 32), 2 warm-ups + {desc["iterations"]} timed steps, median', 'host': desc},
        'e2e': {'value': v, 'unit': 'crops/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def parity_check(args, model, n_crops=4, setup=None):
    """Joints of the benchmarked device mode vs the fp32 oracle port on `n_crops` synthetic crops of the bench workload:
    ||dev - ref||inf / ||ref||inf (SURVEY.md 8d), against the 1e-3 bar of BASELINE.json."""
    from oracle import port
    sd, spec, pcfg = setup or oracle_setup(args)
    crops, k = synthetic(n_crops, args.side, 7)
    torch.set_num_threads(min(effective_cores(), 16))
    with torch.inference_mode():
        ref = port.metrabs_forward(sd, spec, pcfg, args.joints, crops, k)
    dev = next(model.parameters()).device
    out = model((crops.to(dev), k.to(dev))).cpu()
    err = port.relative_error(out, ref)
    return {'joints_rel_err_vs_oracle': err, 'tolerance': 1e-3, 'meets_tolerance': bool(err < 1e-3), 'crops': n_crops,
            'precision_mode': args.precision}


def frames_leg(args, model, device, iters=5):
    """SURVEY.md 8f-1/2: the same crop model fed from FULL FRAMES by this package's Pose3dEstimator - u8 frames + person boxes
    -> pyramid -> per-crop matrices -> ONE warp launch for all num_aug x n_boxes crops -> mtb_forward -> TTA merge - all on
    the device.  8 frames of 720x1280 with 51 boxes in total x 5 augmentations = 255 crops per call (about one bench batch)."""
    from metrabs_b200.multiperson import Pose3dEstimator, warping
    from metrabs_b200.multiperson.multiperson_model import aug_parameters
    j = args.joints
    model.joint_names = [f'j{i}' for i in range(j)]
    model.joint_edges = [[0, 1]]
    est = Pose3dEstimator(model, {'': dict(indices=list(range(j)), names=model.joint_names, edges=[[0, 1]])}, None)
    g = torch.Generator().manual_seed(11)
    n_img, h, w = 8, 720, 1280
    frames = torch.randint(0, 256, (n_img, 3, h, w), generator=g, dtype=torch.uint8).to(device)
    counts = [7, 6, 7, 6, 6, 7, 6, 6]
    boxes = []
    for c in counts:
        xy = torch.rand(c, 2, generator=g) * torch.tensor([w - 400., h - 500.])
        wh = torch.tensor([180., 400.]) * (0.6 + 0.8 * torch.rand(c, 2, generator=g))
        boxes.append(torch.cat([xy, wh, torch.rand(c, 1, generator=g)], dim=1))
    kw = dict(intrinsic_matrix=torch.tensor([[[1100., 0, w / 2], [0, 1100., h / 2], [0, 0, 1]]]),
              distortion_coeffs=torch.tensor([[-0.05, 0.01, 0.0005, -0.0005, 0.001]]),
              extrinsic_matrix=torch.eye(4)[None], world_up_vector=torch.tensor([0., -1., 0.]), default_fov_degrees=55,
              internal_batch_size=0, antialias_factor=1, num_aug=5, average_aug=True, skeleton='', suppress_implausible_poses=False)
    for _ in range(2):
        est._estimate_poses_batched(frames, boxes, **kw)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(iters):
        res = est._estimate_poses_batched(frames, boxes, **kw)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / iters
    n_box = sum(counts)
    # the warp launch alone (255 crops of SxS fp32 written, bilinear gathers from the u8 frames / the pyramid)
    pyr = warping.build_pyramid(frames)
    k_box = kw['intrinsic_matrix'].repeat(n_box, 1, 1).to(device)
    d_box = kw['distortion_coeffs'].repeat(n_box, 1).to(device)
    up = torch.tensor([[0., -1., 0.]]).repeat(n_box, 1).to(device)
    ids = torch.repeat_interleave(torch.arange(n_img), torch.tensor(counts))
    gam, sc, fl, rf = aug_parameters(5)
    new_k, rot, inv, lev = warping.crop_setup(torch.cat(boxes).to(device), k_box, d_box, up, rf, sc, args.side, 1)
    out = torch.empty(5 * n_box, 3, args.side, args.side, device=device)
    for _ in range(2):
        warping.warp_images_with_pyramid(frames, pyr, k_box, inv, d_box, lev, gam / 2.2, args.side, ids, 5, 1, out=out)
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    for _ in range(iters):
        warping.warp_images_with_pyramid(frames, pyr, k_box, inv, d_box, lev, gam / 2.2, args.side, ids, 5, 1, out=out)
    w1.record()
    torch.cuda.synchronize()
    warp_ms = w0.elapsed_time(w1) / iters
    return {'what': 'frames -> poses through metrabs_b200.multiperson.Pose3dEstimator (pyramid, crop setup, one-launch warp, crop model, '
                    'TTA merge), device resident', 'frames': n_img, 'frame_size': [h, w], 'boxes': n_box, 'num_aug': 5,
            'crops_per_call': 5 * n_box, 'ms_per_call': ms, 'crops_per_s': 5 * n_box / (ms / 1e3), 'persons_per_s': n_box / (ms / 1e3),
            'warp_kernel_ms': warp_ms, 'warp_kernel_write_gbs': out.numel() * 4 / (warp_ms / 1e3) / 1e9,
            'poses3d_finite': bool(all(torch.isfinite(p).all() for p in res['poses3d']))}


def time_mode(args, eng, world, rank, device, dist, sharded_inputs):
    """Warm-up + timed loop of one precision mode.  -> dict(elapsed_ms, launches, prof_all (last warm-up step, warm),
    prof_dom, dom_name, clocks, e2e_ms, e2e_mode, graph_ms)."""
    crops_h, k_h, k_all_h, crops_d, k_d, k_all_d, out_d = sharded_inputs
    B, S, J = crops_d.shape[0], args.side, args.joints

    def step():
        if world > 1:  # local backbone + head decode, ONE all-gather of [c2d|c3d], full-batch reconstruction (mtb_forward_sharded)
            return eng.forward_sharded(crops_d, k_all_d, out=out_d)
        return eng.forward(crops_d, k_d, out=out_d)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    graph = None
    if args.graph and world == 1:
        step()
        torch.cuda.synchronize()
        graph = eng.capture_forward(crops_d, k_d, out_d)
    sampler = ClockSampler(device.index)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup - 1, 2)):
        step()
    # the LAST warm-up step with every kernel class bracketed by events: a WARM per-class profile (share_of_step)
    torch.cuda.synchronize()
    eng.profile_begin(None)
    step()
    torch.cuda.synchronize()
    prof_all = eng.profile_end()
    dom_name = max(prof_all, key=lambda n: prof_all[n]['ms'])
    dom_cls = prof_all[dom_name]['cls']
    barrier()
    graph_ms = None
    if graph is not None:
        for _ in range(2):
            graph.replay()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        g0.record()
        for _ in range(args.steps):
            graph.replay()
        g1.record()
        torch.cuda.synchronize()
        graph_ms = g0.elapsed_time(g1)
    eng.profile_begin([dom_cls])
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = sampler.mark()
    ev0.record()
    launches = 0
    for _ in range(args.steps):
        step()
        launches += eng.last_launch_count
    ev1.record()
    barrier()
    t_end = sampler.mark()
    elapsed_ms = ev0.elapsed_time(ev1)
    prof_dom = eng.profile_end()[dom_name]
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    # the legs below reuse out_d: keep what the last timed step returned
    last_out = out_d.cpu() if args.dump_outputs else None

    # ---- end to end through the host-buffer entry points: pinned host crops in, host joints out, EVERY step
    e2e_ms, e2e_mode = None, None
    if world == 1:
        out_h = torch.empty(B, J, 3).pin_memory()
        eng.forward_host(crops_h, k_h, out_h)
        ref_out = out_h.clone()
        pipe_ok = not os.environ.get('MTB_BENCH_SYNC_E2E')
        if pipe_ok:
            out_hs = [torch.empty(B, J, 3).pin_memory(), torch.empty(B, J, 3).pin_memory()]
            try:
                for s_ in (0, 1):  # warm both slots (staging allocations)
                    eng.forward_host_submit(crops_h, k_h, out_hs[s_], s_)
                    eng.forward_host_wait(s_)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for i in range(args.steps):
                    s_ = i & 1
                    eng.forward_host_wait(s_)  # the step that used this slot two steps ago has delivered its joints
                    eng.forward_host_submit(crops_h, k_h, out_hs[s_], s_)
                eng.forward_host_wait(0)
                eng.forward_host_wait(1)
                torch.cuda.synchronize()
                pipe_ms = (time.perf_counter() - t0) * 1e3
                if torch.equal(out_hs[0], ref_out) and torch.equal(out_hs[1], ref_out):
                    e2e_ms = pipe_ms
                    e2e_mode = 'pipelined mtb_forward_host_submit/_wait, 2 slots (H2D of step i+1 overlaps the forward of step i)'
                else:
                    print('bench: pipelined host path disagrees with mtb_forward_host', file=sys.stderr)
            except Exception as e:  # noqa: BLE001
                print(f'bench: pipelined host path failed ({e!r})', file=sys.stderr)
        if e2e_ms is None:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                eng.forward_host(crops_h, k_h, out_h)
            torch.cuda.synchronize()
            e2e_ms = (time.perf_counter() - t0) * 1e3
            e2e_mode = 'synchronous mtb_forward_host per step'
    else:
        # N > 1: every step copies this rank's crops + the batch's intrinsics from pinned host memory, runs the sharded
        # forward (the all-gather ships THIS step's decoded joints) and reads the full result back to the host
        out_all_h = torch.empty(out_d.shape).pin_memory()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            crops_d.copy_(crops_h, non_blocking=True)
            k_all_d.copy_(k_all_h, non_blocking=True)
            eng.forward_sharded(crops_d, k_all_d, out=out_d)
            out_all_h.copy_(out_d, non_blocking=True)
            torch.cuda.synchronize()
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3
        e2e_mode = 'per step: H2D local crops + intrinsics, mtb_forward_sharded (one NCCL all-gather), D2H full joints, sync'
    return dict(elapsed_ms=elapsed_ms, launches=launches, prof_all=prof_all, prof_dom=prof_dom, dom_name=dom_name, clocks=clocks,
                e2e_ms=e2e_ms, e2e_mode=e2e_mode, graph_ms=graph_ms, last_out=last_out)


def run_b200(args):
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch with torch.distributed.run --nproc-per-node N for --gpus N')
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
    S, J = args.side, args.joints
    if args.scaling == 'strong':
        if args.batch % world:
            raise SystemExit(f'--scaling strong needs --batch divisible by the GPU count ({args.batch} % {world})')
        B = args.batch // world   # total work fixed: the batch is split over the ranks (c3: 256 crops -> 32 per GPU at N=8)
    else:
        B = args.batch            # per-GPU work fixed
    B_total = B * world
    if args.dump_outputs and B_total * J * 3 * 4 > DUMP_LIMIT_BYTES:
        raise SystemExit(f'--dump-outputs: {B_total} x {J} x 3 float32 joints exceed {DUMP_LIMIT_BYTES / 1e6:.0f} MB')

    def make_engine(precision):
        a = argparse.Namespace(**vars(args))
        a.precision = precision
        model = build_model(a, device)
        eng = model.engine(device)
        if world > 1:
            def bcast(raw):
                t = torch.tensor(list(raw) if raw is not None else [0] * 128, dtype=torch.uint8, device=device)
                dist.broadcast(t, 0)
                return bytes(t.cpu().tolist())
            eng.comm_init(rank, world, bcast)
        return a, model, eng

    # the full batch's synthetic inputs are generated identically on every rank; each rank keeps its contiguous chunk
    crops_all, k_all = synthetic(B_total, S, 100) if world > 1 and B_total <= 512 else (None, None)
    if crops_all is not None:
        crops_h, k_h = crops_all[rank * B:(rank + 1) * B].contiguous().pin_memory(), k_all[rank * B:(rank + 1) * B].contiguous().pin_memory()
        k_all_h = k_all.pin_memory()
    else:
        crops_h, k_h = synthetic(B, S, 100 + rank)
        crops_h, k_h = crops_h.pin_memory(), k_h.pin_memory()
        k_all_h = (torch.cat([synthetic(B, S, 100 + r)[1] for r in range(world)]) if world > 1 else k_h).pin_memory()
    crops_d, k_d, k_all_d = crops_h.to(device), k_h.to(device), k_all_h.to(device)
    out_d = torch.empty(B_total, J, 3, device=device)
    inputs = (crops_h, k_h, k_all_h, crops_d, k_d, k_all_d, out_d)

    a_main, model, eng = make_engine(args.precision)
    r = time_mode(a_main, eng, world, rank, device, dist, inputs)
    elapsed_ms, e2e_ms = r['elapsed_ms'], r['e2e_ms']
    if world > 1:
        t = torch.tensor([elapsed_ms, e2e_ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms, e2e_ms = t.tolist()

    # the other mode of BASELINE.md section 5 beside the headline: 'tf32x3' (parity mode: meets the 1e-3 bar on tensor cores)
    # when the headline is 'bf16' (fast mode: the reference's own deployment precision class)
    sibling = None
    if args.precision == 'bf16' and not args.no_parity_line:
        a_par = argparse.Namespace(**vars(a_main))
        a_par.steps, a_par.warmup, a_par.graph = min(args.steps, 5), 3, 0
        a_par2, model_par, eng_par = make_engine('tf32x3')
        a_par.precision = 'tf32x3'
        rp = time_mode(a_par, eng_par, world, rank, device, dist, inputs)
        pe, pe2 = rp['elapsed_ms'], rp['e2e_ms']
        if world > 1:
            t = torch.tensor([pe, pe2], device=device, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            pe, pe2 = t.tolist()
        sibling = dict(rp=rp, elapsed_ms=pe, e2e_ms=pe2, steps=a_par.steps, model=model_par, eng=eng_par, args=a_par)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:  # [B_total, J, 3] absolute camera-space joints (mm), the full batch on every rank
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, 'coords3d_abs.npy'), r['last_out'].numpy().astype(np.float32))
    pk = peaks()
    value = B_total * args.steps / (elapsed_ms / 1e3)
    e2e = B_total * args.steps / (e2e_ms / 1e3)
    flops_crop = eng.backbone_flops_per_crop

    def roofline_of(rr, precision):
        prof_dom, prof_all, dom_name = rr['prof_dom'], rr['prof_all'], rr['dom_name']
        total_ms_all = sum(v['ms'] for v in prof_all.values())
        tensor_bound = prof_dom['flops'] > 0 and (prof_dom['flops'] / max(prof_dom['bytes'], 1)) > 100
        if tensor_bound:
            achieved = prof_dom['flops'] / (prof_dom['ms'] / 1e3) / 1e12
            peak, unit, bound = pk['tflops'], 'TFLOP/s', 'tensor'
        else:
            achieved = prof_dom['bytes'] / (prof_dom['ms'] / 1e3) / 1e9
            peak, unit, bound = pk['hbm_gbs'], 'GB/s', 'hbm'
        traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tpath):  # keyed by (workload, precision) then kernel: an ncu capture of ANOTHER config is not quoted
            with open(tpath) as f:
                traffic = json.load(f).get(f'{args.size}@{args.side}:b{B}:{precision}', {}).get(dom_name)
        roof = {'kernel': dom_name, 'bound': bound, 'achieved': achieved, 'peak': peak, 'unit': unit, 'frac': achieved / peak,
                'traffic': traffic, 'launches_timed': prof_dom['launches'],
                'avg_launch_us': prof_dom['ms'] * 1e3 / prof_dom['launches'],
                'share_of_step': prof_all[dom_name]['ms'] / total_ms_all,
                'class_ms_warm_step': {n: round(v['ms'], 3) for n, v in prof_all.items()}}
        # the other tcgen05 conv kernel of the step (fused FusedMBConv blocks) and both together: the dominant CLASS holds the
        # layers that were not fused, so its fraction alone understates what the tensor-core kernels of the step achieve
        tc_names = [n for n in ('tc_conv_kernel', 'fmb_kernel', 'tc32_conv_kernel') if n in prof_all and prof_all[n]['flops'] > 0]
        if bound == 'tensor' and len(tc_names) > 1:
            fl = sum(prof_all[n]['flops'] for n in tc_names)
            ms = sum(prof_all[n]['ms'] for n in tc_names)
            roof['tensor_core_kernels'] = {n: {'ms': round(prof_all[n]['ms'], 3), 'achieved': prof_all[n]['flops'] / (prof_all[n]['ms'] / 1e3) / 1e12,
                                               'frac': prof_all[n]['flops'] / (prof_all[n]['ms'] / 1e3) / 1e12 / peak} for n in tc_names}
            roof['tensor_core_kernels']['combined'] = {'ms': round(ms, 3), 'achieved': fl / (ms / 1e3) / 1e12, 'frac': fl / (ms / 1e3) / 1e12 / peak}
        if precision == 'tf32x3' and bound == 'tensor':
            roof['note'] = ('achieved counts the USEFUL conv FLOPs (2*MACs); the kernel issues three tf32 MMAs per product at half '
                            'the bf16 rate, so its ceiling is peak/6')
            roof['frac_of_tf32x3_ceiling'] = achieved / (peak / 6.0)
        return roof

    setup = None
    parity = None
    if not args.no_parity:
        setup = oracle_setup(a_main)
        parity = parity_check(a_main, model, setup=setup)
    line = {
        'metric': METRIC, 'value': value, 'unit': 'crops/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': elapsed_ms / args.steps, 'higher_is_better': True, 'scaling': args.scaling,
        'vs_baseline': None, 'dtype': {'bf16': 'bf16', 'fp32': 'f32', 'tf32x3': 'tf32x3'}[args.precision], 'data': 'synthetic',
        'config': {'workload': workload_name(args), 'global_batch': B_total, 'crops_per_gpu': B, 'parallelism': f'dp{world}',
                   'precision_mode': args.precision, 'weights': 'conditioned random init (metrabs_b200/init.py)',
                   'l2_policy': f'inputs larger than L2: {B * 3 * S * S * 4 / 1e6:.0f} MB of crops per step'
                                if B * 3 * S * S * 4 > 126e6 else
                                f'{B * 3 * S * S * 4 / 1e6:.0f} MB of crops per step; every step streams > 1 GB of activations through L2 (126 MB)',
                   'multi_gpu_step': ('mtb_forward_sharded: local backbone + head decode, one ncclAllGather of [c2d|c3d], full-batch '
                                      'reconstruction on every rank') if world > 1 else None,
                   'backbone_gflop_per_crop': flops_crop / 1e9,
                   'tensor_util_of_peak': value / world * flops_crop / 1e12 / pk['tflops'],
                   'peaks': pk['source'],
                   'cuda_graph_replay_crops_per_s': (B_total * args.steps / (r['graph_ms'] / 1e3)) if r['graph_ms'] else None},
        'e2e': {'value': e2e, 'unit': 'crops/s',
                'h2d_bytes_per_step': B * 3 * S * S * 4 + (B_total if world > 1 else B) * 36,
                'd2h_bytes_per_step': B_total * J * 3 * 4, 'mode': r['e2e_mode']},
        'gpu_launches': r['launches'],
        'clocks': r['clocks'],
        'roofline': roofline_of(r, args.precision),
        'parity': parity,
    }
    if sibling is not None:
        rp = sibling['rp']
        pv = B_total * sibling['steps'] / (sibling['elapsed_ms'] / 1e3)
        line['parity_mode'] = {
            'precision_mode': 'tf32x3', 'what': 'the SAME workload in the mode that meets the 1e-3 joint tolerance on tensor cores '
            '(tcgen05 kind::tf32, three split products, fp32 accumulation outside the tensor core)',
            'value': pv, 'unit': 'crops/s', 'steps': sibling['steps'], 'ms_per_step': sibling['elapsed_ms'] / sibling['steps'],
            'e2e': {'value': B_total * sibling['steps'] / (sibling['e2e_ms'] / 1e3), 'unit': 'crops/s', 'mode': rp['e2e_mode']},
            'gpu_launches': rp['launches'], 'clocks': rp['clocks'], 'roofline': roofline_of(rp, 'tf32x3'),
            'tensor_util_of_peak': pv / world * flops_crop / 1e12 / pk['tflops'],
            'parity': parity_check(sibling['args'], sibling['model'], setup=setup) if not args.no_parity else None}
    if world == 1 and not args.no_frames:
        try:
            line['frames_pipeline'] = frames_leg(a_main, model, device)
        except Exception as e:  # noqa: BLE001  (an auxiliary leg must not cost the headline line)
            line['frames_pipeline'] = {'error': repr(e)}
    if world == 1 and not args.no_cpu_baseline:
        v, cores, sec, desc = cpu_reference_forward(a_main, args.cpu_sample, 5, 2, setup=setup)
        line['cpu_baseline'] = {'value': v, 'unit': 'crops/s', 'cores': cores, 'kind': 'port',
                                'sample': f'{args.cpu_sample} crops per iteration (chunks <= 32), 2 warm-ups + 5 timed iterations of the '
                                          f'oracle port (torch-cpu fp32), median {sec:.2f} s', 'host': desc}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    import faulthandler
    faulthandler.enable()
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
