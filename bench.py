#!/usr/bin/env python
"""bench.py -- RGB-D pair frames/sec of the se(3)-TrackNet per-frame hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 64] [--precision tf32] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of synthetic input: `batch` (default 64)
independent object tracks of one 480x640 RGB-D frame go through K0 (crop / depth clip / normalise),
the 17-conv two-branch network and K6 (R^3 x so(3) pose update)  -- BASELINE.json configs[1].
With N GPUs every rank runs its own `batch` tracks (weak scaling: 64 tracks per GPU, 512 on 8 =
configs[3]) and the per-step exchange is one NCCL all-gather of the updated poses, issued on a side
stream (nothing on a rank's data path needs its result) and waited for at the start of the next step.
Default --steps: 500 (timed region ~0.4 s); --impl reference: 20 steps of the same 64-pair workload.

Prints ONE JSON line (rank 0).  Keys beyond the base contract:
  roofline      conv stack (8 resident-weight launches + the 6-layer trunk launch) algorithmic FLOPs / their summed
                device time (CUDA events recorded inside libse3tn on the launching stream) vs the tensor peak
  weight_sets_21  the same step with 21 object classes (one checkpoint each, reference README.md:132) in the batch
  parity        N=1: every tensor-core mode vs the CPU oracle on the cpu_baseline sample; N>1: every rank's sharded
                poses vs a single-GPU rerun of the same tracks on rank 0 (must be bit-identical)
  cpu_baseline  the oracle's on_track path (torch CPU + numpy/cv2) timed on this box's host cores
  e2e           same metric through Tracker.on_track_batch with pinned HOST buffers: H2D of the frame,
                poses, rendered views and D2H of the poses inside every timed step
--impl reference: the reference's own CPU implementation of the path (oracle restatement: the
reference code itself cannot travel to the GPU box) on all host threads, bounded sample per step.
--dump-outputs DIR: after the timed steps, the poses the last timed step returned go to DIR/poses.npy (float64, one 4x4 per
track; with N > 1 also DIR/poses_all_ranks.npy, the gathered set).  Inputs are seeded: the same arguments give the same inputs.
"""
import argparse, importlib, json, os, subprocess, sys, threading, time
import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
FLOP_PER_PAIR = 5_527_109_632            # 17 convs, SURVEY.md 8d / BASELINE.md section 2
MAX_INPUT_SETS = 16                      # inputs rotate so consecutive steps differ; at most this many distinct sets
TN, RN = 0.03, 5 * np.pi / 180


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='default 500 (ours) / 20 (--impl reference)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--precision', default='bf16x3', choices=['bf16x3', 'tf32', 'bf16', 'fp32'])
    ap.add_argument('--no-alt', action='store_true', help='skip the secondary precision-mode measurements')
    ap.add_argument('--weight-sets', type=int, default=1, help='object classes (one checkpoint each, reference README.md:132); track i uses set i*G//batch')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-render', action='store_true', help='skip the step-with-rendered-input-A measurement')
    ap.add_argument('--no-g21', action='store_true', help='skip the 21-weight-set leg')
    ap.add_argument('--cpu-seconds', type=float, default=12.0)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the poses the last timed step returned (rank 0) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == 'reference' else 500
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy.  The inputs are seeded, so two builds run with the same arguments can be
    compared file for file."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + '.npy'), a)


def workload_string(nb):
    """config.workload: identical for both arms (the driver compares them)."""
    return ('BASELINE configs[1]: %d synthetic RGB-D pairs/GPU per step, full path K0 crop/normalise -> two-branch 17-conv forward -> '
            'se(3) update, 176x176, one 480x640 frame' % nb)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d, 'MEASURED_PEAKS.json'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        try:
            proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '20'],
                                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            return
        while not self.stop_flag:
            line = proc.stdout.readline()
            if not line:
                break
            self.samples.append([x.strip() for x in line.split(',')])
        proc.terminate()

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace('.', '', 1).isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace('.', '', 1).isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for k, n in enumerate(names) if any(len(s) > 2 + k and s[2 + k].lower().startswith('active') for s in self.samples)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
def usable_cpus():
    """CPUs this process may actually use: affinity mask capped by the cgroup quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def pick_threads(fn):
    """torch CPU throughput is not monotonic in thread count on big hosts: try a few, keep the fastest."""
    best, best_t = None, None
    n = usable_cpus()
    for t in sorted({n, max(1, n // 2), max(1, n // 4), min(n, 32), min(n, 16)}, reverse=True):
        torch.set_num_threads(t)
        fn()
        t0 = time.perf_counter(); fn(); dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = t, dt
    torch.set_num_threads(best)
    return best


def cpu_on_track_rate(synth, seconds, pairs_per_call=8, threads=None):
    """pairs/s of the oracle's hot path (crop+normalise per pair, one batched forward, pose update)."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import se3_oracle as O
    sd = synth.make_state_dict(0)
    mean, std = synth.default_mean_std()
    rgb, depth = synth.raw_frame(0)
    poses = synth.raw_poses(pairs_per_call, seed=0)
    rgbA, depthA = synth.rendered_views(pairs_per_call, poses, seed=0)

    def one_call():
        dA, dB = [], []
        for i in range(pairs_per_call):
            bb = O.compute_bbox(poses[i], synth.CAMERA_K, 200.0, scale=(1000, 1000, 1000))
            rB, zB = O.crop_bbox(rgb, depth, bb, (176, 176))
            (a, b), _ = O.process_data(rgbA[i], depthA[i], poses[i], rB, zB, np.eye(4), mean, std)
            dA.append(torch.from_numpy(a)); dB.append(torch.from_numpy(b))
        out = O.forward(sd, torch.stack(dA), torch.stack(dB))
        return [O.process_predict(poses[i], (out['trans'][i].numpy(), out['rot'][i].numpy())) for i in range(pairs_per_call)]

    threads = pick_threads(one_call)                      # includes warm-up
    t0 = time.perf_counter(); calls = 0
    while True:
        one_call(); calls += 1
        if time.perf_counter() - t0 >= seconds and calls >= 2:
            break
    dt = time.perf_counter() - t0
    ref_poses = np.stack(one_call())
    return calls * pairs_per_call / dt, threads, '%d calls x %d pairs in %.1f s (same frame/pose generators as the GPU arm)' % (calls, pairs_per_call, dt), (rgb, depth, poses, rgbA, depthA, ref_poses)


def run_reference(args, synth, rank, world):
    """--impl reference: CPU, rank 0 only."""
    if rank != 0:
        return
    per_step = args.batch                              # the SAME workload as the GPU arm: every step is all `batch` pairs of one frame
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import se3_oracle as O
    sd = synth.make_state_dict(0)
    mean, std = synth.default_mean_std()
    rgb, depth = synth.raw_frame(0)
    poses = synth.raw_poses(per_step, seed=0)
    rgbA, depthA = synth.rendered_views(per_step, poses, seed=0)

    def step():
        dA, dB = [], []
        for i in range(per_step):
            bb = O.compute_bbox(poses[i], synth.CAMERA_K, 200.0, scale=(1000, 1000, 1000))
            rB, zB = O.crop_bbox(rgb, depth, bb, (176, 176))
            (a, b), _ = O.process_data(rgbA[i], depthA[i], poses[i], rB, zB, np.eye(4), mean, std)
            dA.append(torch.from_numpy(a)); dB.append(torch.from_numpy(b))
        out = O.forward(sd, torch.stack(dA), torch.stack(dB))
        return [O.process_predict(poses[i], (out['trans'][i].numpy(), out['rot'][i].numpy())) for i in range(per_step)]

    threads = pick_threads(step)
    for _ in range(max(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'poses': np.stack(last)})
    val = args.steps * per_step / dt
    sample = 'each step = all %d pairs of the workload (per-pair numpy/cv2 crop + normalise, ONE batched torch CPU forward, per-pair pose update); %d steps' % (per_step, args.steps)
    line = {'impl': 'reference', 'metric': 'rgbd_pair_frames_per_sec', 'value': val, 'unit': 'pairs/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': workload_string(args.batch), 'tracks_per_gpu': args.batch, 'total_tracks': args.batch,
                       'precision': 'fp32 CPU (torch oneDNN)',
                       'note': 'one CPU process on rank 0 whatever --gpus says: at N > 1 the GPU arm processes N x %d pairs per step, this arm still %d' % (args.batch, args.batch)},
            'cpu_baseline': {'value': val, 'unit': 'pairs/s', 'cores': threads, 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    pkg = importlib.import_module('iros20-6d-pose-tracking_b200')
    synth = pkg.synth
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, synth, rank, world)
        return
    import torch.distributed as dist
    dist_mod = importlib.import_module('iros20-6d-pose-tracking_b200.dist')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() == 'VERSION':     # keep stdout to the one JSON line
            os.environ['NCCL_DEBUG'] = 'WARN'
        dist.init_process_group('nccl', device_id=dev)
    nb = args.batch

    eng = pkg.Engine(max_batch=nb, device=local_rank)
    sd = synth.make_state_dict(0)
    mean, std = synth.default_mean_std()
    eng.load_state_dict(sd, 0); eng.set_stats(mean, std, 0)
    G = max(1, args.weight_sets)
    for wid in range(1, G):
        eng.load_state_dict(synth.make_state_dict(wid), wid); eng.set_stats(mean, std, wid)

    # ---- synthetic inputs (SURVEY 8d config 2(ii)), distinct sets resident in HBM -------------------------
    # One set per warm-up step (at most MAX_INPUT_SETS): the library keeps one CUDA graph per distinct set of step arguments
    # (the device pointers are part of it), so every set's graph is recorded during warm-up and the timed steps only replay.
    N_INPUT_SETS = min(MAX_INPUT_SETS, max(args.warmup, 3))
    frames, sets = [], []
    for k in range(N_INPUT_SETS):
        seed = 1000 * rank + k
        rgb, depth = synth.raw_frame(seed)
        poses = synth.raw_poses(nb, seed=seed)
        rgbA, depthA = synth.rendered_views(nb, poses, seed=seed)
        host = dict(rgb=torch.from_numpy(rgb).pin_memory(), depth=torch.from_numpy(depth).pin_memory(),
                    poses=torch.from_numpy(poses).pin_memory(), rgbA=torch.from_numpy(rgbA).pin_memory(),
                    depthA=torch.from_numpy(depthA).pin_memory())
        sets.append((host, {k2: v.to(dev) for k2, v in host.items()}))
    ow = torch.full((nb,), 200.0, dtype=torch.float64, device=dev)
    all_wids = np.tile((np.arange(nb) * G // nb).astype(np.int32), world)       # grouped by id within every rank's slice
    tracker = dist_mod.ShardedTracker(eng, all_wids, synth.CAMERA_K, 200.0, TN, RN, rank, world, args.precision)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2

    def step(k, gather=True):
        d = sets[k % N_INPUT_SETS][1]
        return tracker.step(d['rgb'], d['depth'], d['poses'], d['rgbA'], d['depthA'], gather=(gather and world > 1))

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- (1) device-resident throughput: K steps, per-step CUDA events, L2 flushed between steps -----
    # the clock sampler starts BEFORE the warm-up: nothing but a barrier + synchronize lies between the warm-up steps and the timed
    # ones (an idle pause there lets the part drop its clocks, and the first timed steps would pay for the ramp)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start(); time.sleep(0.3)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    for k in range(max(args.warmup, 3)):
        step(k)
    sync_all()
    for k in range(args.steps):
        flush.zero_()                                   # evict the previous step's lines from L2 (untimed)
        ev[k][0].record()
        last = step(k)
        ev[k][1].record()
        launches += eng.last_launch_count()
    # the last step's pose all-gather runs on the side stream: its completion belongs to the timed region too
    tail = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    tail[0].record(); tracker.wait_gather(); tail[1].record()
    sync_all()
    if args.dump_outputs and rank == 0:          # before later steps reuse the tracker's output buffers
        mine, gathered = last
        dump_outputs(args.dump_outputs, {'poses': mine.cpu().numpy()} if gathered is None else
                     {'poses': mine.cpu().numpy(), 'poses_all_ranks': gathered.cpu().numpy()})
    ms_steps = np.array([a.elapsed_time(b) for a, b in ev])
    total_ms = torch.tensor([float(ms_steps.sum()) + tail[0].elapsed_time(tail[1])], device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    ms_per_step = total_ms / args.steps
    value = nb * world * args.steps / (total_ms * 1e-3)

    # ---- (2) roofline of the conv stack: per-kernel events inside the library ------------------------
    pk, pk_src = peaks()

    def conv_stack_profile(prec, nsteps):
        tracker.precision = prec
        eng.set_profiling(True)
        conv_ms, all_ms = [], []
        for k in range(nsteps):
            flush.zero_()
            step(k, gather=False)
            prof = eng.get_profile()
            conv_ms.append(prof[:14].sum()); all_ms.append(prof)
        eng.set_profiling(False)
        tracker.precision = args.precision
        return float(np.mean(conv_ms)), np.mean(np.stack(all_ms), 0)

    def roofline_of(prec, conv_ms, per_slot):
        achieved = nb * FLOP_PER_PAIR / (conv_ms * 1e-3) / 1e12
        if prec == 'tf32':
            peak, executed = (pk['bf16_tflops_sustained'] if (total_ms >= 250.0 and pk.get('bf16_tflops_sustained')) else pk['bf16_tflops']) / 2.0, 1.0
            note = 'tf32 dense = measured bf16 cuBLAS burst (%s: %.1f TF/s) / 2 (kind::tf32 issues at half the bf16 rate; no tf32 line in the file)' % (pk_src, pk['bf16_tflops'])
        elif prec in ('bf16x3', 'bf16'):
            # burst peak for a short timed region, the sustained (power-capped) one when the kernels run inside a long step loop
            sustained = total_ms >= 250.0 and pk.get('bf16_tflops_sustained')
            peak, executed = (pk['bf16_tflops_sustained'] if sustained else pk['bf16_tflops']), (3.0 if prec == 'bf16x3' else 1.0)
            note = 'measured bf16 cuBLAS %s (%s; burst %.1f, sustained %.1f; timed region %.0f ms).  bf16x3 executes 3 bf16 products per algorithmic MAC, so the tensor pipe does executed_mult x the algorithmic work' % (
                'SUSTAINED throughput' if sustained else 'burst', pk_src, pk['bf16_tflops'], pk.get('bf16_tflops_sustained', 0), total_ms)
        else:
            peak, executed, note = 75.0, 1.0, 'nominal fp32 FFMA peak (no tensor cores in this mode)'
        return {'bound': 'tensor', 'kernel': 'conv_resident_kernel x8 + conv_trunk_kernel x1 (17 convs, 9 launches/step)' if prec != 'fp32' else 'conv_direct_kernel',
                'precision': prec, 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
                'executed_mult': executed, 'tensor_pipe_frac': achieved * executed / peak, 'traffic': None,
                'conv_stack_ms': conv_ms, 'peak_note': note,
                'per_kernel_ms': {'conv': [round(float(x), 4) for x in per_slot[:14]], 'maxpool': [round(float(x), 4) for x in per_slot[14:16]],
                                  'head': round(float(per_slot[16]), 4), 'preprocess': round(float(per_slot[17]), 4),
                                  'pose_update': round(float(per_slot[18]), 4)}}

    cms, slots = conv_stack_profile(args.precision, min(args.steps, 20))
    roofline = roofline_of(args.precision, cms, slots)
    tj = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if os.path.exists(tj):            # dram__bytes_read+write per launch from the committed `ncu --set full` capture
        tr = json.load(open(tj))
        roofline['traffic'] = tr['dram_bytes_per_launch']
        roofline['traffic_note'] = 'NOT measured in this run: dram__bytes_read+write per launch from the committed `ncu --set full` capture of this build (%s; %s)' % (tr['kernel'], tr['source'])

    # ---- (2b) the other tensor-core modes on the same workload (secondary numbers) -------------------
    alt = {}
    if not args.no_alt:
        for prec in [q for q in ('tf32', 'bf16x3', 'bf16') if q != args.precision]:
            tracker.precision = prec
            for k in range(N_INPUT_SETS):          # every input set once: its CUDA graph is recorded here, not in the timed steps
                step(k)
            sync_all()
            ev2 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(args.steps, 20))]
            for k in range(len(ev2)):
                flush.zero_(); ev2[k][0].record(); step(k); ev2[k][1].record()
            sync_all()
            tms = torch.tensor([float(sum(a.elapsed_time(b) for a, b in ev2))], device=dev)
            if world > 1:
                dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            cms2, slots2 = conv_stack_profile(prec, min(args.steps, 10))
            r2 = roofline_of(prec, cms2, slots2)
            alt[prec] = {'value': nb * world * len(ev2) / (float(tms.item()) * 1e-3), 'unit': 'pairs/s', 'ms_per_step': float(tms.item()) / len(ev2),
                         'roofline_frac': r2['frac'], 'tensor_pipe_frac': r2['tensor_pipe_frac'], 'conv_stack_ms': cms2,
                         'conv_ms': r2['per_kernel_ms']['conv']}
        tracker.precision = args.precision

    # ---- (2c) the same step with 21 object classes in the batch (SURVEY 8d config 4: G in {1, 21}) -----------------
    g21 = None
    if not args.no_g21 and G == 1 and args.precision != 'fp32':
        G21 = 21
        for wid in range(1, G21):
            eng.load_state_dict(synth.make_state_dict(wid), wid); eng.set_stats(mean, std, wid)
        wids21 = np.tile((np.arange(nb) * G21 // nb).astype(np.int32), world)
        tr21 = dist_mod.ShardedTracker(eng, wids21, synth.CAMERA_K, 200.0, TN, RN, rank, world, args.precision)

        def step21(k):
            d = sets[k % N_INPUT_SETS][1]
            return tr21.step(d['rgb'], d['depth'], d['poses'], d['rgbA'], d['depthA'], gather=(world > 1))
        for k in range(N_INPUT_SETS):          # every input set once: its CUDA graph is recorded here, not in the timed steps
            step21(k)
        sync_all()
        n21 = min(args.steps, 50)
        ev3 = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n21)]
        for k in range(n21):
            flush.zero_(); ev3[k][0].record(); step21(k); ev3[k][1].record()
        tr21.wait_gather()
        sync_all()
        t21 = torch.tensor([float(sum(a.elapsed_time(b) for a, b in ev3))], device=dev)
        if world > 1:
            dist.all_reduce(t21, op=dist.ReduceOp.MAX)
        v21 = nb * world * n21 / (float(t21.item()) * 1e-3)
        g21 = {'weight_sets': G21, 'value': v21, 'unit': 'pairs/s', 'ms_per_step': float(t21.item()) / n21, 'steps': n21, 'ratio_vs_1_set': v21 / value,
               'note': 'track i uses set i*21//%d: 21 checkpoints (54 MB fp32 each) in the same 8 + 1 conv launches; resident-weight layers reload shared memory when the id changes between a CTA\'s consecutive tiles' % nb}

    # ---- (2d) N > 1: the sharded run must equal a single-GPU run of the same tracks, bit for bit (SURVEY 4 tier 3) ----
    shard_parity = None
    if world > 1:
        d0 = sets[0][1]
        mine_out, gathered = tracker.step(d0['rgb'], d0['depth'], d0['poses'], d0['rgbA'], d0['depthA'], gather=True)
        tracker.wait_gather()
        torch.cuda.synchronize(dev)
        if rank == 0:
            worst, checked = 0.0, 0
            g_np = gathered.cpu().numpy()
            for r in range(world):                      # rank r's input set 0 is seeded 1000*r: regenerate it here and run it on THIS GPU alone
                rgb_r, depth_r = synth.raw_frame(1000 * r)
                poses_r = synth.raw_poses(nb, seed=1000 * r)
                rgbA_r, depthA_r = synth.rendered_views(nb, poses_r, seed=1000 * r)
                t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
                solo, _, _ = eng.track_batch(t(rgb_r), t(depth_r), synth.CAMERA_K, t(poses_r), ow, t(rgbA_r), t(depthA_r), TN, RN,
                                             weight_ids_host=tracker.weight_ids[tracker.shards[r]], precision=args.precision)
                worst = max(worst, float(np.abs(solo.cpu().numpy() - g_np[tracker.shards[r]]).max())); checked += nb
            shard_parity = {'sharded_vs_single_gpu_max_abs_pose_diff': worst, 'tracks': checked, 'bit_identical': worst == 0.0,
                            'note': 'every rank\'s gathered poses vs the same tracks run on rank 0 alone'}

    # ---- (3) end to end through the public API with pinned HOST buffers -----------------------------
    info = {'resolution': 176, 'boundingbox': 10, 'object_width': 200.0,
            'camera': {'focalX': synth.CAMERA_K[0, 0], 'focalY': synth.CAMERA_K[1, 1], 'centerX': synth.CAMERA_K[0, 2],
                       'centerY': synth.CAMERA_K[1, 2], 'height': 480, 'width': 640}}
    trk = pkg.Tracker(info, mean, std, {'state_dict': sd}, model_path=None, engine=eng, precision=args.precision)
    pinned_out = torch.empty(nb, 4, 4, dtype=torch.float64).pin_memory()

    def e2e_step(k):
        # pinned HOST tensors in (uploads pipelined on the Tracker's copy stream), pinned host poses out
        h = sets[k % N_INPUT_SETS][0]
        out = trk.on_track_batch(h['poses'], h['rgb'], h['depth'], h['rgbA'], h['depthA'])
        pinned_out.copy_(out, non_blocking=True)       # this rank's result back to the host
        if world > 1:                                   # exchange step: every rank receives all poses (side stream, see dist.ShardedTracker)
            e2e_gather(out)
        return out

    comm_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    gather_state = {'pending': [], 'last': None}

    def e2e_gather(out):
        cur = torch.cuda.current_stream(dev)
        while len(gather_state['pending']) >= 2:         # at most two gathers in flight (as dist.ShardedTracker): no per-step lock step between ranks
            cur.wait_event(gather_state['pending'].pop(0))
        ready = torch.cuda.Event(); ready.record(cur)
        comm_stream.wait_event(ready)
        with torch.cuda.stream(comm_stream):
            gather_state['last'] = tracker.plan.gather(out)
            done = torch.cuda.Event(); done.record(comm_stream)
            gather_state['pending'].append(done)
        out.record_stream(comm_stream)

    for k in range(3):
        e2e_step(k)
    sync_all()
    e2e_steps = args.steps
    t0 = time.perf_counter()
    for k in range(e2e_steps):
        e2e_step(k)
    torch.cuda.synchronize(dev)
    e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev)
    if world > 1:
        dist.barrier(); dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    h0 = sets[0][0]
    h2d = sum(h0[k2].numel() * h0[k2].element_size() for k2 in ('rgb', 'depth', 'poses', 'rgbA', 'depthA'))
    e2e = {'value': nb * world * e2e_steps / (float(e2e_ms.item()) * 1e-3), 'unit': 'pairs/s',
           'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(pinned_out.numel() * 8),
           'api': 'Tracker.on_track_batch (pinned host tensors in, pinned host poses out; wall clock over the K calls incl. all copies; uploads of call k overlap the kernels of call k-1 on a side stream)'}

    # the clocks belong to the two timed regions above; the nvidia-smi polling thread would only disturb the latency legs below
    clocks = None
    if sampler:
        sampler.stop_flag = True; time.sleep(0.15)
        clocks = sampler.summary()

    # ---- (3b) the same step with input A RENDERED on the device (SURVEY 8f row 2) instead of taken from HBM ----------
    render = None
    if rank == 0 and world == 1 and not args.no_render:
        mesh = synth.mesh(5, seed=0)                       # 20,480 faces / 10,242 vertices
        eng.set_mesh(mesh, 0)
        rgbA_buf = torch.empty((nb, 176, 176, 3), dtype=torch.uint8, device=dev)
        depA_buf = torch.empty((nb, 176, 176), dtype=torch.uint16, device=dev)

        def render_step(k):
            d = sets[k % N_INPUT_SETS][1]
            eng.render(synth.CAMERA_K, d['poses'], ow, None, rgbA_buf, depA_buf)
            return tracker.step(d['rgb'], d['depth'], d['poses'], rgbA_buf, depA_buf, gather=False)
        for k in range(N_INPUT_SETS):          # every input set once: its CUDA graph is recorded here, not in the timed steps
            render_step(k)
        sync_all()
        rsteps = min(args.steps, 20)
        rev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(rsteps)]
        for k in range(rsteps):
            flush.zero_()
            rev[k][0].record(); render_step(k); rev[k][1].record()
        sync_all()
        rms = float(np.mean([a.elapsed_time(b) for a, b in rev]))
        eng.set_profiling(True)
        acc = []
        for k in range(5):
            d = sets[k % N_INPUT_SETS][1]
            eng.render(synth.CAMERA_K, d['poses'], ow, None, rgbA_buf, depA_buf); acc.append(eng.get_profile()[20])
        eng.set_profiling(False)
        kms = float(np.mean(acc))
        render = {'mesh_faces': int(len(mesh['faces'])), 'mesh_vertices': int(len(mesh['pos'])), 'render_kernel_ms': kms,
                  'renders_per_s': nb / (kms * 1e-3), 'step_with_render_ms': rms, 'pairs_per_s_with_render': nb / (rms * 1e-3),
                  'note': 'render_kernel (csrc/render.cu): %d tracks x 176x176, float64 visibility + shading, one launch; replaces the reference\'s two OpenGL renders + glReadPixels per track and frame' % nb}

    # ---- (3c) one object, one frame at a time, numpy in / numpy out: the reference's own calling pattern (predict.py:416) ----
    single = None
    if rank == 0 and world == 1:
        h = sets[0][0]
        f_rgb, f_depth = np.array(h['rgb'].numpy()), np.array(h['depth'].numpy())          # copies: ordinary pageable arrays, as a caller's would be
        p1, a1, d1 = np.array(h['poses'][0].numpy()), np.array(h['rgbA'][0].numpy()), np.array(h['depthA'][0].numpy())
        for _ in range(20):
            trk.on_track(p1, f_rgb, f_depth, rgbA=a1, depthA=d1)
        t0 = time.perf_counter(); reps = 200
        for _ in range(reps):
            trk.on_track(p1, f_rgb, f_depth, rgbA=a1, depthA=d1)
        single = {'ms_per_frame': (time.perf_counter() - t0) / reps * 1e3, 'frames_per_s': reps / (time.perf_counter() - t0),
                  'note': 'Tracker.on_track(prev_pose, rgb, depth) for ONE object: synchronous, pageable numpy frame in (1.5 MB), numpy pose out, wall clock; one se3tn_track_host call per frame'}

    # ---- (4) CPU baseline (rank 0, N=1 only) ---------------------------------------------------------
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, sample, (c_rgb, c_depth, c_poses, c_rgbA, c_depthA, c_ref) = cpu_on_track_rate(synth, args.cpu_seconds)
        cpu = {'value': v, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port', 'sample': sample}
        # the CPU sample doubles as a parity spot check of every tensor-core mode on this workload's generators
        parity = {}
        for prec in ('bf16x3', 'tf32', 'bf16'):
            trk.precision = prec
            got = trk.on_track_batch(c_poses, c_rgb, c_depth, c_rgbA, c_depthA)
            parity[prec] = {'max_abs_pose_err': float(np.abs(got - c_ref).max()), 'pairs': int(len(c_ref))}
        trk.precision = args.precision
        parity['note'] = 'max |pose - CPU oracle pose| over the cpu_baseline sample; the 6-vector gate (rtol 1e-3, atol 1e-4) propagates to <= 1e-4 here'

    if rank == 0:
        line = {'metric': 'rgbd_pair_frames_per_sec', 'value': value, 'unit': 'pairs/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': max(args.warmup, 3), 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': {'tf32': 'tf32', 'bf16x3': 'bf16x3 (bf16 hi/lo split operands, 3 products/MAC, fp32 accumulate)', 'bf16': 'bf16', 'fp32': 'f32'}[args.precision], 'data': 'synthetic',
                'config': {'workload': workload_string(nb),
                           'tracks_per_gpu': nb, 'total_tracks': nb * world, 'precision': args.precision,
                           'parallelism': 'tracks sharded, %d/GPU, NCCL all-gather of poses per step (side stream, overlapped with the next step)' % nb if world > 1 else 'single GPU',
                           'l2': 'flushed between timed steps (256 MiB memset, untimed); %d rotating input sets; per-step CUDA events, max over ranks' % N_INPUT_SETS,
                           'weights': 'random-init (seeded), %d weight set(s)%s' % (G, '' if G == 1 else ' (one per object class; all classes batched into the same conv launches)')},
                'gpu_launches': int(launches), 'launches_per_step': int(launches // max(args.steps, 1)),
                'graph_launches_per_step': 1 if eng.last_step_was_graph() else None,
                'roofline': roofline, 'alt_precisions': alt, 'weight_sets_21': g21, 'parity': parity if world == 1 else shard_parity, 'cpu_baseline': cpu, 'e2e': e2e, 'render': render, 'single_track': single, 'clocks': clocks,
                'ms_per_step_min': float(ms_steps.min()), 'ms_per_step_median': float(np.median(ms_steps))}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    eng.close()


if __name__ == '__main__':
    sys.dont_write_bytecode = True          # the tree may be read-only: a benchmark run leaves it exactly as it found it
    main()
