#!/usr/bin/env python
"""Benchmark of the THA4 poser hot path on B200 (contract: see the task's bench.py section).

    python bench.py --gpus N --steps K --warmup W [--impl reference|torch_cuda] [--workload ...] [--no-extras] [--dump-outputs DIR]

A "step" is one poser forward over one batch of synthetic input.  The headline workload is BASELINE.json configs[1]:
the full five-network poser (mode_07), batch 1 per GPU, the lambda_00 character image, one random pose per step,
eyebrow cache hot (the image does not change between frames, as in the reference's GUI).  Metric: 512x512 RGBA
frames/sec.  Rank 0 prints ONE JSON line:

  value        device-timed throughput with image and poses already resident in HBM;
  e2e          the same through the public API with pinned HOST buffers: H2D of image + pose and D2H of the posed
               frame inside the timed region, every step;
  roofline     the dominant kernel class (implicit-GEMM convolution: tensor bound), measured in a separate profiled
               pass with CUDA events inside the library; roofline_tail is the fused grid_sample + decoder kernel
               (HBM bound), the kernel BASELINE.json's metric names;
  cpu_baseline the CPU oracle (a PyTorch-CPU port of the reference path, oracle/) on this box's host cores.

and -- so that every BASELINE config is on the driver's record -- sub-objects measured in the same run:

  torch_cuda_eager  configs[1] executed by PyTorch-CUDA eager (the oracle's ops on the GPU = what the reference's own
                    CUDA path dispatches): the denominator of BASELINE's ">= 30x" target;
  student_b64       configs[2]: distilled student (mode_14), batch 64 per GPU, shipped lambda_00 weights;
  pose_sweep_512    configs[3]: 512 poses of ONE image, contiguous shards of 512/N per GPU, STRONG scaling, no collective;
  distill           configs[4]: body-morpher distillation steps (teacher fwd + student fwd/bwd + one NCCL all-reduce of
                    the 1.33 MB flat gradient + Adam), per-GPU batch 1, 1000 steps at N = 8, with the final weights
                    compared against a single-process run of the same global batch.
`--impl reference` times the CPU port alone, as the reference arm.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

WORKLOADS = {
    'teacher_b1': dict(mode='mode_07', batch=1, desc='full poser mode_07 forward, batch=1, lambda_00 image, random poses, eyebrow cache hot'),
    'teacher_b1_nocache': dict(mode='mode_07', batch=1, nocache=True, desc='full poser mode_07 forward, batch=1, the image changes every frame (eyebrow-decomposer cache always misses: 645.9 GFLOP/frame)'),
    'pose_sweep_512': dict(mode='mode_07', total=512, desc='BASELINE configs[3]: 512-pose sweep of the lambda_00 image, contiguous shards of 512/N frames per GPU (micro-batches of 32), no collective'),
    'teacher_b16': dict(mode='mode_07', batch=16, desc='full poser mode_07 forward, batch=16 pose sweep on the lambda_00 image'),
    'student_b64': dict(mode='mode_14', batch=64, desc='distilled student mode_14 forward, batch=64, lambda_00 weights, fp16 tensor-core products'),
    'distill_b1': dict(mode='distill', batch=1, desc='body-morpher distill step: teacher mode_07 fwd + student fwd/bwd + gradient all-reduce + Adam, per-GPU batch 1 (reference-faithful: total batch <= 8)'),
}
TEACHER_GFLOP_PER_FRAME = 625.9   # cache-hot (SURVEY.md section 8a)
DISTILL_W, DISTILL_LR = [0.0, 1.0, 1.0, 0.0], 1e-4        # phase 1 of the body schedule: warp + grid-change terms (distiller_config.py:178-186)
L2_NOTE = 'packed weights (657 MB teacher) and activations exceed the 126 MB L2; no explicit flush'


def config_for(workload, batch_per_gpu, world):
    """The `config` object of a bench line -- built by ONE function for both arms, so the driver sees identical configs."""
    wl = WORKLOADS[workload]
    distill = wl['mode'] == 'distill'
    par = ('data parallel, one NCCL all-reduce of the 1.33 MB flat gradient per step (dp%d)' if distill
           else 'frames sharded, no collective (dp%d)') % world
    return {'workload': wl['desc'], 'batch_per_gpu': batch_per_gpu, 'parallelism': par, 'l2': L2_NOTE}


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p['hbm_gbs'], tflops=p['bf16_tflops'], tflops_sustained=p.get('bf16_tflops_sustained'), source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, tflops=1590.0, tflops_sustained=1400.0, source='fallback (B200_PROFILING.md)')


def load_ncu_traffic():
    """DRAM bytes per launch of the named kernels from the committed `ncu --set full` captures (profiles/ncu_traffic.json)."""
    path = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    return json.load(open(path)) if os.path.exists(path) else {}


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        while not self._halt.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(',')
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith('active'):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        return dict(sm_mhz=statistics.median(self.samples) if self.samples else None, sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(self.samples))


def load_image():
    from tha4_b200 import image_util, synthetic
    png = os.path.join(ROOT, 'tests', 'golden', 'data', 'lambda_00.png')
    return image_util.load_poser_image(png) if os.path.exists(png) else synthetic.synthetic_image(0, 1)[0]


def load_state_dicts(mode):
    from tha4_b200 import synthetic
    if mode == 'mode_07':
        return synthetic.teacher_state_dicts(0), 'seeded teacher weights of the reference architecture (trained-like conditioning, tha4_b200/synthetic.py)'
    data = os.path.join(ROOT, 'tests', 'golden', 'data')
    paths = {k: os.path.join(data, 'lambda_00_%s.pt' % k) for k in ('face_morpher', 'body_morpher')}
    if all(os.path.exists(p) for p in paths.values()):
        return {k: torch.load(p, map_location='cpu') for k, p in paths.items()}, 'shipped lambda_00 student weights'
    return synthetic.student_state_dicts(0), 'random-init (seeded) student weights'


def cpu_threads():
    """Host threads for the CPU arm.  PyTorch-CPU convs on these 128-core boxes get *slower* past a few dozen threads
    (measured: 128 threads are 40x slower than 8 on the teacher), so the arm uses min(cores, 32) and says so."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get('THA4_CPU_THREADS', '32'))))


def cpu_port_fps(mode, sds, image, poses, batch, frames_budget, threads, seconds_budget=20.0):
    """Times the CPU oracle (PyTorch-CPU port of the reference path).  Returns (fps, frames, seconds)."""
    from oracle import tha4_oracle
    torch.set_num_threads(threads)
    fn = getattr(tha4_oracle, mode + '_outputs')
    with torch.no_grad():
        dec = None
        if mode == 'mode_07':   # eyebrow cache hot, as in the GPU arm
            dec = tha4_oracle.eyebrow_decomposer(sds['eyebrow_decomposer'], image.unsqueeze(0)[:, :, 64:192, 192:320])
        b = min(batch, 2)
        img_b = image.unsqueeze(0).expand(b, -1, -1, -1).contiguous()
        kw = dict(cached_decomposer_output=[t.expand(b, -1, -1, -1) for t in dec]) if dec is not None else {}
        fn(sds, img_b, poses[:b], **kw)            # warm-up
        t0 = time.perf_counter()
        done = 0
        while done < frames_budget and (done == 0 or time.perf_counter() - t0 < seconds_budget):
            fn(sds, img_b, poses[done % 8:done % 8 + b] if poses.shape[0] >= 8 + b else poses[:b], **kw)
            done += b
        dt = time.perf_counter() - t0
    return done / dt, done, dt


def run_reference(args, rank, world):
    """Reference arm: the reference's own CPU implementation of the path (its PyTorch-CPU port in oracle/)."""
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    from tha4_b200 import synthetic
    sds, _ = load_state_dicts(wl['mode'])
    image = load_image()
    poses = synthetic.random_poses(64, seed=1234)
    threads = cpu_threads()
    per_step_frames = 1 if wl['mode'] == 'mode_07' else 2
    from oracle import tha4_oracle
    torch.set_num_threads(threads)
    fn = getattr(tha4_oracle, wl['mode'] + '_outputs')
    b = per_step_frames
    img_b = image.unsqueeze(0).expand(b, -1, -1, -1).contiguous()
    kw = {}
    times = []
    with torch.no_grad():
        if wl['mode'] == 'mode_07':     # eyebrow cache hot, as in the GPU arm (mode_07.py:56-68)
            dec = tha4_oracle.eyebrow_decomposer(sds['eyebrow_decomposer'], img_b[:, :, 64:192, 192:320])
            kw = dict(cached_decomposer_output=dec)
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            fn(sds, img_b, poses[(i * b) % 32:(i * b) % 32 + b], **kw)
            if i >= args.warmup:
                times.append((time.perf_counter() - t0) / b)
    spf = sum(times) / len(times)
    B = wl.get('batch', max(1, wl.get('total', 1) // world))
    line = {
        'impl': 'reference', 'metric': '512x512 RGBA frames/sec', 'value': 1.0 / spf, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 * spf * B, 'higher_is_better': True,
        'scaling': 'strong' if 'total' in wl else 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': config_for(args.workload, B, world),
        'cpu_baseline': {'value': 1.0 / spf, 'unit': 'frames/s', 'cores': threads, 'kind': 'port',
                         'sample': '%d timed steps of %d frame(s) each of the same workload (PyTorch-CPU port of the reference path, '
                                   '%d of %d host threads)' % (len(times), per_step_frames, threads, os.cpu_count() or 1)},
        'e2e': {'value': 1.0 / spf, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


def torch_cuda_eager_fps(mode, sds, image, poses, B, warmup, steps, dev):
    """The oracle's PyTorch ops executed on the GPU = what the reference's own PyTorch-CUDA eager path does on this box
    (same ops, cuDNN/cuBLAS kernels, TF32 convs allowed as by torch's default).  Returns (fps, ms_per_step)."""
    from oracle import tha4_oracle
    sds = {k: {kk: vv.to(dev) for kk, vv in v.items()} for k, v in sds.items()}
    img = image.to(dev).unsqueeze(0).expand(B, -1, -1, -1).contiguous()
    poses = poses.to(dev)
    fn = getattr(tha4_oracle, mode + '_outputs')
    orig_grid, orig_t0 = tha4_oracle.base_grid, tha4_oracle._timestep_embedding_zero
    tha4_oracle.base_grid = lambda n, h, w, dtype=torch.float32: orig_grid(n, h, w, dtype).to(dev)
    tha4_oracle._timestep_embedding_zero = lambda n, c: orig_t0(n, c).to(dev)
    try:
        kw = {}
        with torch.no_grad():
            if mode == 'mode_07':
                kw = dict(cached_decomposer_output=tha4_oracle.eyebrow_decomposer(sds['eyebrow_decomposer'], img[:, :, 64:192, 192:320]))
            for i in range(warmup):
                fn(sds, img, poses[(i * B) % 32:(i * B) % 32 + B], **kw)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                fn(sds, img, poses[((warmup + i) * B) % 32:((warmup + i) * B) % 32 + B], **kw)
            e1.record()
            torch.cuda.synchronize()
    finally:
        tha4_oracle.base_grid, tha4_oracle._timestep_embedding_zero = orig_grid, orig_t0
    ms = e0.elapsed_time(e1)
    return steps * B / (ms / 1000.0), ms / steps


def run_torch_cuda(args, rank):
    if rank != 0:
        return
    from tha4_b200 import synthetic
    wl = WORKLOADS[args.workload]
    mode = 'mode_14' if wl['mode'] == 'mode_14' else 'mode_07'
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', '0')))
    sds, _ = load_state_dicts(mode)
    B = wl.get('batch', 16)
    fps, ms = torch_cuda_eager_fps(mode, sds, load_image(), synthetic.random_poses(64 + B, seed=1234), B, args.warmup, args.steps, dev)
    emit({'impl': 'torch_cuda_eager', 'metric': '512x512 RGBA frames/sec', 'value': fps, 'unit': 'frames/s', 'ms_per_step': ms,
          'steps': args.steps, 'warmup': args.warmup, 'config': {'workload': wl['desc']},
          'note': 'PyTorch eager on the same GPU running the oracle port (the ops the reference dispatches); context only'})


_REAL_STDOUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries (NCCL prints its version banner there) share fd 1, so
    everything else is sent to stderr and the JSON line is written to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


DUMP_BUDGET_BYTES = 60 << 20          # with the .npy headers, under 64 MB


def dump_outputs(out_dir, named):
    """Writes each (name, tensor) as <out_dir>/<name>.npy in float32.  When the tensors hold more than DUMP_BUDGET_BYTES,
    each one is written flattened and cut to the same share of its elements, taken at positions drawn from a generator
    seeded with the tensor's index, so that two runs with the same arguments write element-for-element comparable files."""
    import numpy
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() for _, t in named)
    keep = min(1.0, DUMP_BUDGET_BYTES / 4 / max(1, total))
    for i, (name, t) in enumerate(named):
        t = t.detach().float()
        if keep < 1.0:
            flat = t.reshape(-1)
            idx = torch.randint(flat.numel(), (max(1, int(flat.numel() * keep)),), generator=torch.Generator().manual_seed(i))
            t = flat[idx.sort().values.to(flat.device)]
        numpy.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy())


def emit(line: dict):
    data = (json.dumps(line) + '\n').encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


class Timer:
    """K steps bracketed by barrier + synchronize on both sides, CUDA events on the launching stream, max over ranks."""

    def __init__(self, world, device):
        self.world, self.device = world, device

    def barrier(self):
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run(self, step, warmup, steps):
        for i in range(warmup):
            step(i)
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(warmup + i)
        e1.record()
        self.barrier()
        return e0.elapsed_time(e1)

    def max_over_ranks(self, *values):
        if self.world == 1:
            return [float(v) for v in values]
        t = torch.tensor([float(v) for v in values], device=self.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]


def profile_pass(ctx, run_steps, steps, rank, all_ranks=False):
    """Per-kernel-class CUDA-event times / work counters of `steps` steps (library option "profile")."""
    prof = {}
    if rank == 0 or all_ranks:
        if rank == 0:
            ctx.set_option('profile', 2)
        run_steps()
        torch.cuda.synchronize()
        if rank == 0:
            for cat in ('conv', 'norm', 'tail', 'attn', 'siren'):
                prof[cat] = {w: ctx.counter('prof_%s_%s' % (w, cat)) for w in ('us', 'launches', 'flops', 'bytes')}
            ctx.set_option('profile', 0)
    return prof


def roofline_objects(prof, steps, peaks, traffic):
    out = {}
    if prof.get('conv', {}).get('us', 0) > 0:
        c = prof['conv']
        ach = c['flops'] / (c['us'] * 1e-6) / 1e12
        out['roofline'] = {'kernel': 'conv_tc_kernel (implicit-GEMM conv: TMA + tcgen05.mma kind::f16/tf32, TMEM accumulator; all conv launches of the step)', 'bound': 'tensor', 'achieved': ach,
                           'peak': peaks['tflops'], 'unit': 'TFLOP/s', 'frac': ach / peaks['tflops'], 'traffic': traffic.get('conv', {}).get('dram_bytes_per_launch'),
                           'peak_source': peaks['source'] + ' dense bf16 burst (= the f16 operand rate; kind::tf32 layers peak at half of it)',
                           'avg_launch_us': c['us'] / max(1, c['launches']), 'launches_per_step': c['launches'] / steps,
                           'share_of_profiled_kernel_time': c['us'] / max(1.0, sum(v['us'] for v in prof.values()))}
    if prof.get('tail', {}).get('us', 0) > 0:
        t = prof['tail']
        ach = t['bytes'] / (t['us'] * 1e-6) / 1e9
        out['roofline_tail'] = {'kernel': 'fused decoder tail (head conv + grid_sample + blend), all teacher sites of the step', 'bound': 'hbm',
                                'achieved': ach, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': ach / peaks['hbm_gbs'],
                                'traffic': traffic.get('tail', {}).get('dram_bytes_per_launch'), 'traffic_source': traffic.get('tail', {}).get('source'),
                                'peak_source': peaks['source'], 'avg_launch_us': t['us'] / max(1, t['launches']),
                                'algorithmic_bytes_per_launch': t['bytes'] / max(1, t['launches'])}
    out['kernel_time_us_per_step'] = {k: v['us'] / steps for k, v in prof.items() if v['us'] > 0}
    return out


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='tha4_b200', choices=['tha4_b200', 'reference', 'torch_cuda'])
    ap.add_argument('--workload', default='teacher_b1', choices=sorted(WORKLOADS))
    ap.add_argument('--strict', type=int, default=0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip the student / pose-sweep / distill / torch-eager sub-objects')
    ap.add_argument('--distill-steps', type=int, default=0, help='0: 1000 at N = 8 (BASELINE configs[4]), 200 otherwise')
    ap.add_argument('--option', action='append', default=[], help='library option name=value (developer A/B runs)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write what the last one returned (the poser '
                    'outputs, or the student weights of a distill step) as DIR/<name>.npy, float32, at most 64 MB in all')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'tha4_b200':
        ap.error('--dump-outputs writes the outputs of the tha4_b200 path only')

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if args.impl == 'torch_cuda':
        run_torch_cuda(args, rank)
        return

    wl = WORKLOADS[args.workload]
    B = wl['batch'] if 'batch' in wl else max(1, wl['total'] // world)     # fixed total: strong scaling
    strong = 'total' in wl
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)
    timer = Timer(world, device)
    peaks, traffic = load_peaks(), load_ncu_traffic()

    from tha4_b200 import synthetic
    from tha4_b200.poser.modes import mode_07, mode_14
    distill = wl['mode'] == 'distill'
    student_mode = wl['mode'] == 'mode_14'
    tsds, tdesc = (None, '') if student_mode else load_state_dicts('mode_07')
    ssds, sdesc = load_state_dicts('mode_14')
    weights_desc = sdesc if student_mode else tdesc + ('; student: ' + sdesc if distill else '')
    image = load_image()
    nposes = (args.warmup + args.steps) * B
    poses = synthetic.random_poses(nposes, seed=1234 + rank)
    poser = mode_14.create_poser(device, state_dicts=ssds) if student_mode else mode_07.create_poser(device, state_dicts=tsds)
    poser.get_modules()
    ctx = poser.get_context()
    ctx.set_option('strict', args.strict)
    for kv in args.option:
        k, v = kv.split('=')
        ctx.set_option(k, int(v))
    if not student_mode:
        poser.protocol.trust_image_identity = True      # this process owns the image tensors it passes (see mode_07.py)
    distiller = None
    if distill:
        from tha4_b200.distill import BodyMorpherDistiller
        distiller = BodyMorpherDistiller(poser, mode_14.load_body_morpher(None, ssds['body_morpher']))

    img_dev = image.to(device).unsqueeze(0).expand(B, -1, -1, -1)
    img_dev = img_dev.contiguous() if (B == 1 or student_mode or distill) else img_dev     # B > 1 teacher: ONE stored image, batch stride 0
    poses_dev = poses.to(device)
    img_alt = None
    if wl.get('nocache'):          # a second image that differs in one pixel value: the cache comparison fails every frame
        img_alt = img_dev.clone()
        img_alt[:, 0, 0, 0] += 1.0 / 512.0

    def step_resident(i):
        if distiller is not None:
            return distiller.train_step(img_dev, poses_dev[i * B:(i + 1) * B], DISTILL_W, DISTILL_LR, want_losses=False)
        return poser.get_posing_outputs(img_alt if (img_alt is not None and (i & 1)) else img_dev, poses_dev[i * B:(i + 1) * B])

    extras = {}
    with torch.no_grad():
        # ---------------- device-resident timing ----------------
        for i in range(args.warmup):
            step_resident(i)
        timer.barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        l0 = ctx.counter('kernel_launches')
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps - 1):
            step_resident(args.warmup + i)
        # only the final step's outputs are kept (for --dump-outputs): holding a step's outputs while the next one runs
        # would move that step's output buffers, and the library replays a frame as a CUDA graph only when they repeat
        last = step_resident(args.warmup + args.steps - 1)
        e1.record()
        timer.barrier()
        ms = e0.elapsed_time(e1)
        launches = ctx.counter('kernel_launches') - l0
        clocks = sampler.stop()
        if args.dump_outputs and rank == 0:      # before any later pass reuses the output buffers
            named = [('student_weights', distiller.flat)] if distiller is not None else \
                [('%s_output_%02d' % (wl['mode'], k), t) for k, t in enumerate(last)]
            dump_outputs(args.dump_outputs, named)
        del last

        # ---------------- end to end through the public API with host buffers ----------------
        img_host = image.unsqueeze(0).contiguous().pin_memory()             # ONE image: a sweep poses it B times
        poses_host = poses.pin_memory()
        out_host = torch.empty((B, 512, 512, 4), dtype=torch.uint8).pin_memory()      # the displayable frame the apps consume
        out_host_f32 = torch.empty((B, 4, 512, 512), dtype=torch.float32).pin_memory()
        img_in = torch.empty((1, 4, 512, 512), device=device)
        img_in2 = torch.empty_like(img_in) if img_alt is not None else None
        pose_in = torch.empty((B, 45), device=device)
        dense = student_mode or distill                                     # these paths take a dense [B,4,512,512] batch
        img_dense = torch.empty((B, 4, 512, 512), device=device) if (dense and B > 1) else None

        def step_e2e(i):
            img_cur = img_in
            if img_alt is not None and (i & 1):      # a different tensor object with different content: the cache must miss
                img_cur = img_in2
                img_cur.copy_(img_host, non_blocking=True)
                img_cur[:, 0, 0, 0] += 1.0 / 512.0
            else:
                img_cur.copy_(img_host, non_blocking=True)
            pose_in.copy_(poses_host[i * B:(i + 1) * B], non_blocking=True)
            if img_dense is not None:
                img_dense.copy_(img_cur.expand(B, -1, -1, -1))
                batch_img = img_dense
            else:
                batch_img = img_cur.expand(B, -1, -1, -1) if B > 1 else img_cur
            if distiller is not None:        # result of a training step = its loss terms, read back on the host
                distiller.train_step(batch_img, pose_in, DISTILL_W, DISTILL_LR, want_losses=True)
                return
            if fp32_frames[0]:
                out_host_f32.copy_(poser.pose(batch_img, pose_in), non_blocking=True)
            else:      # what every app does with the frame (puppeteer.py:325-349), here on the GPU: 1 MB instead of 4 MB over PCIe
                out_host.copy_(poser.pose_to_srgb8(batch_img, pose_in), non_blocking=True)
            torch.cuda.current_stream().synchronize()      # the caller consumes the frame on the host

        fp32_frames = [False]
        ms_e2e = timer.run(step_e2e, args.warmup, args.steps)
        ms_e2e_f32 = None
        if distiller is None:
            fp32_frames[0] = True
            ms_e2e_f32 = timer.run(step_e2e, 3, args.steps)

        # ---------------- profiled pass for the roofline objects ----------------
        prof = profile_pass(ctx, lambda: [step_resident(args.warmup + i) for i in range(args.steps)], args.steps, rank, all_ranks=distiller is not None)

        # ---------------- the other BASELINE configs, same run ----------------
        if args.workload == 'teacher_b1' and not args.no_extras and not args.strict:
            extras = run_extras(args, timer, rank, world, device, poser, ctx, tsds, ssds, image, peaks, traffic)

    ms, ms_e2e = timer.max_over_ranks(ms, ms_e2e)
    if ms_e2e_f32 is not None:
        (ms_e2e_f32,) = timer.max_over_ranks(ms_e2e_f32)
    if world > 1:
        cl = torch.tensor([float(launches)], device=device)
        dist.all_reduce(cl)
        launches = int(cl[0])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    frames = args.steps * B * world
    value = frames / (ms / 1000.0)
    e2e_value = frames / (ms_e2e / 1000.0)
    line = {
        'metric': 'distillation examples/sec' if distill else '512x512 RGBA frames/sec', 'value': value,
        'unit': 'examples/s' if distill else 'frames/s', 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'strong' if strong else 'weak', 'vs_baseline': None,
        'dtype': 'f16/tf32 operands (10-bit mantissa), f32 accumulate, f32 storage outside conv operands' if wl['mode'] in ('mode_07', 'distill') and not args.strict else
                 ('f32 (3xTF32)' if wl['mode'] == 'mode_07' else 'f16 products, f32 accumulate'),
        'data': 'synthetic poses; ' + weights_desc + '; lambda_00.png character image',
        'config': config_for(args.workload, B, world),
        'e2e': {'value': e2e_value, 'unit': 'examples/s' if distill else 'frames/s', 'h2d_bytes_per_step': 4 * 512 * 512 * 4 + B * 45 * 4,
                'd2h_bytes_per_step': 32 if distill else B * 4 * 512 * 512, 'ms_per_step': ms_e2e / args.steps,
                'note': 'every step: one pinned-host image + B poses copied in, poser.pose_to_srgb8() (pose + the display conversion of '
                        'puppeteer.py:325-349 on the GPU), B uint8 RGBA frames copied out and synchronised'},
        'gpu_launches': launches,
        'clocks': clocks,
    }
    if ms_e2e_f32 is not None:
        line['e2e_fp32_frame'] = {'value': frames / (ms_e2e_f32 / 1000.0), 'unit': 'frames/s', 'd2h_bytes_per_step': B * 4 * 512 * 512 * 4,
                                  'ms_per_step': ms_e2e_f32 / args.steps, 'note': 'same loop returning the raw fp32 frame of poser.pose()'}
    if wl['mode'] == 'mode_07':
        line['teacher_tflops_effective'] = (645.9 if wl.get('nocache') else TEACHER_GFLOP_PER_FRAME) * value / world / 1000.0
    line.update(roofline_objects(prof, args.steps, peaks, traffic))
    if prof.get('siren', {}).get('us', 0) > 0:
        line['siren_us_per_step'] = prof['siren']['us'] / args.steps
    if 'roofline' not in line:
        s = prof.get('siren', {})
        line['roofline'] = {'kernel': 'siren fused MLP kernels', 'bound': 'tensor', 'achieved': None, 'peak': peaks['tflops'],
                            'unit': 'TFLOP/s', 'frac': None, 'traffic': None, 'us_per_step': s.get('us', 0) / max(1, args.steps)}
        if s.get('us', 0) > 0:
            ach = 37.89e9 * B * args.steps / (s['us'] * 1e-6) / 1e12
            line['roofline'].update(achieved=ach, frac=ach / peaks['tflops'])
    line['cuda_graphs'] = {'replays': ctx.counter('graph_replays'), 'captures': ctx.counter('graph_captures'), 'failures': ctx.counter('graph_failures'),
                           'note': 'single-chunk teacher forwards whose buffer addresses repeat are replayed as one captured graph (zero-copy)'}
    line.update(extras)
    if 'value' in extras.get('torch_cuda_eager', {}):
        line['torch_cuda_eager_fps'] = extras['torch_cuda_eager']['value']
        line['speedup_vs_torch_cuda_eager'] = value / world / extras['torch_cuda_eager']['value']

    if not args.no_cpu_baseline and world == 1 and not distill:
        threads = cpu_threads()
        budget = 6 if wl['mode'] == 'mode_07' else 12
        fps, nfr, dt = cpu_port_fps(wl['mode'], ssds if student_mode else tsds, image, poses, B, budget, threads)
        line['cpu_baseline'] = {'value': fps, 'unit': 'frames/s', 'cores': threads, 'kind': 'port',
                                'sample': '%d frames of the same workload in %.1f s (PyTorch-CPU port of the reference path in oracle/, '
                                          '%d of %d host threads; /root/reference itself is pure Python and does not exist on the GPU box)' % (nfr, dt, threads, os.cpu_count() or 1)}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_extras(args, timer, rank, world, device, teacher, ctx, tsds, ssds, image, peaks, traffic):
    """BASELINE configs[2..4] and the PyTorch-CUDA denominator, measured in the same process right after the headline.
    Every rank takes part (the sweep shards frames, the distillation steps all-reduce); rank 0 keeps the numbers."""
    from tha4_b200 import synthetic
    from tha4_b200.distill import BodyMorpherDistiller
    from tha4_b200.parallel import shard_range
    from tha4_b200.poser.modes import mode_14
    out = {}
    img1 = image.to(device).unsqueeze(0).contiguous()

    # ---- configs[3]: 512-pose sweep, strong scaling (contiguous shards, no collective) ----
    total = 512
    begin, end = shard_range(total, rank, world)
    nloc = end - begin
    sweep_poses = synthetic.random_poses(total, seed=4321)[begin:end].contiguous()
    sp_dev = sweep_poses.to(device)
    img_b = img1.expand(nloc, -1, -1, -1)                      # ONE stored image, batch stride 0

    def sweep_resident(i):
        return teacher.pose(img_b, sp_dev)

    l0 = ctx.counter('kernel_launches')
    ms_sweep = timer.run(sweep_resident, 1, 2) / 2.0
    sweep_launches = (ctx.counter('kernel_launches') - l0) // 3
    img_host = image.unsqueeze(0).contiguous().pin_memory()
    sp_host = sweep_poses.pin_memory()
    frames_host = torch.empty((nloc, 4, 512, 512), dtype=torch.float32).pin_memory()
    img_in, pose_in = torch.empty_like(img1), torch.empty_like(sp_dev)

    def sweep_e2e(i):
        img_in.copy_(img_host, non_blocking=True)
        pose_in.copy_(sp_host, non_blocking=True)
        frames_host.copy_(teacher.pose(img_in.expand(nloc, -1, -1, -1), pose_in), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    ms_sweep_e2e = timer.run(sweep_e2e, 1, 2) / 2.0
    prof = profile_pass(ctx, lambda: sweep_resident(0), 1, rank)
    ms_sweep, ms_sweep_e2e = timer.max_over_ranks(ms_sweep, ms_sweep_e2e)
    sweep = {'value': total / (ms_sweep / 1000.0), 'unit': 'frames/s', 'scaling': 'strong', 'frames_total': total, 'frames_per_gpu': nloc,
             'ms_per_sweep': ms_sweep, 'gpu_launches_per_sweep_rank0': sweep_launches,
             'e2e': {'value': total / (ms_sweep_e2e / 1000.0), 'unit': 'frames/s', 'h2d_bytes_per_step': 4 * 512 * 512 * 4 + nloc * 45 * 4,
                     'd2h_bytes_per_step': nloc * 4 * 512 * 512 * 4, 'ms_per_sweep': ms_sweep_e2e},
             'config': config_for('pose_sweep_512', nloc, world)}
    ro = roofline_objects(prof, 1, peaks, {})
    for k in ('roofline', 'roofline_tail'):
        if k in ro:
            sweep[k] = {kk: ro[k][kk] for kk in ('bound', 'achieved', 'peak', 'unit', 'frac', 'avg_launch_us')}
    out['pose_sweep_512'] = sweep
    del frames_host
    torch.cuda.empty_cache()

    # ---- configs[4]: distillation steps, per-GPU batch 1, one NCCL all-reduce per step ----
    nsteps = args.distill_steps or (1000 if world == 8 else 200)
    dposes = synthetic.random_poses(nsteps * world, seed=777)              # step i, rank r trains on pose i * world + r
    mine = dposes[rank::world].contiguous().to(device)
    student = mode_14.load_body_morpher(None, {k: v.clone() for k, v in ssds['body_morpher'].items()})
    d = BodyMorpherDistiller(teacher, student)
    for i in range(3):                                                      # warm-up steps on a throw-away optimiser state
        d.train_step(img1, mine[i:i + 1], DISTILL_W, DISTILL_LR, want_losses=False)
    d.reset(ssds['body_morpher'])
    g_dist = None
    if world > 1:       # parity of the collective: the all-reduced mean gradient of step 1 (compared with one process below)
        d.train_step(img1, mine[0:1], DISTILL_W, DISTILL_LR, want_losses=False)
        g_dist = d.grad.clone() / world
        d.reset(ssds['body_morpher'])
    ms_d = timer.run(lambda i: d.train_step(img1, mine[i:i + 1], DISTILL_W, DISTILL_LR, want_losses=False), 0, nsteps)
    (ms_d,) = timer.max_over_ranks(ms_d)
    final_dist = d.flat.clone()
    distill = {'steps': nsteps, 'steps_per_s': nsteps / (ms_d / 1000.0), 'examples_per_s': nsteps * world / (ms_d / 1000.0), 'ms_per_step': ms_d / nsteps,
               'batch_per_gpu': 1, 'global_batch': world, 'comm_bytes_per_step': 331567 * 4 if world > 1 else 0,
               'collective': 'one NCCL all-reduce (sum) of the flat fp32 gradient inside the timed region, then Adam with 1/world scaling' if world > 1 else 'none (one rank)',
               'loss_weights': DISTILL_W, 'lr': DISTILL_LR, 'config': config_for('distill_b1', 1, world)}
    if world > 1 and rank == 0:
        # final-weights parity: the same steps as ONE process with the global batch (poses i*world .. i*world+world-1 per step)
        ref_student = mode_14.load_body_morpher(None, {k: v.clone() for k, v in ssds['body_morpher'].items()})
        r = BodyMorpherDistiller(teacher, ref_student, distributed=False)
        imgw = img1.expand(world, -1, -1, -1).contiguous()
        allp = dposes.to(device)
        g_ref = None
        for i in range(nsteps):
            r.train_step(imgw, allp[i * world:(i + 1) * world], DISTILL_W, DISTILL_LR, want_losses=False)
            if i == 0:
                g_ref = r.grad.clone()
        torch.cuda.synchronize()
        w0 = torch.cat([v.reshape(-1) for v in ssds['body_morpher'].values()]).to(device)
        diff = (final_dist - r.flat)
        u_d, u_r = final_dist - w0, r.flat - w0
        # what both runs learned: the four unweighted L1 means on held-out poses, before and after
        held = synthetic.random_poses(4, seed=4242).to(device)
        scratch = torch.zeros_like(w0)

        def eval_losses(flat):
            acc = [0.0] * 4
            for k in range(held.shape[0]):
                t = teacher.get_posing_outputs(img1, held[k:k + 1])
                l = ctx.siren_morpher_train_step(t[5], held[k:k + 1], t[0], t[2], t[3], DISTILL_W, flat.contiguous(), scratch, True)
                acc = [a + float(b) / held.shape[0] for a, b in zip(acc, l)]
            return acc
        distill['final_weights_vs_single_process'] = {
            'step1_mean_gradient_rel_l2': float((g_dist - g_ref).norm() / g_ref.norm()),
            'max_abs': float(diff.abs().max()), 'rel_l2_of_update': float(diff.norm() / u_r.norm()),
            'cosine_of_updates': float(torch.dot(u_d, u_r) / (u_d.norm() * u_r.norm())), 'update_l2': float(u_r.norm()),
            'heldout_l1_terms_initial': eval_losses(w0), 'heldout_l1_terms_distributed': eval_losses(final_dist),
            'heldout_l1_terms_single_process': eval_losses(r.flat),
            'note': 'same %d steps run by one process with global batch %d.  The collective itself is checked by the step-1 mean '
                    'gradient (all-reduce sum / world vs the batched backward; the residue is the TF32 / f16 rounding of two '
                    'different batch shapes).  The weight trajectories are NOT expected to coincide: Adam (eps 1e-8) moves every '
                    'coordinate by ~lr per step whatever |g|, so the ~3e5 coordinates whose gradient is at the rounding-noise level '
                    'random-walk (lr * sqrt(steps) each -- that is what update_l2 consists of) and decorrelate between any two runs, '
                    'as they do between two runs of the reference on a GPU.  What has to agree is what the runs learned: the '
                    'held-out loss terms (terms 2 and 3 carry the loss weights of this phase)' % (nsteps, world)}
    if world > 1:
        dist.barrier()
    out['distill'] = distill
    del d
    torch.cuda.empty_cache()

    # ---- configs[2]: distilled student, batch 64 per GPU ----
    Bs = 64
    sposer = mode_14.create_poser(device, state_dicts=ssds)
    sposer.get_modules()
    sctx = sposer.get_context()
    s_poses = synthetic.random_poses(8 * Bs, seed=99 + rank).to(device)
    s_img = img1.expand(Bs, -1, -1, -1).contiguous()
    ms_s = timer.run(lambda i: sposer.get_posing_outputs(s_img, s_poses[(i % 8) * Bs:(i % 8 + 1) * Bs]), 3, 10)
    s_host = torch.empty((Bs, 4, 512, 512), dtype=torch.float32).pin_memory()
    sp_host2 = s_poses.cpu().pin_memory()
    s_pose_in = torch.empty((Bs, 45), device=device)
    s_img_dense = torch.empty((Bs, 4, 512, 512), device=device)

    def student_e2e(i):
        img_in.copy_(img_host, non_blocking=True)
        s_pose_in.copy_(sp_host2[(i % 8) * Bs:(i % 8 + 1) * Bs], non_blocking=True)
        s_img_dense.copy_(img_in.expand(Bs, -1, -1, -1))
        s_host.copy_(sposer.pose(s_img_dense, s_pose_in), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    ms_s_e2e = timer.run(student_e2e, 3, 10)
    sprof = profile_pass(sctx, lambda: [sposer.get_posing_outputs(s_img, s_poses[:Bs]) for _ in range(5)], 5, rank)
    ms_s, ms_s_e2e = timer.max_over_ranks(ms_s, ms_s_e2e)
    st = {'value': 10 * Bs * world / (ms_s / 1000.0), 'unit': 'frames/s', 'scaling': 'weak', 'ms_per_step': ms_s / 10,
          'e2e': {'value': 10 * Bs * world / (ms_s_e2e / 1000.0), 'unit': 'frames/s', 'h2d_bytes_per_step': 4 * 512 * 512 * 4 + Bs * 45 * 4,
                  'd2h_bytes_per_step': Bs * 4 * 512 * 512 * 4, 'ms_per_step': ms_s_e2e / 10},
          'config': config_for('student_b64', Bs, world)}
    if sprof.get('siren', {}).get('us', 0) > 0:
        ach = 37.89e9 * Bs * 5 / (sprof['siren']['us'] * 1e-6) / 1e12
        st['roofline'] = {'bound': 'tensor', 'achieved': ach, 'peak': peaks['tflops'], 'unit': 'TFLOP/s', 'frac': ach / peaks['tflops'],
                          'note': '37.89 GFLOP and 131.8 M sin per frame (SURVEY 8d): the MUFU pipe is the co-bound'}
    out['student_b64'] = st
    del sposer, s_host
    torch.cuda.empty_cache()

    # ---- the ">= 30x PyTorch-CUDA" denominator: configs[1] through PyTorch eager on this GPU (rank 0) ----
    if rank == 0:
        try:
            fps, ms_t = torch_cuda_eager_fps('mode_07', tsds, image, synthetic.random_poses(64, seed=1234), 1, 3, 10, device)
            out['torch_cuda_eager'] = {'value': fps, 'unit': 'frames/s', 'ms_per_step': ms_t, 'steps': 10, 'batch': 1,
                                       'note': 'the oracle\'s PyTorch ops on this GPU (cuDNN / cuBLAS, TF32 convs allowed) = what the reference\'s own '
                                               'CUDA path dispatches for configs[1]; denominator of BASELINE\'s ">= 30x" target'}
        except Exception as exc:       # context number only: never fail the bench line on it
            out['torch_cuda_eager'] = {'unavailable': repr(exc)[:200]}
    if world > 1:
        dist.barrier()
    return out


if __name__ == '__main__':
    main()
