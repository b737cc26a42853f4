#!/usr/bin/env python
"""bench.py -- depth-maps/sec of the FastDepth forward path (MobileNetSkipAdd.forward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of synthetic input: batch 64 per GPU,
224x224, fp16, MobileNet-NNConv5(dw)+skipadd (BASELINE.json metric config; weak scaling: every
rank keeps 64 images).  Prints ONE JSON line on rank 0.

  value      whole-job images/s with inputs resident in HBM (CUDA events, max over ranks); `--lanes` (default 3) independent
             forwards are in flight (plan copies with their own activation buffers on their own streams: another batch's kernels fill
             the idle SM time at every kernel boundary); `single_stream` in the line is the strict one-at-a-time replay
  e2e        same metric through the C-ABI host-buffer call fd_forward_host: pinned-host -> device
             copy of the batch and device -> host copy of the depth maps inside the timed region
  roofline   the dominant kernel's achieved HBM GB/s = algorithmic bytes / launch duration
             (each kernel timed alone with CUDA events, L2 flushed between launches)
  cpu_baseline  the oracle port of the reference forward (torch CPU fp32) on this box's host cores,
             bounded sample
  gpu_library_baseline  (N=1) the reference's own eager CUDA forward -- the module's nn.Conv2d / BatchNorm2d / ReLU6 /
             F.interpolate children run by PyTorch + cuDNN (cudnn.benchmark=True), fp16 and fp32, NCHW and channels_last --
             on the same B200: the existing-Blackwell-library bar (SURVEY.md 8d).  Outside the product's timed region.
  eval       BASELINE config 4's shape: bf16, 64 images per rank, per-image metrics on device, ONE all-reduce(SUM) of
             11 doubles (NCCL under torchrun); prints delta1 / RMSE next to the oracle's, the all-reduce time and whether
             the N-rank sums equal the sums of a single rank that ran every image (bit for bit, fp64)
  --impl reference : times ONLY that CPU implementation (the reference is pure Python on PyTorch;
             /root/reference does not exist on the GPU box, so the oracle port stands in).
  --dump-outputs DIR : after the timed steps, writes the depth maps the timed path returned in its last step (rank 0) as
             DIR/depth.npy (float32).  Inputs and weights are seeded, so two builds run with the same arguments can be
             compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = 'depth-maps/sec @224x224 b64'
UNIT = 'images/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=64, help='images per GPU')
    ap.add_argument('--hw', type=int, nargs=2, default=[224, 224])
    ap.add_argument('--dtype', default='fp16', choices=['fp16', 'bf16', 'fp32'])
    ap.add_argument('--widths', default='stock', choices=['stock', 'pruned'])
    ap.add_argument('--path', type=int, default=1)
    ap.add_argument('--fold-head', type=int, default=1)
    ap.add_argument('--graph', type=int, default=1)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--stage-iters', type=int, default=10)
    ap.add_argument('--no-lib-baseline', action='store_true', help='skip the cuDNN-eager leg')
    ap.add_argument('--no-eval', action='store_true', help='skip the bf16 sharded-evaluation leg (config 4)')
    ap.add_argument('--e2e-steps', type=int, default=200)
    ap.add_argument('--lanes', type=int, default=3, help='batches in flight: independent plan copies on their own streams '
                                                         '(fastdepth_b200.engine.ForwardLanes); 1 = strict single stream')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the last timed step\'s depth maps to DIR/depth.npy')
    return ap.parse_args()


def peaks():
    """(HBM GB/s, sustained dense 16-bit TFLOP/s, SM MHz, source)"""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return (float(d['hbm_gbs']), float(d.get('bf16_tflops_sustained', 1467.7)), float(d.get('sm_max_mhz', 1965.0)),
                'measured (MEASURED_PEAKS.json hbm_gbs burst copy; bf16_tflops_sustained)')
    return 6650.0, 1400.0, 1965.0, 'fallback (B200_PROFILING.md)'


NOMINAL_HBM_GBS = 8000.0        # the figure north_star quotes
DUMP_MAX_ELEMS = 12 << 20       # 48 MiB of float32: keeps a dump well under 64 MB


def dump_outputs(out_dir, y):
    """Write ``y`` as out_dir/depth.npy in float32.  An output of more than DUMP_MAX_ELEMS elements is replaced by a fixed sample:
    the flattened elements at DUMP_MAX_ELEMS positions drawn with a fixed seed (the same positions for the same shape)."""
    import numpy as np
    a = y.detach().float().cpu().numpy()
    if a.size > DUMP_MAX_ELEMS:
        pos = np.sort(np.random.Generator(np.random.PCG64(0)).choice(a.size, size=DUMP_MAX_ELEMS, replace=False))
        a = a.reshape(-1)[pos]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'depth.npy'), a)


def eager_reference_forward(model, x):
    """The reference forward (models.py:706-732) run by PyTorch's own operators on the module's children: the
    existing-library baseline (cuDNN convolutions, ~122 kernel launches per forward).  Bench-only; the product's
    ``forward`` never takes this route."""
    import torch.nn.functional as F
    keep = {}
    for i in range(14):
        x = getattr(model, 'conv%d' % i)(x)
        if i in (1, 3, 5):
            keep[i] = x
    add_after = {4: 1, 3: 3, 2: 5}
    for j in range(1, 6):
        x = getattr(model, 'decode_conv%d' % j)(x)
        x = F.interpolate(x, scale_factor=2, mode='nearest')
        if j in add_after:
            x = x + keep[add_after[j]]
    return model.decode_conv6(x)


def gpu_library_baseline(widths, sd, n, h, w, dev, ours_value, iters=20):
    """img/s of the eager cuDNN forward at batch n for {fp16, fp32} x {NCHW, channels_last}; CUDA events, synchronised."""
    import models
    from fastdepth_b200 import synthetic
    prev = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True                      # reference main.py:10
    out = {'batch': n, 'api': 'torch %s eager / cuDNN %s, cudnn.benchmark=True' % (torch.__version__, torch.backends.cudnn.version())}
    x32 = synthetic.synthetic_input(n, h, w, seed=0).to(dev)
    try:
        for dname, dt in (('fp16', torch.float16), ('fp32', torch.float32)):
            for lname, fmt in (('nchw', torch.contiguous_format), ('channels_last', torch.channels_last)):
                m = models.MobileNetSkipAdd((h, w), pretrained=False, widths=widths)
                m.load_state_dict(sd)
                m = m.eval().to(dev).to(dt).to(memory_format=fmt)
                x = x32.to(dt).contiguous(memory_format=fmt)
                with torch.no_grad():
                    for _ in range(5):
                        y = eager_reference_forward(m, x)
                    torch.cuda.synchronize(dev)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(iters):
                        y = eager_reference_forward(m, x)
                    e1.record()
                    torch.cuda.synchronize(dev)
                out['%s_%s' % (dname, lname)] = n * iters / (e0.elapsed_time(e1) * 1e-3)
                del m, y
    finally:
        torch.backends.cudnn.benchmark = prev
    best16 = max(out['fp16_nchw'], out['fp16_channels_last'])
    out.update({'unit': UNIT, 'best_fp16': best16, 'ours_over_best_fp16': ours_value / best16,
                'ours_over_fp32_nchw': ours_value / out['fp32_nchw'],
                'note': 'reference forward (models.py:706-732) through PyTorch eager on the same GPU; fp32 NCHW is what '
                        'main.py feeds (main.py:68), fp16 is the like-for-like precision of `value`'})
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (recipe's clocks line)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                f = [s.strip() for s in out.strip().split(',')]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = set()
        for s in self.samples:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.samples[0][1]), 'reasons': sorted(reasons),
                'samples': len(self.samples), 'power_w_max': max(float(s[2]) for s in self.samples)}


def build_sd(widths_name):
    from fastdepth_b200 import synthetic
    widths = synthetic.STOCK_WIDTHS if widths_name == 'stock' else synthetic.PRUNED_WIDTHS
    return widths, synthetic.synthetic_state_dict(widths, seed=1)


def usable_cpus():
    """CPUs this process may really use: the affinity mask, capped by the cgroup CPU quota (a container that shows 128
    cores but is throttled to a few turns a 128-thread OpenMP run into seconds per image)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ('/sys/fs/cgroup/cpu.max', '/sys/fs/cgroup/cpu/cpu.cfs_quota_us'):
        try:
            txt = open(path).read().split()
            if path.endswith('cpu.max'):
                if txt[0] != 'max':
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def pick_cpu_threads(sd, h, w):
    """The reference arm is meant to use all the host threads it can use WELL: sweep the thread count upwards on a
    one-image forward and keep the fastest (stops as soon as more threads make it slower).  Returns (threads, note)."""
    from fastdepth_b200 import synthetic
    from oracle import fastdepth_oracle as orc          # the CPU baseline leg may execute the oracle
    torch.set_grad_enabled(False)
    top = usable_cpus()
    cands = sorted({c for c in (4, 8, 16, 32, 64, 128, 256, top // 2, top) if 1 <= c <= top})
    x1 = synthetic.synthetic_input(1, h, w, seed=0)
    best_t, best_c, log = None, cands[0], []
    for c in cands:
        torch.set_num_threads(c)
        orc.skipadd_forward(sd, x1)
        t0 = time.perf_counter(); orc.skipadd_forward(sd, x1); t = time.perf_counter() - t0
        log.append('%d:%.0fms' % (c, t * 1e3))
        if best_t is None or t < best_t:
            best_t, best_c = t, c
        elif t > 1.5 * best_t:
            break
    torch.set_num_threads(best_c)
    return best_c, 'threads swept on a 1-image forward (%s of %d usable CPUs)' % (' '.join(log), top)


def cpu_forward_rate(sd, h, w, budget_s, min_steps, warmup, batch=None):
    """Time the oracle port of the reference forward on the host cores; returns (img/s, batch, steps, s/step, last output)."""
    from fastdepth_b200 import synthetic
    from oracle import fastdepth_oracle as orc          # the CPU baseline leg may execute the oracle
    torch.set_grad_enabled(False)
    if batch is None:
        x1 = synthetic.synthetic_input(1, h, w, seed=0)
        orc.skipadd_forward(sd, x1)
        t0 = time.perf_counter(); orc.skipadd_forward(sd, x1); t1 = time.perf_counter() - t0
        batch = max(1, min(8, int(1.0 / max(t1, 1e-3))))   # ~1 s of work per step, main.py feeds bs 1 (l.41)
    x = synthetic.synthetic_input(batch, h, w, seed=0)
    for _ in range(warmup):
        orc.skipadd_forward(sd, x)
    times = []
    t_start = time.perf_counter()
    while len(times) < min_steps or (budget_s and time.perf_counter() - t_start < budget_s and len(times) < 10 * min_steps):
        t0 = time.perf_counter()
        y = orc.skipadd_forward(sd, x)
        times.append(time.perf_counter() - t0)
        if budget_s and time.perf_counter() - t_start > budget_s and len(times) >= min_steps:
            break
    per = sum(times) / len(times)
    return batch / per, batch, len(times), per, y


def run_eval(rank, world, dev, widths, sd, h, w, n, lanes=1):
    """BASELINE config 4's shape on however many ranks there are: bf16, n images per rank, image-sharded, per-image
    metrics on device, ONE all-reduce(SUM) of 11 doubles (reference metrics.py:71-95, main.py:80-82).  Returns rank 0's
    report.  Outside every timed region of the headline metric; the oracle is used here as the checker only (targets
    around its fp32 prediction, SURVEY.md 8d, and its own per-image metrics on the same pairs)."""
    import torch.distributed as dist
    import models
    from fastdepth_b200 import evaluate, synthetic
    from fastdepth_b200.plan import METRIC_NAMES, metrics_accumulate
    from oracle import fastdepth_oracle as orc           # checker only
    dt = torch.bfloat16
    torch.set_grad_enabled(False)
    m = models.MobileNetSkipAdd((h, w), pretrained=False, widths=widths)
    m.load_state_dict(sd)
    m = m.eval().to(dev).to(dt)
    x = synthetic.synthetic_input(n, h, w, seed=5000 + rank)
    torch.set_num_threads(max(1, min(32, usable_cpus() // max(1, world))))
    ref = orc.skipadd_forward(sd, x)
    tgt = synthetic.synthetic_target(ref, seed=6000 + rank)
    xd, td = x.to(dev).to(dt), tgt.to(dev)
    # (a) the sharded evaluation through the product's own entry point (forward + device metrics + the one collective)
    ours, sums = evaluate.evaluate(m, [(xd[:n // 2], td[:n // 2]), (xd[n // 2:], td[n // 2:])], dev, return_sums=True, lanes=min(2, lanes))
    # (b) the collective alone, timed on the device: 11 doubles, latency only
    ar_us = None
    if world > 1:
        scratch = torch.ones(11, dtype=torch.float64, device=dev)
        for _ in range(10):
            dist.all_reduce(scratch)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            dist.all_reduce(scratch)
        e1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1) / 50 * 1e3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ar_us = t.item()
    # (c) the oracle's metrics on the same (image, target) pairs, reduced the same way
    om, cnt = orc.average_per_image(ref.numpy(), tgt.numpy())
    osum = torch.tensor([om[k] * cnt for k in METRIC_NAMES] + [float(cnt)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(osum)
    oracle_avg = {k: osum[i].item() / osum[-1].item() for i, k in enumerate(METRIC_NAMES)}
    # (d) bookkeeping: ONE rank runs every rank's images; its fp64 sums must equal the all-reduced ones bit for bit
    if world > 1:
        xs_all = [torch.empty_like(xd) for _ in range(world)]
        ts_all = [torch.empty_like(td) for _ in range(world)]
        dist.all_gather(xs_all, xd)
        dist.all_gather(ts_all, td)
    else:
        xs_all, ts_all = [xd], [td]
    same = None
    if rank == 0:
        one = evaluate.new_sums(dev)
        for xa, ta in zip(xs_all, ts_all):
            metrics_accumulate(m(xa), ta, one)
        torch.cuda.synchronize(dev)
        same = bool(torch.equal(one, sums))
    del m
    return {'config': 'BASELINE config 4 shape: bf16, %d images per rank x %d rank(s) = %d, image-sharded' % (n, world, n * world),
            'dtype': 'bf16', 'images': int(round(ours['count'])), 'delta1': ours['delta1'], 'rmse_mm': ours['rmse'],
            'absrel': ours['absrel'], 'delta1_oracle_fp32': oracle_avg['delta1'], 'rmse_mm_oracle_fp32': oracle_avg['rmse'],
            'absrel_oracle_fp32': oracle_avg['absrel'],
            'collective': ('NCCL all_reduce(SUM) of 11 fp64 (88 B), %d ranks' % world) if world > 1 else 'none (1 rank)',
            'allreduce_us': ar_us, 'n_rank_sums_equal_single_rank_sums_bitwise': same}


def run_reference(args, rank):
    if rank != 0:
        return
    widths, sd = build_sd(args.widths)
    h, w = args.hw
    # torchrun exports OMP_NUM_THREADS=1 for every worker; the reference arm is meant to use all host threads it can
    cores, thread_note = pick_cpu_threads(sd, h, w)
    # batch <= 8 per step on purpose: that is where the CPU forward is fastest per image (batch 64 measured 31 img/s against 77-240
    # at batch 8 on the same cores: the activations fall out of the caches), and the reference arm should be the reference at its best
    rate, batch, steps, per, y = cpu_forward_rate(sd, h, w, budget_s=0, min_steps=max(1, args.steps), warmup=max(1, args.warmup))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': rate, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': steps,
        'warmup': max(1, args.warmup), 'ms_per_step': per * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'MobileNet-NNConv5(dw)+skipadd %s widths, %dx%d, reference forward on host CPU' %
                               (args.widths, h, w), 'batch_per_step': batch, 'global_batch': batch},
        'cpu_baseline': {'value': rate, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '%d steps of batch %d (fp32, torch CPU, NCHW) -- the reference is pure Python on '
                                   'PyTorch and /root/reference is absent on the GPU box, so the oracle port runs; %s' % (steps, batch, thread_note)},
        'e2e': {'value': rate, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        run_reference(args, rank)
        return

    import torch.distributed as dist
    import models
    from fastdepth_b200 import synthetic
    from fastdepth_b200.engine import SkipAddEngine

    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    dtype = {'fp16': torch.float16, 'bf16': torch.bfloat16, 'fp32': torch.float32}[args.dtype]
    h, w = args.hw
    n = args.batch
    widths, sd = build_sd(args.widths)
    model = models.MobileNetSkipAdd((h, w), pretrained=False, widths=widths)
    model.load_state_dict(sd)
    model = model.eval().to(dev).to(dtype)
    from fastdepth_b200.engine import ForwardLanes
    opts = {'path': args.path, 'fold_head': args.fold_head, 'graph': args.graph}
    eng = SkipAddEngine(model)                      # the module's own (single-stream) engine: parity check, eval leg, per-kernel table
    for k, v in opts.items():
        eng.set_option(k, v)
    model.__dict__['_fd_engine'] = eng
    R = max(1, args.lanes)
    lanes = ForwardLanes(model, lanes=R, options=opts)

    # 4 rotating input batches (different images per rank); a step moves >1 GB through HBM, far more
    # than the 126 MB L2, so nothing of the previous step's input survives in cache.
    n_rot = 4
    xs = [synthetic.synthetic_input(n, h, w, seed=100 * rank + i).to(dev).to(dtype) for i in range(n_rot)]
    y = torch.empty((n, 1, h, w), dtype=dtype, device=dev)
    plan = eng.plan_for(xs[0])
    stream = torch.cuda.current_stream(dev)
    sp = stream.cuda_stream
    lane_plans = lanes.plans_for(xs[0])
    lane_streams = lanes.streams_for(dev)
    lane_y = [torch.empty((n, 1, h, w), dtype=dtype, device=dev) for _ in range(R)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, warmup, fan=None):
        """CUDA-event time of `steps` calls of fn.  `fan`: the lane streams the calls are spread over -- they all wait for the
        start event and the end event (on the main stream) waits for all of them."""
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for s_ in (fan or ()):
            s_.wait_event(e0)
        for i in range(steps):
            fn(i)
        for s_ in (fan or ()):
            stream.wait_stream(s_)
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    # ---- value: device-resident inputs ---------------------------------------------------------
    # `lanes` forwards in flight: step i runs on lane i % R (own plan copy, own stream); R = 1 is the strict single-stream replay
    ms_single = timed(lambda i: plan.forward(xs[i % n_rot], y, sp), args.steps, max(3, args.warmup))
    if R > 1:
        ms_total = timed(lambda i: lane_plans[i % R].forward(xs[i % n_rot], lane_y[i % R], lane_streams[i % R].cuda_stream),
                         args.steps, max(3, args.warmup) * R, fan=lane_streams)
    else:
        ms_total = ms_single
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lane_y[(args.steps - 1) % R] if R > 1 else y)
    # ---- e2e: pinned host buffers through the C-ABI pipeline (fd_pipeline_submit / fd_pipeline_wait): every step
    # uploads its batch from pinned host memory and downloads its depth maps; up to 3 batches are in flight so
    # the PCIe copies overlap the forward of the neighbouring steps.  Timed on the host clock between device-wide
    # synchronisations (the work spans three streams), max over ranks.
    xh = [x.cpu().pin_memory() for x in xs[:3]]
    yh = [torch.empty((n, 1, h, w), dtype=dtype).pin_memory() for _ in range(3)]
    xh_l = [xh for _ in range(R)]                                    # pinned inputs are read-only: shared by the lanes
    yh_l = [[torch.empty((n, 1, h, w), dtype=dtype).pin_memory() for _ in range(3)] for _ in range(R)]
    e2e_steps = max(6, args.steps, args.e2e_steps)      # ~0.13 s per repeat at batch 64: long enough to be stable

    def run_pipeline(k):
        # every lane has its own fd_pipeline (three batches in flight each: copies of one batch overlap the forward of its
        # neighbours); batches go round-robin over the lanes, the host waits for a batch 2 * R submissions later
        pending = []
        for i in range(k):
            lane = i % R
            pending.append((lane_plans[lane], lane_plans[lane].pipeline_submit(xh_l[lane][(i // R) % 3], yh_l[lane][(i // R) % 3])))
            if len(pending) > 2 * R:
                p_, t_ = pending.pop(0)
                p_.pipeline_wait(t_)
        for p_, t_ in pending:
            p_.pipeline_wait(t_)

    run_pipeline(8)
    reps = []
    for _ in range(3):                                    # median of three repeats (max over ranks each)
        barrier()
        t0 = time.perf_counter()
        run_pipeline(e2e_steps)
        torch.cuda.synchronize(dev)
        el = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(el, op=dist.ReduceOp.MAX)
        reps.append(el.item() * 1e3)
    ms_e2e = sorted(reps)[1]
    # the plain synchronous call, for reference
    ms_sync = timed(lambda i: plan.forward_host(xh[i % 3], yh[i % 3], sp), 5, 2) / 5
    clocks = sampler.summary() if sampler else None

    value = world * n * args.steps / (ms_total * 1e-3)
    e2e_value = world * n * e2e_steps / (ms_e2e * 1e-3)

    # ---- config-4 evaluation leg: every rank takes part (forward in bf16, device metrics, the path's one collective)
    eval_info = None
    if not args.no_eval and (h, w) == (224, 224):
        eval_info = run_eval(rank, world, dev, widths, sd, h, w, n, lanes=R)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- per-kernel roofline (rank 0, each kernel alone, L2 flushed) ---------------------------
    hbm_peak, tensor_peak, sm_mhz, peak_src = peaks()
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    steps = plan.time_steps(xs[0], y, sp, warmup=2, iters=args.stage_iters, flush_l2=True)
    for s in steps:
        s['gbs'] = s['alg_bytes'] / (s['ms'] * 1e-3) / 1e9 if s['ms'] > 0 else 0.0
        s['frac'] = s['gbs'] / hbm_peak
        s['tflops'] = 2 * s['macs'] / (s['ms'] * 1e-3) / 1e12 if s['ms'] > 0 else 0.0
        s['dense_tflops'] = 2 * s['dense_macs'] / (s['ms'] * 1e-3) / 1e12 if s['ms'] > 0 else 0.0
        # the three floors of a fused stage: HBM (algorithmic bytes), the SIMT FMA pipe for the depthwise taps (128 FMA lanes
        # per SM and clock, north_star keeps them off the tensor cores) and the tensor pipe for the dense contraction
        s['hbm_floor_us'] = s['alg_bytes'] / (hbm_peak * 1e9) * 1e6
        s['fma_floor_us'] = s['dw_macs'] / (n_sms * 128.0 * sm_mhz * 1e6) * 1e6
        s['tensor_floor_us'] = 2 * s['dense_macs'] / (tensor_peak * 1e12) * 1e6
        s['floor_us'] = max(s['hbm_floor_us'], s['fma_floor_us'], s['tensor_floor_us'])
    top = max(steps, key=lambda s: s['ms'])
    # DRAM traffic of that kernel from the committed `ncu --set full` capture of the same configuration (if any)
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'r02_final_traffic.json')
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, 'profiles', 'r01_final_traffic.json')
    if os.path.exists(tpath) and args.widths == 'stock' and args.dtype == 'fp16' and n == 64 and (h, w) == (224, 224) and args.path == 1:
        tj = json.load(open(tpath))['stages'].get(top['stage_name'])
        if tj:
            traffic = (tj['dram_read_mb'] + tj['dram_write_mb']) * 1e6
    sum_ms = sum(s['ms'] for s in steps)
    alg_total = sum(s['alg_bytes'] for s in steps)

    # ---- parity on this very configuration (2 images vs the oracle) ------------------------------
    from oracle import fastdepth_oracle as orc           # checker only
    with torch.no_grad():
        got = model(xs[0][:2].clone()).float().cpu()
    sdq = {k: (v.to(dtype).float() if v.is_floating_point() else v) for k, v in sd.items()}
    want = orc.skipadd_forward(sdq, xs[0][:2].float().cpu())
    denom = torch.maximum(want.abs(), want.abs().mean())
    max_rel = ((got - want).abs() / denom).max().item()
    tgt = synthetic.synthetic_target(want, seed=1)
    m_ours, _ = orc.average_per_image(got.numpy(), tgt.numpy())
    m_ref, _ = orc.average_per_image(want.numpy(), tgt.numpy())

    lib = None
    if not args.no_lib_baseline and world == 1 and args.dtype == 'fp16':
        lib = gpu_library_baseline(widths, sd, n, h, w, dev, value)

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        ccores, thread_note = pick_cpu_threads(sd, h, w)
        rate, cb, csteps, per, _ = cpu_forward_rate(sd, h, w, budget_s=15.0, min_steps=3, warmup=1)
        cpu = {'value': rate, 'unit': UNIT, 'cores': ccores, 'kind': 'port',
               'sample': '%d forwards of batch %d at %dx%d, fp32 torch CPU (oracle port of reference models.py:706-732), '
                         '%.2f s each; %s' % (csteps, cb, h, w, per, thread_note)}

    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': max(3, args.warmup), 'ms_per_step': ms_total / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': {'fp16': 'f16', 'bf16': 'bf16', 'fp32': 'f32'}[args.dtype],
        'data': 'synthetic',
        'config': {'workload': 'MobileNet-NNConv5(dw)+skipadd (%s widths) forward, batch %d/GPU, %dx%d, %s'
                               % (args.widths, n, h, w, args.dtype),
                   'global_batch': n * world, 'parallelism': 'image-sharded x%d (no data-path collective)' % world,
                   'path': args.path, 'fold_head': args.fold_head, 'graph': args.graph,
                   'in_flight': R, 'in_flight_note': '%d independent forwards in flight (plan copies with their own activation buffers on their '
                                                     'own streams, fastdepth_b200.engine.ForwardLanes): every step is a '
                                                     'complete forward of its own batch; the strict single-stream replay is `single_stream`' % R,
                   'l2': '4 rotating input batches; one step streams %.2f GB through HBM (>> 126 MB L2)' % (alg_total / 1e9),
                   'weights': 'random-init (synthetic recipe seed 1)'},
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': xh[0].numel() * xh[0].element_size(),
                'd2h_bytes_per_step': yh[0].numel() * yh[0].element_size(), 'ms_per_step': ms_e2e / e2e_steps,
                'api': 'fd_pipeline_submit/fd_pipeline_wait (C-ABI, pinned host buffers, 3 batches in flight per lane, %d lane(s))' % R,
                'steps': e2e_steps, 'repeats_ms': [round(r, 3) for r in reps], 'statistic': 'median of 3 repeats, max over ranks each',
                'sync_call_ms_per_step': ms_sync, 'sync_call_api': 'fd_forward_host'},
        'single_stream': {'value': world * n * args.steps / (ms_single * 1e-3), 'unit': UNIT, 'ms_per_step': ms_single / args.steps,
                          'note': 'one forward at a time on one stream (CUDA-graph replay): the latency of a batch'},
        'gpu_launches': plan.launches_per_forward() * args.steps,
        'launches_per_step': plan.launches_per_forward(),
        'clocks': clocks,
        # the dominant kernel's own roofline: a merged multi-layer stage (the conv7..11 chain keeps its intermediates in shared
        # memory) sits far past the ridge -- its dense contraction, not its 28 MB of external bytes, is what bounds it
        'roofline': {**({'bound': 'tensor', 'achieved': top['dense_tflops'], 'peak': tensor_peak, 'unit': 'TFLOP/s',
                         'frac': top['dense_tflops'] / tensor_peak, 'hbm_gbs': top['gbs'], 'hbm_frac': top['frac']}
                        if top['tensor_floor_us'] > top['hbm_floor_us'] else
                        {'bound': 'hbm', 'achieved': top['gbs'], 'peak': hbm_peak, 'unit': 'GB/s', 'frac': top['frac']}),
                     'frac_nominal_8tbs': top['gbs'] / NOMINAL_HBM_GBS,
                     'traffic': traffic, 'traffic_source': os.path.basename(tpath) if traffic else None,
                     'kernel': top['kernel'], 'stage': top['stage_name'], 'peak_source': peak_src,
                     'kernel_ms': top['ms'], 'share_of_step': top['ms'] / sum_ms,
                     'alg_bytes': top['alg_bytes'],
                     # a fused depthwise stage also has a SIMT floor: taps / (128 FMA lanes x SMs x clock); when that exceeds
                     # the HBM time the HBM fraction of even a perfect kernel is hbm_floor / fma_floor
                     'hbm_floor_us': top['hbm_floor_us'], 'fma_floor_us': top['fma_floor_us'],
                     'tensor_floor_us': top['tensor_floor_us'],
                     'frac_ceiling_given_fma_floor': min(1.0, top['hbm_floor_us'] / max(top['floor_us'], 1e-9)),
                     'frac_of_binding_floor': top['floor_us'] / (top['ms'] * 1e3),
                     'whole_step': {'alg_bytes': alg_total, 'gbs_at_value': alg_total / (ms_total / args.steps * 1e-3) / 1e9,
                                    'frac_at_value': alg_total / (ms_total / args.steps * 1e-3) / 1e9 / hbm_peak,
                                    'frac_nominal_8tbs': alg_total / (ms_total / args.steps * 1e-3) / 1e9 / NOMINAL_HBM_GBS,
                                    'sum_of_isolated_kernel_ms': sum_ms,
                                    'sum_of_binding_floors_us': sum(s['floor_us'] for s in steps)}},
        'stages': [{'stage': s['stage_name'], 'kernel': s['kernel'], 'ms': round(s['ms'], 5),
                    'alg_mb': round(s['alg_bytes'] / 1e6, 3), 'gbs': round(s['gbs'], 1), 'frac': round(s['frac'], 4),
                    'frac_8tbs': round(s['gbs'] / NOMINAL_HBM_GBS, 4), 'tflops': round(s['tflops'], 2),
                    'hbm_floor_us': round(s['hbm_floor_us'], 2), 'fma_floor_us': round(s['fma_floor_us'], 2),
                    'tensor_floor_us': round(s['tensor_floor_us'], 2),
                    'frac_of_floor': round(s['floor_us'] / (s['ms'] * 1e3), 4) if s['ms'] > 0 else 0.0} for s in steps],
        'parity': {'max_rel_err_vs_oracle': max_rel, 'delta1': m_ours['delta1'], 'delta1_oracle': m_ref['delta1'],
                   'rmse_mm': m_ours['rmse'], 'rmse_mm_oracle': m_ref['rmse']},
        'cpu_baseline': cpu,
        'gpu_library_baseline': lib,
        'eval': eval_info,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
