#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 wavelet filterbank engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|aten] [--config headline|c5]
                    [--dump-outputs DIR]
    (N>1: run as  python -m torch.distributed.run --nproc-per-node N bench.py --gpus N ...)

One "step" = one pass of the hot path over one batch of synthetic input:
    DWTForward(J=3,'db4','symmetric') on randn(128,32,512,512)          (BASELINE.json configs[1])
  + DTCWTForward(J=3,'near_sym_a','qshift_a') on randn(64,3,1024,1024)  (BASELINE.json configs[2])
i.e. the two transforms BASELINE.json's metric names ("Mpixels/sec DWT J=3 db4 + DTCWT J=3 fwd").
`value` = input pixels of both transforms on all ranks / device time (max over ranks), inputs resident in HBM.
Inputs (4.3 GB + 0.8 GB) are far larger than the 126 MB L2, so no explicit flush is needed (config.l2).

Also on the JSON line:
  parts        per-transform figures incl. the other BASELINE configs (inverses, ScatLayer x2, the config-5 shard shape),
               each {ms, alg_bytes, GBps, frac of the measured HBM peak} (N = 1 only, to bound the run time)
  roofline     the dominant kernel (the level-1 pyramid kernel = one DWTForward(J=1) call), algorithmic bytes over
               live CUDA-event time; whole_transform = the same for the complete transforms
  cpu_baseline the oracle port on the host cores (bounded sample, >= 3 repetitions, spread reported)
  e2e          host pinned buffers -> public nn.Module API -> host pinned buffers, copies inside the timed region
  gather       (N > 1) the same step followed by ONE NCCL all-gather of every output tensor (north_star's
               "single NCCL gather at the end"): value_with_gather, bytes and GB/s moved per rank
  clocks, gpu_launches

--impl reference : the CPU implementation of the same path (oracle port, all host threads) on a bounded sample;
                   rank 0 only, never multiplied by the GPU count.
--impl aten      : the reference's GPU op sequence re-written independently from the closed forms (symmetric-extension
                   gather + depthwise F.conv2d + slicing), i.e. the "existing kernels" bar on the same B200.
--config c5      : BASELINE.json configs[4]: DWTForward J=4 db8 (zero) on N=1024, C=16, 2048x2048, sharded over N,
                   streamed through the GPUs in chunks; yl is all-gathered at the end (the band-passes stay rank-resident).
--dump-outputs DIR : after the timed steps, write what the last step returned (yl and every yh[j] of both transforms,
                   rank 0) as DIR/<name>.npy, float32; see dump_outputs().  The inputs are seeded, so two builds run with
                   the same arguments can be compared output for output.  Headline config of --impl ours only.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DWT_SHAPE = (128, 32, 512, 512)
DTCWT_SHAPE = (64, 3, 1024, 1024)
SCAT_SHAPE = (256, 3, 256, 256)
C5_CHUNK = (8, 16, 2048, 2048)
METRIC = 'Mpixels/sec DWT J=3 db4 + DTCWT J=3 fwd'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'aten'])
    ap.add_argument('--config', default='headline', choices=['headline', 'c5'])
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-parts', action='store_true')
    ap.add_argument('--no-gather', action='store_true')
    ap.add_argument('--dwt-batch', type=int, default=DWT_SHAPE[0])
    ap.add_argument('--dtcwt-batch', type=int, default=DTCWT_SHAPE[0])
    ap.add_argument('--c5-n-total', type=int, default=1024)
    ap.add_argument('--c5-chunk', type=int, default=16)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None)
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs is not None and (a.impl != 'ours' or a.config != 'headline'):
        ap.error('--dump-outputs is only supported for the headline config of --impl ours')
    return a


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


def dwt_alg_bytes(planes, H, W, L, J):
    h, w, tot = H, W, H * W
    for _ in range(J):
        h, w = (h + L - 1) // 2, (w + L - 1) // 2
        tot += 3 * h * w
    return 4.0 * planes * (tot + h * w)


# ------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on a bounded sample (also the cpu_baseline of the GPU arm)

def _set_host_threads(n):
    """All host cores for the OpenMP oracle, whatever the launcher exported (torchrun presets OMP_NUM_THREADS=1)."""
    import ctypes
    os.environ['OMP_NUM_THREADS'] = str(n)
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
    except Exception:
        pass
    try:
        ctypes.CDLL('libgomp.so.1').omp_set_num_threads(int(n))
    except Exception:
        pass


def cpu_sample(dwt_n=8, dtcwt_n=None, reps=3):
    import numpy as np
    cores = os.cpu_count() or 1
    if dtcwt_n is None:   # the oracle parallelises over planes (3 per image): give every host thread one
        dtcwt_n = max(8, min(64, (cores + 2) // 3))
    _set_host_threads(cores)
    from oracle import oracle as orc
    from pytorch_wavelets_b200 import wavelets
    from pytorch_wavelets_b200.dtcwt import coeffs
    orc.lib()
    _set_host_threads(cores)
    w = wavelets.Wavelet('db4')
    h0, h1 = np.array(w.dec_lo[::-1]), np.array(w.dec_hi[::-1])
    h0o, _, h1o, _ = coeffs.biort('near_sym_a')
    q = coeffs.qshift('qshift_a')
    l1 = (h0o[::-1].ravel(), h1o[::-1].ravel())
    qs = tuple(q[i][::-1].ravel() for i in (0, 1, 4, 5))
    rng = np.random.default_rng(0)
    xd = rng.standard_normal((dwt_n,) + DWT_SHAPE[1:]).astype(np.float32)
    xt = rng.standard_normal((dtcwt_n,) + DTCWT_SHAPE[1:]).astype(np.float32)
    orc.dwt_forward(xd[:2], (h0, h1, h0, h1), 3, 'symmetric')  # warm-up (page-in, threads)
    orc.dtcwt_forward(xt[:2], l1, qs, 3)
    td, tt = [], []
    for _ in range(reps):
        t = time.perf_counter()
        orc.dwt_forward(xd, (h0, h1, h0, h1), 3, 'symmetric')
        td.append(time.perf_counter() - t)
        t = time.perf_counter()
        orc.dtcwt_forward(xt, l1, qs, 3)
        tt.append(time.perf_counter() - t)
    # the same MIX of work as one GPU step: pixels weighted like the full workload; median of the repetitions
    med = lambda v: sorted(v)[len(v) // 2]
    pd, pt = float(np.prod(DWT_SHAPE)), float(np.prod(DTCWT_SHAPE))
    rate_d, rate_t = xd.size / med(td), xt.size / med(tt)
    step_time = pd / rate_d + pt / rate_t
    spread = max((max(td) - min(td)) / med(td), (max(tt) - min(tt)) / med(tt))
    return {
        'value': (pd + pt) / step_time / 1e6,
        'dwt_mpix_s': rate_d / 1e6,
        'dtcwt_mpix_s': rate_t / 1e6,
        'spread': spread,
        'cores': cores,
        'sample': 'DWT %dx%dx%dx%d + DTCWT %dx%dx%dx%d, median of %d, weighted to the full step mix' % (
            (dwt_n,) + DWT_SHAPE[1:] + (dtcwt_n,) + DTCWT_SHAPE[1:] + (reps,)),
        'step_s': step_time,
        'sample_s': sum(td) + sum(tt),
    }


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    vals = []
    t0 = time.perf_counter()
    r = None
    for i in range(args.warmup + args.steps):
        r = cpu_sample(dwt_n=8, reps=3)
        if i >= args.warmup:
            vals.append(r)
        if time.perf_counter() - t0 > 120:  # keep the whole arm within a few minutes
            break
    if not vals:
        vals = [r]
    v = sorted(x['value'] for x in vals)[len(vals) // 2]
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'Mpix/s', 'n_gpus': args.gpus,
        'steps': len(vals), 'warmup': args.warmup, 'ms_per_step': 1e3 * sum(x['step_s'] for x in vals) / len(vals),
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, 1),
        'cpu_baseline': {'value': v, 'unit': 'Mpix/s', 'cores': vals[-1]['cores'], 'kind': 'port',
                         'sample': vals[-1]['sample'] + '; each step = one such sample, step time extrapolated',
                         'spread_within_step': max(x['spread'] for x in vals),
                         'spread_over_steps': (max(x['value'] for x in vals) - min(x['value'] for x in vals)) / v,
                         'dwt_mpix_s': vals[-1]['dwt_mpix_s'], 'dtcwt_mpix_s': vals[-1]['dtcwt_mpix_s']},
        'e2e': {'value': v, 'unit': 'Mpix/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'note': 'reference arm = CPU oracle port of the reference algorithm (oracle/wave_oracle.c, OpenMP over planes, '
                'all host threads of ONE host, whatever --gpus says); the reference is pure Python and cannot travel to '
                'the GPU box. The value is per host and is not multiplied by the GPU count.',
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {
        'workload': 'DWTForward(J=3,db4,symmetric) %dx32x512x512 + DTCWTForward(J=3,near_sym_a,qshift_a) '
                    '%dx3x1024x1024 fp32 per GPU (BASELINE configs[1]+configs[2])' % (args.dwt_batch, args.dtcwt_batch),
        'per_gpu_pixels': args.dwt_batch * 32 * 512 * 512 + args.dtcwt_batch * 3 * 1024 * 1024,
        'parallelism': 'batch-sharded replicas x%d, outputs rank-resident (a second timed leg adds the NCCL gather)' % world,
        'l2': 'inputs (>=5 GB per step) exceed the 126 MB L2; no explicit flush',
    }


# ------------------------------------------------------------------------------------------------------
# clocks sampler (pynvml)

class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, 'nvmlClocksEventReasonHwSlowdown', 0x8): 'hw_slowdown',
            getattr(nv, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40): 'hw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20): 'sw_thermal_slowdown',
            getattr(nv, 'nvmlClocksEventReasonSwPowerCap', 0x4): 'sw_power_cap',
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.005)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {'sm_mhz': (s[len(s) // 2] if s else None), 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(s)}


def bind_to_gpu_numa(index):
    """Pin this process (and the pinned host buffers it allocates afterwards) to the CPUs NVML reports as local to
    the GPU, so that the 8 ranks of a box do not all stream host memory through one socket."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = os.cpu_count() or 1
        words = (n + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * i + b for i, wd in enumerate(mask) for b in range(64) if (wd >> b) & 1 and 64 * i + b < n]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {'cpus': len(cpus), 'first': cpus[0], 'last': cpus[-1]}
    except Exception as exc:
        return {'error': repr(exc)[:120]}
    return None


# ------------------------------------------------------------------------------------------------------

def setup_dist(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback for the product path)')
    numa = bind_to_gpu_numa(local)
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    return torch, dist, world, rank, local, dev, numa


def timed(torch, fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


DUMP_CAP = 1 << 20   # elements per dumped array: the 8 arrays of a step stay under 64 MB


def dump_outputs(torch, out_dir, arrays):
    """Write each (name, tensor) as out_dir/<name>.npy in float32.  A tensor of at most DUMP_CAP elements is written
    whole, with its shape; a larger one as the 1-D array of DUMP_CAP of its elements, taken in flat (C) order at
    positions drawn without replacement by a generator seeded from the name, so that every run and every build with
    the same shapes samples the same elements."""
    import zlib
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays:
        t = t.detach()
        if t.numel() > DUMP_CAP:
            rng = np.random.default_rng(zlib.crc32(name.encode()))
            idx = np.sort(rng.choice(t.numel(), DUMP_CAP, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy().astype(np.float32))


def run_ours(args):
    torch, dist, world, rank, local, dev, numa = setup_dist(args)
    import pytorch_wavelets_b200 as pw
    from pytorch_wavelets_b200 import _ffi, parallel
    _ffi.lib()
    peak, peak_src = load_peaks()

    dshape = (args.dwt_batch,) + DWT_SHAPE[1:]
    tshape = (args.dtcwt_batch,) + DTCWT_SHAPE[1:]
    torch.manual_seed(1234 + rank)
    xd = torch.randn(dshape, device=dev)
    xt = torch.randn(tshape, device=dev)
    dwt = pw.DWTForward(J=3, wave='db4', mode='symmetric').to(dev)
    dtc = pw.DTCWTForward(J=3, biort='near_sym_a', qshift='qshift_a').to(dev)
    pix_d, pix_t = xd.numel(), xt.numel()
    warm = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for _ in range(warm):
            a, b = dwt(xd), dtc(xt)
        del a, b
    barrier()

    # -- timed region: the whole step, device events; per-call events through the FFI hook for the level table
    rec = _ffi.CallRecorder()
    sampler = ClockSampler(local)
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    barrier()
    with rec, torch.no_grad():
        ev[0].record()
        for _ in range(args.steps):
            a = dwt(xd)
        ev[1].record()
        for _ in range(args.steps):
            b = dtc(xt)
        ev[2].record()
    barrier()
    clocks = sampler.stop()
    t_d = ev[0].elapsed_time(ev[1]) / 1e3
    t_t = ev[1].elapsed_time(ev[2]) / 1e3
    calls = rec.summary()
    launches = rec.count
    kernels_per_step = 3 + 3   # DWT: pyramid level 1 + 2 streaming levels; DTCWT: 3 levels (see DESIGN.md section 4)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(torch, args.dump_outputs,
                     [('dwt_yl', a[0])] + [('dwt_yh%d' % j, h) for j, h in enumerate(a[1])] +
                     [('dtcwt_yl', b[0])] + [('dtcwt_yh%d' % j, h) for j, h in enumerate(b[1])])
    del a, b

    tt = torch.tensor([t_d + t_t, t_d, t_t], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_total, t_d, t_t = [float(v) for v in tt.tolist()]
    value = world * (pix_d + pix_t) * args.steps / t_total / 1e6
    alg_d = dwt_alg_bytes(dshape[0] * dshape[1], 512, 512, 8, 3)
    alg_t = 4.0 * tshape[0] * tshape[1] * (1024 * 1024 * (1 + 3 + 0.75 + 0.1875) + 256 * 256)
    parts = {
        'dwt_fwd': {'ms': 1e3 * t_d / args.steps, 'mpix_s': world * pix_d * args.steps / t_d / 1e6, 'alg_bytes': alg_d,
                    'GBps': alg_d * args.steps / t_d / 1e9, 'frac': alg_d * args.steps / t_d / 1e9 / peak},
        'dtcwt_fwd': {'ms': 1e3 * t_t / args.steps, 'mpix_s': world * pix_t * args.steps / t_t / 1e6, 'alg_bytes': alg_t,
                      'GBps': alg_t * args.steps / t_t / 1e9, 'frac': alg_t * args.steps / t_t / 1e9 / peak},
    }

    # -- roofline of the dominant kernel: the level-1 pyramid kernel, timed alone as DWTForward(J=1) (= one launch)
    roof = None
    # The J = 1 launch writes 4.4 GB of freshly allocated outputs per call; its time depends on where those land (1.55 ms in
    # most processes / batches, up to 1.64 ms in others, with the J = 3 step time unchanged: profiles/r02_notes.md).  The cache is
    # emptied first so that the placement is the first-call one, and the median of five batches is reported with all five.
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    with torch.no_grad():
        dwt1 = pw.DWTForward(J=1, wave='db4', mode='symmetric').to(dev)
        # five batches of >= 10 launches; the median batch average is reported (one transiently slow batch -- seen once in
        # ~10 runs: 1.65 vs 1.55 ms with clean clocks -- must not decide the headline fraction) and all five are kept
        t1_batches = [timed(torch, lambda: dwt1(xd), max(10, args.steps // 2), warm=3 if i == 0 else 1) / 1e3 for i in range(5)]
        t1 = sorted(t1_batches)[2]
    alg1 = dwt_alg_bytes(dshape[0] * dshape[1], 512, 512, 8, 1)
    # secondary (SURVEY 8(d)): the traffic of a one-pass-per-level design, i.e. the algorithmic bytes plus every inter-level
    # low-pass written once and read once (DWT: 259^2 and 133^2 per plane; DTCWT: 1024^2 and 512^2 per plane)
    design_d = alg_d + 2 * 4.0 * dshape[0] * dshape[1] * (259 * 259 + 133 * 133)
    design_t = alg_t + 2 * 4.0 * tshape[0] * tshape[1] * (1024 * 1024 + 512 * 512)
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
        if args.dwt_batch == DWT_SHAPE[0]:
            traffic = tj.get('dwt_pyramid 512x512 L8 J1', {}).get('dram_bytes_per_launch')
    except Exception:
        pass
    roof = {'bound': 'hbm', 'kernel': 'dwt_pyramid<8> (level 1 of DWTForward: TMA row loads, bulk stores), %dx512x512' % (dshape[0] * 32),
            'achieved': alg1 / t1 / 1e9, 'peak': peak, 'unit': 'GB/s', 'frac': alg1 / t1 / 1e9 / peak, 'traffic': traffic,
            'peak_source': peak_src, 'alg_bytes_per_launch': alg1, 'avg_launch_ms': 1e3 * t1,
            'launch_ms_batches': [round(1e3 * t, 4) for t in t1_batches],
            'share_of_step': t1 * args.steps / (t_d + t_t),
            'whole_transform': {'dwt_fwd_GBps': parts['dwt_fwd']['GBps'], 'dwt_frac': parts['dwt_fwd']['frac'],
                                'dtcwt_fwd_GBps': parts['dtcwt_fwd']['GBps'], 'dtcwt_frac': parts['dtcwt_fwd']['frac'],
                                'per_level_design': {
                                    'note': 'algorithmic bytes + each inter-level low-pass written and read once (the '
                                            'traffic of a one-pass-per-level design); frac = of the measured HBM peak',
                                    'dwt_bytes': design_d, 'dwt_frac': design_d / parts['dwt_fwd']['ms'] / 1e6 / peak,
                                    'dtcwt_bytes': design_t,
                                    'dtcwt_frac': design_t / parts['dtcwt_fwd']['ms'] / 1e6 / peak}},
            'calls': {k: {'avg_ms': round(v['avg_ms'], 4), 'GBps': round(v['alg_bytes'] / v['avg_ms'] / 1e6, 1)}
                      for k, v in sorted(calls.items())}}

    # -- the other BASELINE configurations (N = 1 only: keeps the multi-GPU runs short)
    if world == 1 and not args.no_parts:
        with torch.no_grad():
            idwt = pw.DWTInverse(wave='db4', mode='symmetric').to(dev)
            c = dwt(xd)
            ms = timed(torch, lambda: idwt(c), 5)
            parts['dwt_inv'] = {'ms': ms, 'mpix_s': pix_d / ms / 1e3, 'alg_bytes': alg_d, 'GBps': alg_d / ms / 1e6,
                                'frac': alg_d / ms / 1e6 / peak}
            del c
            idtc = pw.DTCWTInverse(biort='near_sym_a', qshift='qshift_a').to(dev)
            c = dtc(xt)
            ms = timed(torch, lambda: idtc(c), 5)
            parts['dtcwt_inv'] = {'ms': ms, 'mpix_s': pix_t / ms / 1e3, 'alg_bytes': alg_t, 'GBps': alg_t / ms / 1e6,
                                  'frac': alg_t / ms / 1e6 / peak}
            del c
            xs = torch.randn(SCAT_SHAPE, device=dev)
            sc = torch.nn.Sequential(pw.ScatLayer(), pw.ScatLayer()).to(dev)
            ms = timed(torch, lambda: sc(xs), 10)
            alg_s = 4.0 * SCAT_SHAPE[0] * (3 * 256 * 256 + 2 * 21 * 128 * 128 + 147 * 64 * 64)
            parts['scat2_c4'] = {'ms': ms, 'mpix_s': xs.numel() / ms / 1e3, 'alg_bytes': alg_s, 'GBps': alg_s / ms / 1e6,
                                 'frac': alg_s / ms / 1e6 / peak, 'shape': list(SCAT_SHAPE)}
            del xs
            x5 = torch.randn(C5_CHUNK, device=dev)
            f5 = pw.DWTForward(J=4, wave='db8', mode='zero').to(dev)
            ms = timed(torch, lambda: f5(x5), 5)
            alg_5 = dwt_alg_bytes(C5_CHUNK[0] * C5_CHUNK[1], 2048, 2048, 16, 4)
            # fp32 FMAs of the separable banks: per level, per output position 2 rows x 2 filters x L (W pass) + 4 x L (H pass)
            fma = 0.0
            h = w = 2048
            for _ in range(4):
                h, w = (h + 15) // 2, (w + 15) // 2
                fma += C5_CHUNK[0] * C5_CHUNK[1] * h * w * 8 * 16
            parts['c5_shard_fwd'] = {'ms': ms, 'mpix_s': x5.numel() / ms / 1e3, 'alg_bytes': alg_5, 'GBps': alg_5 / ms / 1e6,
                                     'frac': alg_5 / ms / 1e6 / peak, 'fp32_tflops': 2 * fma / ms / 1e9,
                                     'shape': list(C5_CHUNK), 'note': 'per-GPU chunk of configs[4]; --config c5 runs the sharded job'}
            del x5

    # -- N > 1: the same step followed by the single NCCL gather of every output tensor
    gather = None
    if world > 1 and not args.no_gather:
        try:
            gsteps = min(args.steps, 5)
            try:     # the C ABI's own NCCL communicator; torch.distributed's NCCL group if it cannot be created
                comm = parallel.Communicator.from_torch_distributed()
                transport = 'b200w_allgather (C ABI, NCCL communicator created with b200w_comm_init)'
            except Exception as exc:
                comm, transport = None, 'torch.distributed.all_gather (NCCL); C-ABI communicator unavailable: %r' % (exc,)
            with torch.no_grad():
                out = parallel.gather_pyramid(dwt(xd), world * dshape[0], comm=comm)
                out2 = parallel.gather_pyramid(dtc(xt), world * tshape[0], comm=comm)
                gbytes = sum(t.numel() * 4 for t in [out[0]] + list(out[1])) + sum(t.numel() * 4 for t in [out2[0]] + list(out2[1]))
                del out, out2
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(gsteps):
                    o1 = parallel.gather_pyramid(dwt(xd), world * dshape[0], comm=comm)
                    o2 = parallel.gather_pyramid(dtc(xt), world * tshape[0], comm=comm)
                    del o1, o2
                e1.record()
                barrier()
            tg = torch.tensor([e0.elapsed_time(e1) / 1e3], device=dev, dtype=torch.float64)
            dist.all_reduce(tg, op=dist.ReduceOp.MAX)
            tg = float(tg.item())
            t_coll = tg / gsteps - t_total / args.steps
            recv = gbytes * (world - 1) / world
            gather = {'value_with_gather': world * (pix_d + pix_t) * gsteps / tg / 1e6, 'unit': 'Mpix/s',
                      'ms_per_step': 1e3 * tg / gsteps, 'collective': 'NCCL all_gather of yl and every yh[j], both transforms',
                      'transport': transport,
                      'gathered_bytes_per_rank': gbytes, 'received_bytes_per_rank': recv,
                      'collective_ms': 1e3 * t_coll, 'recv_GBps_per_rank': recv / max(t_coll, 1e-9) / 1e9, 'steps': gsteps}
        except Exception as exc:
            gather = {'error': repr(exc)[:200]}

    # -- end to end through the public API with HOST buffers (pinned), H2D + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        try:
            e2e = run_e2e(torch, dist, pw, dev, world, dshape, tshape, min(args.steps, 5))
            e2e['numa_binding'] = numa
        except Exception as exc:  # e.g. not enough pinnable host memory for N ranks: report, do not lose the line
            e2e = {'value': None, 'unit': 'Mpix/s', 'error': repr(exc)[:200]}
            if world > 1:
                try:
                    dist.barrier()
                except Exception:
                    pass

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        c = cpu_sample()
        cpu = {'value': c['value'], 'unit': 'Mpix/s', 'cores': c['cores'], 'kind': 'port', 'sample': c['sample'],
               'spread': c['spread'], 'dwt_mpix_s': c['dwt_mpix_s'], 'dtcwt_mpix_s': c['dtcwt_mpix_s'],
               'sample_seconds': c['sample_s']}

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': 'Mpix/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': warm, 'ms_per_step': 1e3 * t_total / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args, world), 'parts': parts, 'roofline': roof, 'cpu_baseline': cpu,
            'e2e': e2e, 'gather': gather, 'clocks': clocks,
            'gpu_launches': kernels_per_step * args.steps, 'abi_calls': launches,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(torch, dist, pw, dev, world, dshape, tshape, steps):
    """Same step through the public nn.Module API, inputs in pinned host memory, every output copied back to
    pinned host memory, all inside the timed region.  The batch is processed in chunks on three streams
    (H2D / compute / D2H) so copies overlap compute; PCIe is the bound."""
    from pytorch_wavelets_b200 import pipeline
    dwt = pw.DWTForward(J=3, wave='db4', mode='symmetric').to(dev)
    dtc = pw.DTCWTForward(J=3).to(dev)
    hd = torch.empty(dshape, pin_memory=True)
    ht = torch.empty(tshape, pin_memory=True)
    hd[:8].normal_()
    ht[:8].normal_()
    for i in range(8, hd.shape[0], 8):      # synthetic host data: a few random images repeated (cheap to generate)
        hd[i:i + 8].copy_(hd[:min(8, hd.shape[0] - i)])
    for i in range(8, ht.shape[0], 8):
        ht[i:i + 8].copy_(ht[:min(8, ht.shape[0] - i)])
    pd = pipeline.HostPipeline(dwt, hd.shape, dev, chunk=16)
    pt = pipeline.HostPipeline(dtc, ht.shape, dev, chunk=8)
    for _ in range(2):
        pd.run(hd)
        pt.run(ht)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        pd.run(hd)
        pt.run(ht)
    t1.record()
    torch.cuda.synchronize()
    t = t0.elapsed_time(t1) / 1e3
    tt = torch.tensor([t], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t = float(tt.item())
    pix = hd.numel() + ht.numel()
    h2d, d2h = 4 * pix, pd.out_bytes + pt.out_bytes
    return {'value': world * pix * steps / t / 1e6, 'unit': 'Mpix/s',
            'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
            'ms_per_step': 1e3 * t / steps, 'steps': steps,
            'pcie_GBps_per_rank': {'h2d': h2d * steps / t / 1e9, 'd2h': d2h * steps / t / 1e9,
                                   'note': 'both directions overlap; each figure = bytes of that direction / wall time'},
            'how': 'pinned host in/out, chunked 3-stream pipeline through DWTForward/DTCWTForward.forward'}


# ------------------------------------------------------------------------------------------------------
# --config c5: BASELINE.json configs[4], sharded over N, chunk-streamed

def run_c5(args):
    torch, dist, world, rank, local, dev, numa = setup_dist(args)
    import pytorch_wavelets_b200 as pw
    from pytorch_wavelets_b200 import parallel
    peak, peak_src = load_peaks()
    lo, hi = parallel.shard_bounds(args.c5_n_total, world, rank)
    chunk = args.c5_chunk
    n_chunks = min((hi - lo + chunk - 1) // chunk, args.steps)     # a step = one chunk per GPU
    torch.manual_seed(100 + rank)
    x = torch.randn(chunk, 16, 2048, 2048, device=dev)
    f = pw.DWTForward(J=4, wave='db8', mode='zero').to(dev)
    sampler = ClockSampler(local)
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            f(x)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler.start()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        yls = []
        for _ in range(n_chunks):
            yl, yh = f(x)          # band-passes are consumed in place (rank-resident), the low-pass is kept
            yls.append(yl)
        e[1].record()
        ylr = torch.cat(yls, 0)
        if world > 1:
            ylg = parallel.gather_pyramid(ylr, world * ylr.shape[0])
        e[2].record()
        torch.cuda.synchronize()
    clocks = sampler.stop()
    t = torch.tensor([e[0].elapsed_time(e[1]) / 1e3, e[0].elapsed_time(e[2]) / 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_c, t_g = [float(v) for v in t.tolist()]
    pix = world * n_chunks * x.numel()
    alg = dwt_alg_bytes(chunk * 16, 2048, 2048, 16, 4) * n_chunks
    if rank == 0:
        print(json.dumps({
            'metric': 'Mpixels/sec DWTForward J=4 db8 (BASELINE configs[4])', 'value': pix / t_c / 1e6, 'unit': 'Mpix/s',
            'n_gpus': world, 'steps': n_chunks, 'warmup': max(args.warmup, 3), 'ms_per_step': 1e3 * t_c / n_chunks,
            'higher_is_better': True, 'scaling': 'strong (N=%d total) measured on the first %d chunk(s) of every shard' % (args.c5_n_total, n_chunks),
            'dtype': 'f32', 'data': 'synthetic', 'vs_baseline': None,
            'config': {'workload': 'DWTForward(J=4,db8,zero) N=%d C=16 2048x2048 sharded over N across %d GPU(s), chunks of %d images'
                                   % (args.c5_n_total, world, chunk), 'shard': [lo, hi], 'l2': 'chunk input 1.07 GB >> L2'},
            'value_with_gather': pix / t_g / 1e6, 'gather': 'NCCL all_gather of yl only (band-passes stay rank-resident: '
            'the full pyramid of configs[4] is 282 GB and fits no single GPU -- SURVEY 8(e))',
            'roofline': {'bound': 'hbm', 'achieved': alg / t_c / 1e9, 'peak': peak, 'unit': 'GB/s', 'frac': alg / t_c / 1e9 / peak,
                         'peak_source': peak_src, 'per_gpu': True, 'traffic': None}, 'clocks': clocks}), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------
# --impl aten: the reference's GPU op sequence, written independently from the closed forms of SURVEY section 8
# (extension by index gather, depthwise conv2d, slicing).  Not the product: the bar the product has to beat.

def run_aten(args):
    torch, dist, world, rank, local, dev, numa = setup_dist(args)
    import pytorch_wavelets_b200 as pw
    from tools.aten_arm import dwt_fwd, dtcwt_fwd

    dwt = pw.DWTForward(J=3, wave='db4', mode='symmetric').to(dev)
    dtc = pw.DTCWTForward(J=3).to(dev)
    f_lo, f_hi = dwt.h0_col.reshape(-1), dwt.h1_col.reshape(-1)
    taps = [getattr(dtc, n).reshape(-1) for n in ('h0o', 'h1o', 'h0a', 'h0b', 'h1a', 'h1b')]
    torch.manual_seed(1234 + rank)
    with torch.no_grad():
        # same operator? check against the product on a small batch before timing
        xs, xts = torch.randn(2, 32, 512, 512, device=dev), torch.randn(2, 3, 1024, 1024, device=dev)
        a, b = dwt_fwd(xs, f_lo, f_hi, 3), dwt(xs)
        err = max(float((a[0] - b[0]).abs().max()), max(float((p - q).abs().max()) for p, q in zip(a[1], b[1])))
        a, b = dtcwt_fwd(xts, *taps, 3), dtc(xts)
        err_t = max(float((a[0] - b[0]).abs().max()), max(float((p - q).abs().max()) for p, q in zip(a[1], b[1])))
        assert err < 1e-4 and err_t < 1e-3, ('aten arm computes a different operator', err, err_t)
        del a, b, xs, xts
        # ATen materialises several full-size intermediates: run the batch in slices that fit comfortably
        db, tb = 32, 16
        xd = torch.randn((db,) + DWT_SHAPE[1:], device=dev)
        xt = torch.randn((tb,) + DTCWT_SHAPE[1:], device=dev)
        nd, nt = args.dwt_batch // db, args.dtcwt_batch // tb

        def step():
            for _ in range(nd):
                dwt_fwd(xd, f_lo, f_hi, 3)
            for _ in range(nt):
                dtcwt_fwd(xt, *taps, 3)
        steps = min(args.steps, 5)
        ms = timed(torch, step, steps, warm=max(2, min(args.warmup, 3)))
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    pix = args.dwt_batch * 32 * 512 * 512 + args.dtcwt_batch * 3 * 1024 * 1024
    if rank == 0:
        print(json.dumps({'impl': 'aten', 'metric': METRIC, 'value': world * pix / ms / 1e3, 'unit': 'Mpix/s', 'n_gpus': world,
                          'steps': steps, 'ms_per_step': ms, 'higher_is_better': True, 'dtype': 'f32', 'data': 'synthetic',
                          'config': workload_config(args, world), 'max_abs_diff_vs_product': {'dwt': err, 'dtcwt': err_t},
                          'note': 'depthwise F.conv2d + index_select extension + slicing on the same B200 (the op sequence of '
                                  'the reference GPU path, re-derived from the closed forms); batch processed in slices of '
                                  '%d / %d images to bound ATen\'s intermediates' % (db, tb)}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    elif a.impl == 'aten':
        run_aten(a)
    elif a.config == 'c5':
        run_c5(a)
    else:
        run_ours(a)
