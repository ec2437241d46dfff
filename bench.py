#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE config 2.

    metric   leapfrog-steps x chains / sec   (plain HMC, D-dim isotropic Gaussian)
    workload config 2: D=1024 isotropic N(0,I), 256 chains per GPU, L=10, eps=0.05, S=1000 iterations, burn=0
    step     one pass of the hot path over one batch: ONE persistent-kernel launch advancing all chains of the rank
             through all S iterations (gibbs -> H -> L leapfrog steps -> H -> MH -> sample write), = C*S*L chain-steps

    python bench.py --gpus N --steps K --warmup W            (under torchrun for N > 1: one rank per GPU)
    python bench.py ... --dump-outputs DIR                    (+ the last timed step's outputs as DIR/<name>.npy)
    python bench.py --impl reference ...                      (the reference's algorithm on the host cores)

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import ctypes
import gc
import json
import os
import signal
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

D, C_PER_GPU, S, L, EPS = 1024, 256, 1000, 10, 0.05
WARP_INST_PER_LAUNCH = 836294520           # config 2, E=4 K=1 geometry: ncu smsp__inst_executed.sum of one launch
                                           # (profiles/r2_prof_hmc_run.summary.txt; 1076063104 before the packed fp32x2 leapfrog)
METRIC = 'leapfrog-steps x chains / sec'
UNIT = 'chain-steps/s'
REFERENCE_ARM_BUDGET_S = 75.0              # wall-clock bound of `--impl reference` whatever --steps says


def workload_config(world):
    """The `config` object BOTH arms report, key for key: BASELINE config 2."""
    return {'workload': 'BASELINE config 2: D=1024 isotropic Gaussian, plain HMC, 256 chains/GPU, L=10, '
                        'eps=0.05, S=1000 iterations per step',
            'chains_per_gpu': C_PER_GPU, 'dim': D, 'L': L, 'iterations_per_step': S,
            'parallelism': 'chains sharded over %d GPU(s), no data-path collective; one all-gather collects the samples'
                           % world}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return json.load(f)
    except Exception:
        return {}


def measured_peak_hbm():
    p = measured_peaks()
    if 'hbm_gbs' in p:
        return float(p['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


# ----------------------------------------------------------------------------------------------------------
# host topology: usable logical CPUs, physical cores, cgroup quota, NUMA node of a GPU
# ----------------------------------------------------------------------------------------------------------
def host_cpus():
    """{'logical': CPUs this process may run on, 'physical_cores': distinct (socket, core) pairs among them,
    'cgroup_quota': CPUs' worth of cgroup cpu.max quota or None, 'workers': processes the CPU arm starts}."""
    try:
        usable = sorted(os.sched_getaffinity(0))
    except Exception:
        usable = list(range(os.cpu_count() or 1))
    phys = set()
    try:
        cpu = pid = cid = None
        with open('/proc/cpuinfo') as f:
            for ln in f.read().splitlines() + ['']:
                if ln.startswith('processor'):
                    cpu = int(ln.split(':')[1])
                elif ln.startswith('physical id'):
                    pid = int(ln.split(':')[1])
                elif ln.startswith('core id'):
                    cid = int(ln.split(':')[1])
                elif not ln.strip():
                    if cpu is not None and cpu in usable and pid is not None and cid is not None:
                        phys.add((pid, cid))
                    cpu = pid = cid = None
    except Exception:
        pass
    quota = None
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            q, per = f.read().split()
            if q != 'max':
                quota = float(q) / float(per)
    except Exception:
        pass
    workers = len(usable)
    if quota:
        workers = max(1, min(workers, int(quota + 0.5)))
    return {'logical': len(usable), 'physical_cores': len(phys) or None, 'cgroup_quota': quota, 'workers': workers}


def _parse_cpulist(txt):
    cpus = set()
    for part in txt.strip().split(','):
        if not part:
            continue
        if '-' in part:
            a, b = part.split('-')
            cpus.update(range(int(a), int(b) + 1))
        else:
            cpus.add(int(part))
    return cpus


def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and therefore every page it first-touches, pinned host blocks included) to the NUMA node its
    GPU hangs off: CPU affinity = the node's cpulist, memory policy = MPOL_PREFERRED that node.  Must run BEFORE the
    first pinned allocation.  Returns a small dict for the bench line; never raises."""
    info = {'bound': False}
    try:
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        idx = local_rank
        if vis:
            ids = [v.strip() for v in vis.split(',') if v.strip()]
            if local_rank < len(ids) and ids[local_rank].isdigit():
                idx = int(ids[local_rank])
        h = nv.nvmlDeviceGetHandleByIndex(idx)
        bdf = nv.nvmlDeviceGetPciInfo(h).busId
        bdf = (bdf.decode() if isinstance(bdf, bytes) else bdf).lower()
        if len(bdf.split(':')[0]) == 8:                       # NVML prints an 8-digit domain, sysfs uses 4
            bdf = bdf[4:]
        with open('/sys/bus/pci/devices/%s/numa_node' % bdf) as f:
            node = int(f.read())
        info['pci'] = bdf
        if node < 0:
            info['node'] = None
            return info
        with open('/sys/devices/system/node/node%d/cpulist' % node) as f:
            cpus = _parse_cpulist(f.read())
        allowed = cpus & set(os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
        info.update(node=node, cpus=len(allowed), bound=bool(allowed))
        # set_mempolicy(MPOL_PREFERRED, {node}): x86_64 syscall 238; harmless if refused (first touch under the CPU
        # affinity above already allocates locally)
        try:
            libc = ctypes.CDLL(None, use_errno=True)
            mask = (ctypes.c_ulong * 16)()
            mask[node // 64] = 1 << (node % 64)
            rc = libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(16 * 64))
            info['mempolicy'] = 'preferred' if rc == 0 else 'refused (errno %d)' % ctypes.get_errno()
        except Exception as e:                                # pragma: no cover
            info['mempolicy'] = 'unavailable: %s' % e
    except Exception as e:
        info['error'] = str(e)[:120]
    return info


_HUGE_KEEP = []


def pinned_host_block(shape):
    """The page-locked host block the e2e legs copy / stream the samples into.  BENCH_HUGEPAGES=1: an anonymous mapping
    advised to transparent huge pages (2 MiB), first-touched under the NUMA policy above and registered with
    cudaHostRegister -- fewer IOMMU translations per byte of device-to-host DMA than 4 KiB pages when several GPUs write
    into one socket's memory.  Falls back to torch's pin_memory().  Returns (tensor, description)."""
    import math
    n = int(math.prod(shape)) * 4
    if os.environ.get('BENCH_HUGEPAGES', '0') == '1':
        try:
            import mmap
            size = (n + (1 << 21) - 1) & ~((1 << 21) - 1)
            mm = mmap.mmap(-1, size + (1 << 21), flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS)
            base = ctypes.addressof(ctypes.c_char.from_buffer(mm))
            off = (-base) & ((1 << 21) - 1)
            libc = ctypes.CDLL(None, use_errno=True)
            libc.madvise.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
            rc = libc.madvise(ctypes.c_void_p(base + off), size, 14)                    # MADV_HUGEPAGE
            t = torch.frombuffer(mm, dtype=torch.float32, count=n // 4, offset=off).view(shape)
            t.zero_()                                                                   # first touch (NUMA policy applies)
            err = torch.cuda.cudart().cudaHostRegister(t.data_ptr(), n, 0)
            if int(err) != 0 or not t.is_pinned():
                raise RuntimeError('cudaHostRegister -> %s' % err)
            _HUGE_KEEP.append(mm)
            return t, 'mmap + MADV_HUGEPAGE (rc %d) + cudaHostRegister' % rc
        except Exception as e:                                  # pragma: no cover
            sys.stderr.write('BENCH_HUGEPAGES: falling back to pin_memory(): %s\n' % e)
    return torch.empty(shape, dtype=torch.float32).pin_memory(), 'torch pin_memory() (cudaHostAlloc)'


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port: same Python loop + autograd as hamiltorch.sample) on host cores
# ----------------------------------------------------------------------------------------------------------
def _cpu_chain(args):
    seed, n_iter = args
    import torch as _t
    _t.set_num_threads(1)
    from hamiltorch_b200 import targets as T
    from oracle import hmc_oracle as O
    tgt = T.GaussianIso(D)
    _t.manual_seed(seed)
    init = 0.1 * _t.randn(D)
    t0 = time.perf_counter()
    O.sample_hmc(tgt, init, num_samples=n_iter, num_steps_per_sample=L, step_size=EPS)
    return time.perf_counter() - t0


class CpuArm:
    """One pool of worker processes (one per usable CPU, 1 torch thread each -- intra-op threads do not help at D=1024,
    BASELINE.md section 3), created ONCE and reused for every step.  A step = every worker runs `n_iter` iterations of
    one independent config-2 chain through the reference's per-chain Python loop."""

    def __init__(self, workers):
        import multiprocessing as mp
        self.workers = workers
        self.pool = mp.get_context('fork').Pool(workers)
        self.k = 0

    def step(self, n_iter):
        t0 = time.perf_counter()
        self.pool.map(_cpu_chain, [(1000 + self.k * self.workers + i, n_iter) for i in range(self.workers)], chunksize=1)
        self.k += 1
        return time.perf_counter() - t0

    def close(self):
        self.pool.terminate()
        self.pool.join()


def cpu_sample_text(host, n_iter, steps_done):
    return ('%d independent chains (1 per usable CPU; %s physical cores, %d logical%s) x %d iterations x L=%d of '
            'config 2 per step, %d step(s)' % (host['workers'], host['physical_cores'] or '?', host['logical'],
                                               (', cgroup quota %.1f' % host['cgroup_quota']) if host['cgroup_quota'] else '',
                                               n_iter, L, steps_done))


def cpu_baseline_quick(budget_s=12.0):
    """The cpu_baseline leg of the B200 arm: a bounded sample, forked BEFORE this process touches CUDA."""
    host = host_cpus()
    arm = CpuArm(host['workers'])
    try:
        arm.step(2)                                           # page the workers in
        t_cal = arm.step(20)                                  # calibration
        n_iter = int(max(50, min(2000, 20 * (budget_s / max(t_cal, 1e-3)))))
        wall = arm.step(n_iter)
    finally:
        arm.close()
    rate = host['workers'] * n_iter * L / wall
    return {'value': rate, 'unit': UNIT, 'cores': host['workers'], 'physical_cores': host['physical_cores'],
            'logical_cpus': host['logical'], 'cgroup_quota': host['cgroup_quota'], 'kind': 'port',
            'sample': cpu_sample_text(host, n_iter, 1) + ', %.1f s wall' % wall}


def run_reference_arm(args, rank, world):
    """`--impl reference`: the oracle port on all usable host CPUs, bounded to REFERENCE_ARM_BUDGET_S of wall clock
    whatever --steps / --warmup say (the driver gives this arm a per-N time slot): the per-step sample size is chosen
    from a calibration step so that warm-up + K steps fit, the JSON line is also printed if the run is cut short
    (SIGTERM / SIGINT) with the steps completed so far."""
    if rank != 0:
        return
    t_start = time.perf_counter()
    host = host_cpus()
    arm = CpuArm(host['workers'])
    state = {'t': 0.0, 'steps': 0, 'n_iter': 0, 'printed': False}

    def emit(cut_short=False):
        if state['printed']:
            return
        state['printed'] = True
        steps_done = max(state['steps'], 1)
        n_iter = max(state['n_iter'], 1)
        t_tot = state['t'] if state['steps'] else max(time.perf_counter() - t_start, 1e-9)
        value = (host['workers'] * n_iter * L * state['steps'] / t_tot) if state['steps'] else 0.0
        sample = cpu_sample_text(host, n_iter, state['steps'])
        cfg = workload_config(args.gpus)
        line = {
            'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * t_tot / steps_done,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            # identical to the B200 arm's `config`; what a reference step is lives in cpu_baseline.sample (independent
            # chains of config 2 through the reference's per-chain Python loop; the rate is per chain-step, so it
            # extrapolates linearly to the full 256 x 1000 job)
            'config': cfg,
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': host['workers'],
                             'physical_cores': host['physical_cores'], 'logical_cpus': host['logical'],
                             'cgroup_quota': host['cgroup_quota'], 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'steps_completed': state['steps'], 'cut_short': bool(cut_short),
            'wall_s': time.perf_counter() - t_start,
        }
        print(json.dumps(line), flush=True)

    def on_term(signum, frame):
        emit(cut_short=True)
        try:
            arm.pool.terminate()
        finally:
            os._exit(0)

    signal.signal(signal.SIGTERM, on_term)
    signal.signal(signal.SIGINT, on_term)
    try:
        arm.step(2)                                           # page the workers in (imports, first autograd call)
        t_cal = arm.step(10)                                  # calibration
        budget = max(5.0, REFERENCE_ARM_BUDGET_S - (time.perf_counter() - t_start) - 3.0)
        per_step = budget / (args.steps + (1 if args.warmup > 0 else 0))
        n_iter = args.cpu_iters if args.cpu_iters > 0 else int(max(4, min(2000, 10 * per_step / max(t_cal, 1e-3))))
        state['n_iter'] = n_iter
        if args.warmup > 0:
            arm.step(n_iter)
        for _ in range(args.steps):
            state['t'] += arm.step(n_iter)
            state['steps'] += 1
            if time.perf_counter() - t_start > REFERENCE_ARM_BUDGET_S + 15.0:
                break                                         # a box slower than its calibration step: stop early
        emit(cut_short=state['steps'] < args.steps)
    finally:
        arm.close()


# ----------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM / memory clock + throttle reasons sampled every 20 ms while the timed regions run.  In-process NVML
    (nvidia_ml_py) on a daemon thread: one nvmlInit before the warm-up, then ~50 us queries -- no subprocess attaching to
    the driver while kernels are being launched (an `nvidia-smi -lms` loop did stall launches for milliseconds now and
    then).  Falls back to that loop only if NVML cannot be imported."""
    REASONS = (('hw_slowdown', 'nvmlClocksEventReasonHwSlowdown'),
               ('hw_thermal_slowdown', 'nvmlClocksEventReasonHwThermalSlowdown'),
               ('sw_thermal_slowdown', 'nvmlClocksEventReasonSwThermalSlowdown'),
               ('sw_power_cap', 'nvmlClocksEventReasonSwPowerCap'))
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc, self.thread = index, None, None
        self.sm, self.mem, self.mx, self.reasons, self.stop_flag = [], [], [], set(), False

    def _visible_index(self):
        vis = os.environ.get('CUDA_VISIBLE_DEVICES')
        if vis:
            ids = [v.strip() for v in vis.split(',') if v.strip()]
            if self.index < len(ids) and ids[self.index].isdigit():
                return int(ids[self.index])
        return self.index

    def _loop(self, nv, h):
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mem.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_MEM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for name, const in self.REASONS:
                    if r & getattr(nv, const):
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self._visible_index())
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)))
            self.thread = threading.Thread(target=self._loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            sm, mem = sorted(self.sm), sorted(self.mem)
            return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(self.mx) if self.mx else None,
                    'mem_mhz': mem[len(mem) // 2] if mem else None,
                    'reasons': sorted(self.reasons), 'samples': len(sm), 'source': 'nvml'}
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ''
        sm, mx, reasons = [], [], set()
        names = [n for n, _ in self.REASONS]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm), 'source': 'nvidia-smi'}


# ----------------------------------------------------------------------------------------------------------
# BASELINE configs 3, 4, 5 on this rank's GPU (reported under `other_configs`; config 2 is the headline)
# ----------------------------------------------------------------------------------------------------------
def _event_timed(fn, reps):
    """Device time per call of `fn` (a public-API call that enqueues its work and returns): CUDA events around `reps` calls
    enqueued BEHIND a spinning head-start kernel, so that the host's per-call overhead (0.5-1 ms of Python, more on a
    loaded box: config 5's launch is 0.5 ms) runs ahead of the GPU instead of showing up as idle time between the events."""
    w1 = fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    w2 = fn()                                                # host-side cost of one call
    host_s = time.perf_counter() - t0
    torch.cuda.synchronize()
    # both warm-up results were alive at once: the caching allocator now holds TWO blocks of every size a call allocates, so
    # the timed `r = fn()` sequence (previous result alive while the next call allocates) never reaches cudaMalloc -- which
    # synchronises with the head-start kernel (measured: 31 ms per call instead of 0.4)
    del w1, w2
    head_s = min(0.2, 1.5 * reps * host_s + 2e-3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(int(head_s * 1.9e9))                   # ~head_s of SM-clock spinning on the stream
    e0.record()
    r = None
    for _ in range(reps):
        r = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, r


def other_configs(dev, rank, world):
    """One device-timed launch (after one warm-up launch) of BASELINE configs 3, 4 and 5 with this rank's share of the
    chains, in-kernel Philox, inputs resident in HBM.  Returns {name: {...}} with per-rank chain-steps/s; the caller
    sums over ranks.  Each entry names its kernel and the roofline that bounds it."""
    import torch.nn as nn
    import hamiltorch_b200 as hb
    from hamiltorch_b200 import targets as T
    out = {}
    peaks = measured_peaks()
    # ---- config 3: explicit RMHMC, 2-D funnel, softabs 1e6, omega 10, 512 chains per GPU, L=10, eps=.05, S=200 ----
    C3, S3 = 512, 200
    init3 = torch.tensor([0., 1.], device=dev).repeat(C3, 1)
    ms, res = _event_timed(lambda: hb.sample_chains(
        T.Funnel(2), init3, num_samples=S3, num_steps_per_sample=10, step_size=0.05, jitter=1e-3, softabs_const=1e6,
        explicit_binding_const=10, sampler=hb.Sampler.RMHMC, integrator=hb.Integrator.EXPLICIT,
        metric=hb.Metric.SOFTABS, rng='philox', seed=2, chain_offset=rank * C3), reps=3)
    out['config3'] = {'workload': 'explicit RMHMC, 2-D funnel, softabs 1e6, omega=10, jitter 1e-3, 512 chains/GPU, '
                                  'L=10, eps=0.05, S=200', 'kernel': 'rmhmc2_quad_kernel', 'bound': 'latency (serial recurrence of 3L+3 stages)',
                      'kernel_ms': ms, 'value': C3 * S3 * 10 / (ms * 1e-3), 'unit': UNIT,
                      'accept_rate': float(res.accepted.float().mean()),
                      'log_prob_error_rate': float(res.diverged.float().mean())}
    # ---- config 4: Linear(64,128)-ReLU-Linear(128,1) BNN (D=8449), N=1024 in M=4 splits, symmetric split HMC,
    #      64 chains over 8 GPUs = 8 per GPU (all 64 on one GPU when world == 1), L=10, eps=5e-4, S=300 ----
    C4 = 64 if world == 1 else max(1, 64 // world)
    S4 = 300
    g = torch.Generator().manual_seed(0)
    X = torch.randn(1024, 64, generator=g)
    w = torch.randn(64, 1, generator=g)
    y = torch.sin(X @ w / 8) + 0.1 * torch.randn(1024, 1, generator=g)
    torch.manual_seed(0)
    model = nn.Sequential(nn.Linear(64, 128), nn.ReLU(), nn.Linear(128, 1))
    descs = [T.MLPRegression.from_model(model, X[m * 256:(m + 1) * 256], y[m * 256:(m + 1) * 256], None, 100.,
                                        prior_scale=4) for m in range(4)]
    D4 = descs[0].dim
    init4 = (hb.util.flatten(model).detach()[None] + 0.01 * torch.randn(C4, D4, generator=g)).to(dev)
    ones = torch.ones(D4)
    ms, res = _event_timed(lambda: hb.sample_chains(
        descs, init4, num_samples=S4, num_steps_per_sample=10, step_size=5e-4, inv_mass=ones,
        integrator=hb.Integrator.SPLITTING, rng='philox', seed=3, chain_offset=rank * C4), reps=1)
    flops = 68.7e6 * C4 * S4 * 10                        # SURVEY 8d: 68.7 MFLOP per chain-step
    tf = flops / (ms * 1e-3) / 1e12
    peak_tc = float(peaks.get('bf16_tflops_sustained', 2250.0)) / 6.0      # tf32 = bf16/2, 3 UMMAs per product
    out['config4'] = {'workload': 'BNN 64-128-1 (D=8449) regression, N=1024, M=4 symmetric split HMC, %d chains/GPU, '
                                  'L=10, eps=5e-4, S=300' % C4, 'kernel': 'mlp_run_kernel (tcgen05 3xTF32)',
                      'bound': 'tensor', 'kernel_ms': ms, 'value': C4 * S4 * 10 / (ms * 1e-3), 'unit': UNIT,
                      'algorithmic_tflops': tf, 'roofline_frac': tf / peak_tc, 'roofline_peak_tflops': peak_tc,
                      'accept_rate': float(res.accepted.float().mean())}
    # ---- config 5: HMC_NUTS step-size adaptation, D=4096 isotropic Gaussian, 1024 chains over 8 GPUs = 128 per GPU,
    #      L=10, eps0=0.1, burn=100, S=150 ----
    C5, D5, S5, B5 = 128, 4096, 150, 100
    init5 = (0.1 * torch.randn(C5, D5, generator=g)).to(dev)
    ms, res = _event_timed(lambda: hb.sample_chains(
        T.GaussianIso(D5), init5, num_samples=S5, num_steps_per_sample=10, step_size=0.1, burn=B5,
        sampler=hb.Sampler.HMC_NUTS, rng='philox', seed=1, chain_offset=rank * C5), reps=3)
    out['config5'] = {'workload': 'HMC_NUTS (dual averaging), D=4096 isotropic Gaussian, 128 chains/GPU, L=10, '
                                  'eps0=0.1, burn=100, S=150', 'kernel': 'hmc_run_kernel<ISO,NONE,NUTS=1>',
                      'bound': 'issue/latency (HBM traffic = retained samples only)', 'kernel_ms': ms,
                      'note': 'kernel_ms = device time of the whole public-API call (its memsets / copies + the launch), host '
                              'overhead hidden behind a head-start kernel',
                      'value': C5 * S5 * 10 / (ms * 1e-3), 'unit': UNIT,
                      'median_adapted_step_size': float(res.step_size.median()),
                      'post_burn_accept_rate': float(res.accepted[:, B5 + 1:].float().mean())}
    # ---- SURVEY 8d's "D=64 Gaussian-Hessian variant" of config 3: explicit RMHMC with the metric solve as a dense
    #      contraction, 512 chains per GPU, dense-precision Gaussian, L=10, S=200 -- the persistent small-D flow kernel ----
    C6, D6, S6 = 512, 64, 200
    A6 = torch.randn(D6, D6, generator=g, dtype=torch.float64) / D6 ** 0.5
    tgt6 = T.GaussianFull(torch.zeros(D6), cov=A6 @ A6.t() + 0.5 * torch.eye(D6, dtype=torch.float64))
    init6 = (0.5 * torch.randn(C6, D6, generator=g)).to(dev)
    ms, res = _event_timed(lambda: hb.sample_chains(
        tgt6, init6, num_samples=S6, num_steps_per_sample=10, step_size=0.1, explicit_binding_const=10,
        sampler=hb.Sampler.RMHMC, integrator=hb.Integrator.EXPLICIT, metric=hb.Metric.HESSIAN, rng='philox', seed=4,
        chain_offset=rank * C6), reps=3)
    sm_clk = float(peaks.get('sm_max_mhz', 1965.0)) * 1e6
    smem_peak = torch.cuda.get_device_properties(dev).multi_processor_count * 128.0 * sm_clk / 1e9     # GB/s
    mv_bytes = C6 * S6 * (6 * 10 + 4) * D6 * D6 * 4.0      # every warp-matvec streams the D x D matrix once (R = 1 chain per warp)
    out['rmhmc_dense_metric_d64'] = {
        'workload': 'explicit RMHMC, constant dense metric (Gaussian-Hessian variant of config 3, SURVEY 8d), D=64, '
                    '512 chains/GPU, L=10, eps=0.1, S=200', 'kernel': 'flow_small_kernel<2,1> (one launch per run)',
        'bound': 'shared-memory bandwidth (matrices resident in smem; 128 B/clk/SM)', 'kernel_ms': ms,
        'note': 'kernel_ms = device time of the whole public-API call (metric factorisation cached per target)',
        'value': C6 * S6 * 10 / (ms * 1e-3), 'unit': UNIT, 'smem_gbs': mv_bytes / (ms * 1e-3) / 1e9,
        'smem_peak_gbs': smem_peak, 'roofline_frac': mv_bytes / (ms * 1e-3) / 1e9 / smem_peak,
        'accept_rate': float(res.accepted.float().mean())}
    return out


# ----------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------
DUMP_SLOT_STRIDE = 32


def dump_outputs(dirname, res):
    """--dump-outputs: what engine.hmc_run returned for the last timed step (rank 0's chains), one float32 .npy per
    array.  Of the (C, S, D) sample block (1 GiB) every chain's slots 0, 32, 64, ... and the last slot are written
    (33 of S = 1000, 33 MiB); the other arrays are written whole: final_state (C, D), accepted and diverged (C, S),
    step_size and num_rejected (C,).  The inputs depend only on the seeds in this file and --steps, so two builds run
    with the same arguments can be compared file by file."""
    import numpy as np
    slots = sorted(set(range(0, S, DUMP_SLOT_STRIDE)) | {S - 1})
    arrays = {'samples': res.samples[:, slots], 'final_state': res.final_state, 'accepted': res.accepted,
              'diverged': res.diverged, 'step_size': res.step_size, 'num_rejected': res.num_rejected}
    for name, t in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), t.float().cpu().numpy())


def run_b200_arm(args, rank, world, local_rank):
    import torch.distributed as dist
    import hamiltorch_b200 as hb
    from hamiltorch_b200 import engine, targets as T, _native as N

    N.require_cuda()
    cpu_base = None
    if world == 1 and not args.no_cpu_baseline:
        # fork the CPU workers BEFORE this process touches CUDA / NVML, spins up torch's intra-op pool or narrows its
        # CPU affinity to the GPU's NUMA node
        cpu_base = cpu_baseline_quick()
    numa = bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {'bound': False, 'skipped': True}
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group('nccl', device_id=dev)

    C = C_PER_GPU                                   # weak scaling: every rank owns 256 chains
    chain_offset = rank * C
    tgt = engine.NativeTarget(T.GaussianIso(D), dev)
    ld = N.padded_ld(D)

    def init_of(r):                                 # rank r's params_init (any rank can rebuild any shard's inputs)
        return 0.1 * torch.randn(C, D, generator=torch.Generator().manual_seed(1234 + r))

    q0_host = init_of(rank).pin_memory()
    q0 = q0_host.to(dev)
    out = torch.empty((C, S, ld), dtype=torch.float32, device=dev)           # 1 GiB: 8x the 126 MB L2
    host_out, host_out_pages = pinned_host_block((C, S, ld))
    stats_local = torch.zeros((max(args.steps, args.warmup, 1), C, 2), dtype=torch.float32, device=dev)
    stats = torch.empty((world,) + tuple(stats_local.shape), dtype=torch.float32, device=dev)
    gathered = torch.empty((world, C, S, ld), dtype=torch.float32, device=dev) if world > 1 else None

    def step(seed, q=None, offset=None, dst=None):
        return engine.hmc_run(tgt, q0 if q is None else q, S, L, EPS, seed=seed,
                              chain_offset=chain_offset if offset is None else offset, out=out if dst is None else dst,
                              device=dev, tuning=int(os.environ.get('HMCX_TUNING', '0')))

    def keep_stats(k, res):               # per-chain summary of step k (reject count, final step size), device side
        stats_local[k, :, 0].copy_(res.num_rejected)
        stats_local[k, :, 1].copy_(res.step_size)

    def gather_stats():                   # every rank's per-chain summaries (tiny)
        if world > 1:
            dist.all_gather_into_tensor(stats.view(-1), stats_local.view(-1))
        else:
            stats[0].copy_(stats_local)

    def gather_samples():                 # SURVEY 8e: the run's one real collective -- every rank's sample block
        dist.all_gather_into_tensor(gathered.view(-1), out.view(-1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # The clock sampler is started BEFORE the warm-up (NVML initialisation must not land inside a timed region); its
    # 20 ms polls then run through the warm-up and all timed regions.
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
        time.sleep(0.2)
    barrier()

    # ---- warm-up: the W requested steps, then (still untimed) until the GPU has been busy for >= 1.5 s AND the last
    #      16 steps are within 3 % of the fastest seen.  A freshly leased box ran the first ~second of launches up to
    #      several times slower with the SM clock already reported at maximum (round-1 notes) and a 13-step warm-up (25 ms
    #      of GPU time) left round 1's SCALE N=1 point 18 % slow; the warm-up is now bounded by GPU-busy time, not by a
    #      step count.  Hard limits: 6 s / 4000 steps.
    for w in range(args.warmup):
        keep_stats(w, step(w))
        if world > 1:
            gather_samples()
    gather_stats()
    barrier()
    extra_warmup, best, stable, busy_ms, t_w = 0, float('inf'), 0, 0.0, time.time()
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    warm_trace = []
    while extra_warmup < 4000 and time.time() - t_w < 6.0 and (stable < 16 or busy_ms < 1500.0):
        w0.record()
        step(1000 + extra_warmup)
        w1.record()
        torch.cuda.synchronize()
        ms = w0.elapsed_time(w1)
        if extra_warmup < 4 or extra_warmup % 100 == 0:
            warm_trace.append(round(ms, 4))
        extra_warmup += 1
        busy_ms += ms
        best = min(best, ms)
        stable = stable + 1 if ms <= 1.03 * best else 0
    barrier()

    # ---- device-timed region: EXACTLY K steps, inputs resident in HBM ----
    # The stream is first given ~25 ms of head start -- 16 more UNTIMED steps queued right after the barrier -- so that
    # the host has queued all K timed launches before the first timed event executes: the events then bracket K kernels
    # running back to back on the device, and a host hiccup (allocator, GC, a CFS throttle of the container's CPU quota)
    # cannot leak into a device-side timestamp.  Real steps, not a spin kernel: the GPU must not see an idle gap between
    # the warm-up and the timed region (after ~25 ms of near-idle spinning single steps of 20 - 40 ms were measured: the
    # power state drops although NVML keeps reporting the maximum SM clock).
    def head_start():
        for i in range(16):
            step(5000 + i)

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 2)]
    for e_ in ev:                                  # create the CUDA events now, not lazily inside the timed region
        e_.record()
    # Python's cyclic garbage collector is parked for the timed regions: a generation-2 pass over the heap torch leaves
    # behind takes 20 - 400 ms, lands at an allocation count (deterministically in the SECOND timed step of this script:
    # measured 19.6, 41.5 and 436 ms against 1.51 ms for every other step) and starves the launch queue.
    gc.collect()
    gc.disable()
    barrier()
    head_start()
    ev[0].record()
    res = None
    for k in range(args.steps):
        ev[1 + 2 * k].record()
        res = step(100 + k)
        ev[2 + 2 * k].record()
        keep_stats(k, res)
        # drop the result before the next call allocates its (small) output tensors: with two result sets alive the
        # caching allocator has to cudaMalloc a new segment inside the timed region, and cudaMalloc behind a full launch
        # queue was measured at 7 - 436 ms (always in the second timed step) against 1.51 ms for every other step
        if k + 1 < args.steps:
            res = None
    gather_stats()
    ev[-1].record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)         # before the legs below overwrite `out`, which holds res.samples
    res = None
    t_total_ms = ev[0].elapsed_time(ev[-1])
    step_ms = [ev[1 + 2 * k].elapsed_time(ev[2 + 2 * k]) for k in range(args.steps)]
    t_kernel_ms = sum(step_ms) / args.steps
    rejected = stats[:, :args.steps, :, 0].sum().item()

    # ---- the same K steps, each followed by the all-gather of its samples (SURVEY 8e / north_star: "a single NCCL
    #      all-gather over NVLink to collect samples"), device-timed: value_with_gather ----
    t_gather_total_ms = t_allgather_ms = None
    gather_check = None
    if world > 1 and not args.no_gather_samples:
        gather_samples()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps)]
        for e_ in a_ev + [g0, g1]:
            e_.record()
        barrier()
        head_start()
        g0.record()
        for k in range(args.steps):
            step(100 + k)
            a_ev[2 * k].record()
            gather_samples()
            a_ev[2 * k + 1].record()
        g1.record()
        barrier()
        t_gather_total_ms = g0.elapsed_time(g1)
        t_allgather_ms = sum(a_ev[2 * k].elapsed_time(a_ev[2 * k + 1]) for k in range(args.steps)) / args.steps
        # cross-rank check ON HARDWARE: `gathered` holds the last step (seed 100+K-1) of every rank; this rank
        # recomputes EVERY shard alone (that shard's params_init and chain_offset, same seed) and compares bit for bit:
        # G GPUs == one GPU.
        scratch = torch.empty_like(out)
        seed_last = 100 + args.steps - 1
        equal = True
        for r in range(world):
            step(seed_last, q=init_of(r).to(dev), offset=r * C, dst=scratch)
            equal = equal and bool(torch.equal(scratch, gathered[r]))
        flag = torch.tensor([1 if equal else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        # order-independent checksum of the gathered block (identical on every rank, and to a 1-GPU run of all shards)
        csum = int(gathered.view(torch.int32).to(torch.int64).sum().item()) & 0xFFFFFFFFFFFF
        gather_check = {'shards_recomputed_on_every_rank': world, 'bitwise_equal_to_single_gpu_runs': bool(flag.item()),
                        'checksum48': csum}
        del scratch

    # ---- e2e: public API, HOST buffers, H2D of the inputs and D2H of the result inside the timed region ----
    def e2e_step(seed):
        r = hb.sample_chains(T.GaussianIso(D), q0_host, num_samples=S, num_steps_per_sample=L, step_size=EPS,
                             rng='philox', seed=seed, chain_offset=chain_offset, out=out)
        host_out.copy_(r.samples_padded, non_blocking=True)
        return r

    # the same call with the reference's store_on_GPU=False contract (samplers.py:1008-1012): `out` is the pinned host
    # block, the kernel's retained-row stores go over PCIe while the chains run -- no device sample buffer, no D2H copy
    def e2e_stream_step(seed):
        return hb.sample_chains(T.GaussianIso(D), q0_host, num_samples=S, num_steps_per_sample=L, step_size=EPS,
                                rng='philox', seed=seed, chain_offset=chain_offset, out=host_out)

    # ... and with the windowed delivery: the run in E2E_WINDOWS windows of iterations, each window's samples leaving through
    # the copy engine on a second stream while the next window computes (engine.hmc_run host_windows)
    E2E_WINDOWS = 8

    def e2e_window_step(seed):
        return hb.sample_chains(T.GaussianIso(D), q0_host, num_samples=S, num_steps_per_sample=L, step_size=EPS,
                                rng='philox', seed=seed, chain_offset=chain_offset, out=host_out,
                                host_windows=E2E_WINDOWS)

    def time_e2e(fn):
        fn(7)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = max(1, min(args.steps, 3))
        e0.record()
        for k in range(n):
            fn(200 + k)
        e1.record()
        barrier()
        return e0.elapsed_time(e1) / n

    t_e2e_copy_ms = time_e2e(e2e_step)
    t_e2e_stream_ms = time_e2e(e2e_stream_step)
    t_e2e_window_ms = time_e2e(e2e_window_step)
    # both paths return the same bytes to the host; check it once on rank-local data (outside the timed regions)
    e2e_step(999)
    torch.cuda.synchronize()
    ref_rows, ref_first = host_out[:, -1].clone(), host_out[:, 1].clone()
    e2e_stream_step(999)
    torch.cuda.synchronize()
    assert torch.equal(ref_rows, host_out[:, -1]), 'streamed samples differ from the copied ones'
    host_out[:, 1].zero_()
    host_out[:, -1].zero_()
    e2e_window_step(999)
    torch.cuda.synchronize()
    assert torch.equal(ref_rows, host_out[:, -1]) and torch.equal(ref_first, host_out[:, 1]), \
        'window-delivered samples differ from the copied ones'

    # ---- streaming leapfrog kernel (the HBM-roofline form of samplers.leapfrog): state >> L2, L=1 ----
    Cs = 32768                                           # 32768 x 1024 fp32 = 128 MiB per array, 4 arrays
    qs = torch.randn(Cs, D, device=dev)
    ps = torch.randn(Cs, D, device=dev)
    qo, po = torch.empty_like(qs), torch.empty_like(ps)
    eps_vec = torch.full((Cs,), EPS, device=dev)
    lib, mass0 = N.load_library(), engine.NativeMass(None, D, dev)

    def stream_launch():          # straight through the C ABI with pre-allocated buffers: no host work between launches
        rc = lib.hmcx_leapfrog(tgt.ref(), mass0.ref(), N.ptr(qs), N.ptr(ps), N.ptr(eps_vec), Cs, ld, 1, N.ptr(qo),
                               N.ptr(po), None, None, N.stream_ptr(dev))
        N.check(rc, 'hmcx_leapfrog')

    for _ in range(3):
        stream_launch()
    torch.cuda.synchronize()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_s = 20
    s0.record()
    for _ in range(n_s):
        stream_launch()
    s1.record()
    torch.cuda.synchronize()
    t_stream_ms = s0.elapsed_time(s1) / n_s
    del qs, ps, qo, po
    clk = clocks.stop() if rank == 0 else None        # sampled across all timed regions above (all under load)
    gc.enable()

    # ---- BASELINE configs 3 / 4 / 5 with this rank's share of their chains ----
    others = None
    if not args.no_other_configs:
        del out, gathered
        torch.cuda.empty_cache()
        others = other_configs(dev, rank, world)

    # max over ranks of every timing; sum over ranks of the other configs' rates
    names = ['total', 'kernel', 'e2e_copy', 'stream', 'e2e_stream', 'e2e_window', 'gather_total', 'allgather']
    vals = [t_total_ms, t_kernel_ms, t_e2e_copy_ms, t_stream_ms, t_e2e_stream_ms, t_e2e_window_ms, t_gather_total_ms or 0.0,
            t_allgather_ms or 0.0]
    if others:
        for k in sorted(others):
            names.append('o_' + k)
            vals.append(others[k]['kernel_ms'])
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tm = dict(zip(names, t.tolist()))
    t_total_ms, t_kernel_ms, t_stream_ms = tm['total'], tm['kernel'], tm['stream']
    t_e2e_copy_ms, t_e2e_stream_ms, t_e2e_window_ms = tm['e2e_copy'], tm['e2e_stream'], tm['e2e_window']
    t_e2e_ms = min(t_e2e_copy_ms, t_e2e_stream_ms, t_e2e_window_ms)

    if rank == 0:
        units_per_step = world * C * S * L
        ms_per_step = t_total_ms / args.steps
        value = units_per_step / (ms_per_step * 1e-3)
        peak, peak_src = measured_peak_hbm()
        algo_bytes = C * S * D * 4 + C * D * 4          # per launch: every retained sample written once + init read once
        achieved = algo_bytes / (t_kernel_ms * 1e-3) / 1e9
        stream_bytes = Cs * D * 16                       # B_step = 16*D B per leapfrog-step x chain (SURVEY 8d)
        stream_gbs = stream_bytes / (t_stream_ms * 1e-3) / 1e9
        h2d, d2h = C * D * 4, C * S * ld * 4
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        sm_mhz = float((clk or {}).get('sm_mhz') or 1965.0)
        issue_peak = n_sm * 4 * sm_mhz * 1e6 / 1e9
        sorted_ms = sorted(step_ms)
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(world),
            'run_notes': {'rng': 'in-kernel Philox4x32-10',
                          'l2_policy': 'each step streams 1.0 GiB of samples (8x the 126 MB L2); no explicit flush',
                          'extra_untimed_warmup_steps': extra_warmup, 'warmup_gpu_busy_ms': busy_ms,
                          'warmup_step_ms_trace': warm_trace,
                          'timed_step_ms': {'min': sorted_ms[0], 'median': sorted_ms[len(sorted_ms) // 2],
                                            'max': sorted_ms[-1], 'all': [round(x, 4) for x in step_ms]},
                          'numa': numa, 'host_block': host_out_pages,
                          'parity': 'config 2: samples bit-exact vs the reference (tests/test_hmc_gpu.py); config 5 (NUTS): '
                                    'bit-exact under the reference step-size schedule (teacher forcing); configs 3/4: see '
                                    'DESIGN.md section 4 for the measured tolerances'},
            'roofline': {'bound': 'hbm', 'kernel': 'hmc_run_kernel<ISO,NONE,E=4,K=1,PHILOX,NUTS=0>', 'achieved': achieved, 'peak': peak,
                         'unit': 'GB/s', 'frac': achieved / peak,
                         # dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full capture
                         # profiles/r2_prof_hmc_run.summary.txt (1.20 MB read + 989.99 MB written)
                         'traffic': 991.2e6, 'peak_source': peak_src,
                         'algorithmic_bytes_per_launch': algo_bytes, 'kernel_ms': t_kernel_ms,
                         'note': 'fused trajectory kernel: L=10 steps per 4*D bytes written, fp32-issue bound by design; '
                                 'see roofline_streaming for the HBM-bound form'},
            # what actually bounds the fused kernel: warp-instruction issue.  Instructions per launch are static for this
            # geometry (ncu smsp__inst_executed.sum, profiles/r2_prof_hmc_run.summary.txt); time is measured live.
            'roofline_issue': {'bound': 'issue', 'kernel': 'hmc_run_kernel<ISO,NONE,E=4,K=1>',
                               'warp_instructions_per_launch': WARP_INST_PER_LAUNCH,
                               'achieved': WARP_INST_PER_LAUNCH / (t_kernel_ms * 1e-3) / 1e9,
                               'peak': issue_peak, 'unit': 'G warp-inst/s',
                               'frac': WARP_INST_PER_LAUNCH / (t_kernel_ms * 1e-3) / 1e9 / issue_peak,
                               'peak_source': '%d SMs x 4 schedulers x %.0f MHz (sampled under load)' % (n_sm, sm_mhz)},
            'roofline_streaming': {'bound': 'hbm', 'kernel': 'leapfrog_kernel<ISO,NONE> L=1, 32768x1024 state',
                                   'achieved': stream_gbs, 'peak': peak, 'unit': 'GB/s', 'frac': stream_gbs / peak,
                                   'algorithmic_bytes_per_launch': stream_bytes, 'kernel_ms': t_stream_ms,
                                   'chain_steps_per_s': Cs / (t_stream_ms * 1e-3)},
            'e2e': {'value': units_per_step / (t_e2e_ms * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                    'd2h_bytes_per_step': d2h, 'ms_per_step': t_e2e_ms,
                    'pcie_gbs_per_rank': (h2d + d2h) / (t_e2e_ms * 1e-3) / 1e9,
                    'path': ('hb.sample_chains(out=<pinned host block>, host_windows=%d): windows of iterations, each '
                             'delivered by the copy engine while the next computes' % E2E_WINDOWS
                             if t_e2e_window_ms <= min(t_e2e_stream_ms, t_e2e_copy_ms) else
                             'hb.sample_chains(out=<pinned host block>): kernel streams the samples to the host'
                             if t_e2e_stream_ms <= t_e2e_copy_ms else
                             'hb.sample_chains(out=<device block>) + D2H copy of the samples'),
                    'ms_per_step_copy_path': t_e2e_copy_ms, 'ms_per_step_stream_path': t_e2e_stream_ms,
                    'ms_per_step_window_path': t_e2e_window_ms},
            'gpu_launches': args.steps,
            'accept_rate': 1.0 - rejected / (world * C * S * args.steps),
            'clocks': clk,
        }
        if t_gather_total_ms is not None:
            ms_g = tm['gather_total'] / args.steps
            line['allgather_samples_ms'] = tm['allgather']
            line['ms_per_step_with_gather'] = ms_g
            line['value_with_gather'] = units_per_step / (ms_g * 1e-3)
            line['allgather_gbs_per_rank'] = (world - 1) * C * S * ld * 4 / (tm['allgather'] * 1e-3) / 1e9
            line['gather_check'] = gather_check
        if others:
            oc = {}
            for k in sorted(others):
                e = dict(others[k])
                e['kernel_ms'] = tm['o_' + k]                           # max over ranks
                units = e['value'] * others[k]['kernel_ms'] * 1e-3      # this rank's chain-steps per launch
                e['value'] = world * units / (e['kernel_ms'] * 1e-3)    # whole job: every rank runs the same share
                if 'algorithmic_tflops' in e:
                    e['algorithmic_tflops_per_gpu'] = e.pop('algorithmic_tflops') * others[k]['kernel_ms'] / e['kernel_ms']
                    e['roofline_frac'] = e['algorithmic_tflops_per_gpu'] / e['roofline_peak_tflops']
                if 'smem_gbs' in e:
                    e['smem_gbs'] = e['smem_gbs'] * others[k]['kernel_ms'] / e['kernel_ms']          # per GPU
                    e['roofline_frac'] = e['smem_gbs'] / e['smem_peak_gbs']
                e['n_gpus'] = world
                oc[k] = e
            line['other_configs'] = oc
        if cpu_base is not None:
            line['cpu_baseline'] = cpu_base
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--cpu-iters', type=int, default=0,
                    help='reference arm: iterations per chain and step (0 = sized from a calibration step so that the '
                         'whole run fits the %d s budget)' % REFERENCE_ARM_BUDGET_S)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gather-samples', action='store_true',
                    help='N > 1: skip the timed all-gather of every step\'s samples (value_with_gather)')
    ap.add_argument('--no-other-configs', action='store_true', help='skip BASELINE configs 3 / 4 / 5')
    ap.add_argument('--no-numa-bind', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='B200 arm: write the outputs of the last timed step to DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs:
        if args.impl != 'b200':
            ap.error('--dump-outputs applies to the B200 arm')
        os.makedirs(args.dump_outputs, exist_ok=True)      # fail before any GPU work if DIR cannot be created
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference_arm(args, rank, world)
        return
    if world != args.gpus:
        if args.gpus > 1:
            raise SystemExit('launch with torchrun --nproc-per-node %d for --gpus %d' % (args.gpus, args.gpus))
    run_b200_arm(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
