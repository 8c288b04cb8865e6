#!/usr/bin/env python
"""bench.py -- Bussgang-GMM estimates/sec (N=64 antennas, K=64 components, 1-bit) on B200.

One "step" = one pass of the hot path (observe -> 1-bit quantise -> Bussgang-GMM 'all' estimate -> NMSE
accumulators) over one batch of 2^20 synthetic observations per GPU at one SNR of the sweep -10..30 dB
(BASELINE.json configs[1]); the per-SNR component parameters are precomputed and resident.

  value      whole-job estimates/s with channels + noise already in HBM (CUDA events, max over ranks)
  e2e        the same metric through Gmm_nbit.estimate_from_y's C entry point on HOST (pinned) complex128 pilots:
             host->device and device->host copies inside the timed region; pcie_frac = its PCIe traffic over the
             measured concurrent H2D + D2H bandwidth of this box
  roofline   the dense estimate kernel timed alone (burst: 5 launches; sustained: >= 2 s back to back):
             algorithmic 16*K*N^2 flop per estimate; traffic from the committed ncu capture (profiles/r02_traffic.json)
  config5    BASELINE.json configs[4] (K = 256, sample-sharded, strong scaling): a fixed GLOBAL batch split over the ranks,
             NMSE per SNR all-reduced once per sweep -- the curve the driver's 1/2/4/8 scaling run records
  cpu_baseline  the reference's own CPU implementation on the host cores (see --impl reference), bounded sample

`--dump-outputs DIR` writes what the timed path computes in its last step (rank 0; see dump_outputs) as DIR/<name>.npy, for
comparing two builds output for output: the inputs are seeded, so the same arguments give the same inputs on every run.

`--impl reference` times the UNMODIFIED reference (`oracle/_ref`, vendored by oracle/build_ref.py): `Gmm_nbit.estimate_from_y`
under the `mp.Pool(cpu_count() // 2).starmap` pattern of Bussgang_GMM.py:29-32, 282-287, plus the single-process rate and the
numpy port (oracle) as extra figures.  Without `oracle/_ref` it times the port (`kind: "port"`).
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ANT, N_COMP, N_BITS = 64, 64, 1
SNRS = list(range(-10, 31, 5))
BATCH = 1 << 20
METRIC = 'Bussgang-GMM estimates/sec (M=64,K=64,1-bit)'
UNIT = 'estimates/s'
FLOP_PER_EST = 16 * N_COMP * N_ANT * N_ANT          # SURVEY.md section 8(d)
WORKLOAD = f"Bussgang-GMM 'full' 1-bit N={N_ANT} K={N_COMP} mode=all, SNR sweep -10..30 dB (BASELINE configs[1])"
C5_COMP = 256                                        # BASELINE configs[4]
C5_GLOBAL = 1 << 23                                  # global observations per step (a stated fraction of the 1e8 of configs[4])
REF_TASK_PILOTS = 512                                # pilots per pool task of the reference arm (prepare: 0.44 s, then ~245 est/s)
DUMP_ROWS = 1 << 14                                  # estimates kept by --dump-outputs: 16 Ki rows of 64 complex128 = 16 MiB


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        return dict(burst=float(p['bf16_tflops']), sustained=float(p.get('bf16_tflops_sustained', p['bf16_tflops'])),
                    hbm=float(p['hbm_gbs']), src='measured (MEASURED_PEAKS.json)')
    except Exception:
        return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src='fallback (B200_PROFILING.md)')


def committed_traffic(kernel, pilots):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/r02_traffic.json, written by
    tools/ncu_traffic.py from the .ncu-rep), scaled from the captured batch to `pilots` (the traffic is linear in the batch:
    the parameters stay in L2)."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')))[kernel]
        return float(t['dram_bytes_per_pilot']) * pilots, t.get('source')
    except Exception:
        return None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
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
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def make_params(K=N_COMP):
    from quantized_channel_estimation_b200 import synthetic      # seeded synthetic generators (SURVEY.md section 8d P-rand)
    return synthetic.random_psd_gmm(K, N_ANT, seed=0)


# ------------------------------------------------------------------------------------------------ CPU arm

def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count() or 1)
    except Exception:
        pass


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([i.get('num_threads', 1) for i in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_port_rate(means, covs, w, n_obs, snr=10, seed=123):
    """The numpy oracle (port of gmm:166-243, batched over samples) on n_obs observations: (est/s, seconds)."""
    from oracle import qce_oracle as orc
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, n_obs, seed=seed)
    r = orc.get_observation_nbit(h, snr, noise, None, N_BITS)
    t0 = time.perf_counter()
    orc.gmm_estimate_from_y(means, covs, w, r, snr, n_summands_or_proba='all', n_bits=N_BITS)
    dt = time.perf_counter() - t0
    return n_obs / dt, dt


def mp_gmm(obj, *args):
    """The reference's pool worker (Bussgang_GMM.py:16-17)."""
    return obj.estimate_from_y(*args)


def pool_worker_init(threads):
    """cpu_count() // 2 pool processes that each spin up a BLAS team over ALL cores thrash (the matrices are 64 x 64): the host's
    threads are divided among the processes instead, so that the arm uses every core once."""
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=threads)
    except Exception:
        pass


def reference_model(means, covs, w):
    """An unmodified reference Gmm_nbit holding the seeded parameters exactly as a fitted model holds them (SURVEY 8c)."""
    from oracle import build_ref
    Gmm_nbit, _, _ = build_ref.import_reference()
    g = Gmm_nbit(n_components=means.shape[0], covariance_type='full')
    g.params['zero_mean'] = True
    g.means_cplx, g.covs_cplx = means.copy(), covs.copy()
    g.gm.weights_ = w.copy()
    return g


def pilots_for(means, covs, w, n, snr, seed):
    from oracle import qce_oracle as orc
    h, noise, _ = orc.sample_gmm_channels(means, covs, w, n, seed=seed)
    return orc.get_observation_nbit(h, snr, noise, None, N_BITS)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from oracle import build_ref
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))      # (a parent bound to one NUMA node must not confine the CPU arm)
    except Exception:
        pass
    means, covs, w = make_params()
    ncpu = os.cpu_count() or 1
    if not build_ref.available():
        # no vendored reference: the numpy port of the same algorithm
        use_all_host_threads()
        sample = 4096
        for _ in range(args.warmup):
            cpu_port_rate(means, covs, w, 256)
        t = 0.0
        for i in range(args.steps):
            t += cpu_port_rate(means, covs, w, sample, snr=SNRS[i % len(SNRS)], seed=1000 + i)[1]
        val, kind, cores = sample * args.steps / t, 'port', blas_threads()
        desc = f'{sample} observations per step (numpy oracle, batched over samples), {ncpu} host cpus; oracle/_ref absent'
        extra = {}
        ms_step = 1e3 * t / args.steps
    else:
        # the reference's own pattern: a process pool, starmap over argument lists (Bussgang_GMM.py:29-32, 282-287).  The reference
        # builds one task per SNR; a step here is ONE SNR of the sweep (like the GPU arm), so its pilots are split into one task per
        # pool process -- every task pays the reference's per-call _prepare_for_prediction.  Pool size: the reference takes
        # cpu_count() // 2 processes and lets every one of them start a BLAS team over all cores; one single-threaded worker per
        # host cpu is the faster use of the same cores for these 64 x 64 products (8 cpus: 789 vs 474 est/s), so that is what is timed.
        n_proc = max(1, ncpu)
        g = reference_model(means, covs, w)
        per_step = n_proc * REF_TASK_PILOTS
        pool = mp.Pool(processes=n_proc, initializer=pool_worker_init, initargs=(max(1, ncpu // n_proc),))

        def step(i, n_task=REF_TASK_PILOTS):
            snr = SNRS[i % len(SNRS)]
            r = pilots_for(means, covs, w, n_proc * n_task, snr, 1000 + i)
            tasks = [[g, r[p * n_task:(p + 1) * n_task], snr, N_ANT, None, 'all', N_BITS, 'uniform', (None, None, None)] for p in range(n_proc)]
            t0 = time.perf_counter()
            pool.starmap(mp_gmm, tasks)
            return time.perf_counter() - t0
        for i in range(args.warmup):
            step(i, 8)
        t = sum(step(i) for i in range(args.steps))
        pool.close()
        pool.join()
        val, kind, cores = per_step * args.steps / t, 'reference', n_proc
        ms_step = 1e3 * t / args.steps
        # extra figures: the same unmodified code in ONE process, and the numpy port (batched over samples, all BLAS threads)
        use_all_host_threads()
        r1 = pilots_for(means, covs, w, 256, 10, 77)
        t0 = time.perf_counter()
        g.estimate_from_y(r1, 10, N_ANT, None, 'all', N_BITS, 'uniform', (None, None, None))
        single = 256 / (time.perf_counter() - t0)
        cpu_port_rate(means, covs, w, 256)
        port, _ = cpu_port_rate(means, covs, w, 4096)
        extra = {'single_process': single, 'port_batched_numpy': port, 'port_threads': blas_threads()}
        desc = (f'unmodified reference Gmm_nbit.estimate_from_y (oracle/_ref), mp.Pool({n_proc}).starmap of single-threaded workers, {REF_TASK_PILOTS} pilots per task, '
                f'{per_step} per step at one SNR, {ncpu} host cpus')
    cpu = {'value': val, 'unit': UNIT, 'cores': cores, 'kind': kind, 'sample': desc}
    cpu.update(extra)
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'c128', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'batch_per_step': int(round(val * ms_step * 1e-3)),
                       'note': 'bounded sample of the same workload on the host cores'},
            'cpu_baseline': cpu,
            'e2e': {'value': val, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess():
    """The CPU arm in a process of its own (a pool forked from a process that holds a CUDA context is asking for trouble):
    one bounded step, its JSON line's cpu_baseline object."""
    env = dict(os.environ)
    for k in ('OMP_NUM_THREADS', 'MKL_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        env.pop(k, None)
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '2', '--warmup', '1'],
                             env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith('{'):
                return json.loads(ln)['cpu_baseline']
        return {'error': (out.stderr or 'no output')[-300:]}
    except Exception as e:       # the baseline is a reported figure, never a reason to lose the bench line
        return {'error': repr(e)[:300]}


# ------------------------------------------------------------------------------------------------ GPU arm

def synth_channels(torch, covs_chol, w_t, B, gen, dev):
    """h = C_k^{1/2} g, k ~ Cat(w), complex64 like SCMMulti; noise complex128 CN(0, 1)."""
    K, N = covs_chol.shape[0], covs_chol.shape[1]
    lab = torch.multinomial(w_t, B, replacement=True, generator=gen)
    order = torch.argsort(lab)
    counts = torch.bincount(lab, minlength=K).tolist()
    g = torch.view_as_complex(torch.randn((B, N, 2), generator=gen, device=dev, dtype=torch.float64)) * np.sqrt(0.5)
    h = torch.empty((B, N), dtype=torch.complex64, device=dev)
    o = 0
    for k, c in enumerate(counts):
        if c:
            idx = order[o:o + c]
            h[idx] = (g[idx] @ covs_chol[k].T).to(torch.complex64)
            o += c
    noise = torch.view_as_complex(torch.randn((B, N, 2), generator=gen, device=dev, dtype=torch.float64)) * np.sqrt(0.5)
    return h, noise.contiguous()


def bind_to_gpu_numa(torch, local):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off (before any pinned allocation: first touch then puts the
    staging buffers on that node too), so that 8 ranks do not pull their pinned DMA through one socket's memory controllers."""
    try:
        p = torch.cuda.get_device_properties(local)
        bdf = f'{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0'
        node = int(open(f'/sys/bus/pci/devices/{bdf}/numa_node').read())
        if node < 0:
            return {'node': None, 'note': 'single NUMA node (sysfs reports -1)'}
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {'node': node, 'cpus': len(cpus), 'pci': bdf}
    except Exception as e:
        return {'node': None, 'note': repr(e)[:120]}


def pcie_peak(torch, dev, mib=256, reps=4):
    """Concurrent pinned H2D + D2H copy bandwidth of this process's GPU (GB/s, sum of both directions)."""
    n = mib << 20
    a_h, b_h = torch.empty(n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
    a_d, b_d = torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    for it in range(reps + 1):
        if it == 1:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            a_d.copy_(a_h, non_blocking=True)
        with torch.cuda.stream(s2):
            b_h.copy_(b_d, non_blocking=True)
    torch.cuda.synchronize()
    return 2 * n * reps / (time.perf_counter() - t0) / 1e9


def dump_outputs(path, torch, model, quant, h, noise, snr, precision):
    """The last timed step's call made once more on the same inputs, with the estimates kept (the same kernels: the timed call
    already computes every estimate for its accumulators).  ``nmse_acc.npy`` float64 [3] holds what this one call returns, starting
    from zero (sum |h_est - h|^2, sum |h|^2, pilots), not the timed loop's running sums; the kernels add it up with float64
    atomics, so its last bits may depend on the order in which blocks finish.  ``h_est_sample.npy`` float64 [DUMP_ROWS, N, 2] holds
    the real and imaginary parts of a fixed, seeded sample of rows of its estimates (the whole batch is 1 GiB)."""
    h_est, acc = model.pipeline(quant, h, noise, 10 ** (-snr / 20), 'all', precision, want_est=True)
    rows = np.sort(np.random.default_rng(0).choice(h_est.shape[0], min(DUMP_ROWS, h_est.shape[0]), replace=False))
    sample = torch.view_as_real(h_est[torch.as_tensor(rows, device=h_est.device)])
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, 'nmse_acc.npy'), acc.cpu().numpy())
    np.save(os.path.join(path, 'h_est_sample.npy'), sample.cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=9)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=BATCH)
    ap.add_argument('--precision', default='auto', choices=['auto', 'tc', 'fp64'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-config5', action='store_true')
    ap.add_argument('--sustain-seconds', type=float, default=2.0)
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        if args.dump_outputs:
            ap.error('--dump-outputs needs --impl b200')
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    import quantized_channel_estimation_b200 as qce
    from quantized_channel_estimation_b200 import _lib, engine

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa = bind_to_gpu_numa(torch, local)
    _lib.require_device()
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    means, covs, w = make_params()
    gmm = qce.Gmm_nbit(n_components=N_COMP, covariance_type='full').set_parameters(means, covs, w, zero_mean=True)
    gmm.precision = args.precision
    eye = np.eye(N_ANT, dtype=complex)
    models = [gmm._prepared(eye, s, N_BITS, 'uniform', None) for s in SNRS]          # resident per-SNR parameters
    quant = engine.Quantizer.get(N_BITS)
    B = args.batch

    # synthetic data, generated on the device (seeded by rank)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    Lc = torch.linalg.cholesky(torch.as_tensor(covs, device=dev))
    h, noise = synth_channels(torch, Lc, torch.as_tensor(w, device=dev), B, gen, dev)
    acc = torch.zeros((len(SNRS), 3), dtype=torch.float64, device=dev)
    acc_sweep, acc_total = torch.zeros_like(acc), torch.zeros_like(acc)
    del Lc

    def step(i):
        j = i % len(SNRS)
        models[j].pipeline(quant, h, noise, 10 ** (-SNRS[j] / 20), 'all', args.precision, acc=acc[j])
        # the path's only exchange: ONE all-reduce of the [n_snr, 3] NMSE accumulators per completed SNR sweep
        if world > 1 and j == len(SNRS) - 1:
            dist.all_reduce(acc_sweep.copy_(acc))
            acc_total.add_(acc_sweep)
            acc.zero_()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    for i in range(max(args.warmup, len(SNRS))):      # every resident per-SNR model is exercised before the clock starts
        step(i)
    barrier()
    acc.zero_()
    acc_total.zero_()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.nvtx.range_push('qce_timed_region')      # lets `ncu --nvtx --nvtx-include qce_timed_region/` list exactly these launches
    ev0.record()
    for i in range(args.steps):
        step(i)
    if world > 1:                                        # remainder of an unfinished sweep (inside the timed region)
        dist.all_reduce(acc_sweep.copy_(acc))
        acc_total.add_(acc_sweep)
    ev1.record()
    torch.cuda.nvtx.range_pop()
    barrier()
    launches = _lib.launch_count() - l0
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    value = world * B * args.steps / (ms * 1e-3)
    accs = (acc_total if world > 1 else acc).cpu().numpy()

    # --- roofline: the dense estimate kernel alone on resident quantised pilots
    pk = peaks()
    import ctypes as C
    lib = _lib.load()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    r = qce.get_observation_nbit(h, SNRS[4], n_bits=N_BITS, noise=noise)
    out = torch.empty((B, N_ANT), dtype=torch.complex128, device=dev)
    tc_used = args.precision in ('auto', 'tc') and lib.qce_format_pilots(models[4].handle, stream, C.c_void_p(r.data_ptr()), B) == 0
    if tc_used:
        def kernel_only():
            _lib.check(lib.qce_estimate_formatted(models[4].handle, stream, B, C.c_void_p(out.data_ptr()), None, None))
    else:
        def kernel_only():
            models[4].estimate(r, 'all', 'fp64')
    for _ in range(2):
        kernel_only()
    torch.cuda.synchronize()
    # burst: like the peak it is compared with ("best of 10" short runs in MEASURED_PEAKS.json) -- the best of a few 5-launch regions,
    # each after a short idle so that the power budget the long timed region above used up has recovered; every region is reported
    reps, bursts = 5, []
    for _ in range(4):
        time.sleep(0.5)
        ev0.record()
        for _ in range(reps):
            kernel_only()
        ev1.record()
        torch.cuda.synchronize()
        bursts.append(ev0.elapsed_time(ev1) / reps)
    k_ms = min(bursts)
    # sustained: the same launch back to back for >= sustain_seconds (one CUDA-event pair around the whole region)
    n_sus = max(reps, int(args.sustain_seconds * 1e3 / k_ms) + 1)
    ev0.record()
    for _ in range(n_sus):
        kernel_only()
    ev1.record()
    torch.cuda.synchronize()
    sus_ms = ev0.elapsed_time(ev1) / n_sus
    achieved = FLOP_PER_EST * B / (k_ms * 1e-3) / 1e12
    achieved_sus = FLOP_PER_EST * B / (sus_ms * 1e-3) / 1e12
    kname = 'dense_tc_kernel' if tc_used else 'dense_fp64_kernel'
    traffic, traffic_src = committed_traffic(kname, B)
    roofline = {'bound': 'tensor', 'achieved': achieved, 'peak': pk['burst'], 'unit': 'TFLOP/s', 'frac': achieved / pk['burst'],
                'traffic': traffic, 'traffic_unit': 'bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)',
                'traffic_source': traffic_src, 'algorithmic_bytes': (256 + 1024) * B if tc_used else None,
                'kernel': kname, 'kernel_ms': k_ms, 'burst_ms_all': bursts,
                'peak_source': f"{pk['src']}: bf16 burst (best of 10 short runs) for the best of {len(bursts)} {reps}-launch regions, 0.5 s idle before each",
                'sustained': {'achieved': achieved_sus, 'peak': pk['sustained'], 'frac': achieved_sus / pk['sustained'],
                              'frac_of_burst_peak': achieved_sus / pk['burst'], 'kernel_ms': sus_ms, 'launches': n_sus,
                              'seconds': sus_ms * n_sus * 1e-3, 'peak_source': f"{pk['src']}: bf16 sustained (4 s back to back)"},
                'algorithmic_flop_per_estimate': FLOP_PER_EST,
                'tensor_passes': 2 if tc_used else None,
                'note': ('FP16 hi/lo split: 2 tensor passes per algorithmic flop; cta_group::2 MMAs' if tc_used else
                         'complex128 SIMT kernel: bounded by the FP64 pipe (~40 TFLOP/s), not the tensor pipe')}
    del out

    # --- e2e: host pinned complex128 pilots -> estimate_from_y's C entry point -> host estimates
    e2e = None
    if not args.no_e2e:
        from quantized_channel_estimation_b200.engine import parse_mode
        barrier()                      # every rank measures its copy ceiling at the same time: the contended figure is the honest one
        pcie = pcie_peak(torch, dev)
        pcie_all = pcie
        if world > 1:
            t = torch.tensor([pcie], device=dev, dtype=torch.float64)
            dist.all_reduce(t)
            pcie_all = float(t.item())
        r_host = torch.empty((B, N_ANT), dtype=torch.complex128).pin_memory()
        r_host.copy_(r.cpu())
        gmm.estimate_from_y(r_host.numpy()[:4096], SNRS[4], N_ANT, n_summands_or_proba='all', n_bits=N_BITS)
        out_host = torch.empty((B, N_ANT), dtype=torch.complex128).pin_memory()
        mode, n_top, rho = parse_mode('all')
        prec = _lib.PREC_TC if tc_used else _lib.PREC_FP64

        def e2e_step(j):
            _lib.check(lib.qce_estimate_host(models[j].handle, C.c_void_p(r_host.data_ptr()), B, mode, n_top, rho, prec,
                                             C.c_void_p(out_host.data_ptr())))
        for i in range(2):
            e2e_step(i % len(SNRS))
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            e2e_step(i % len(SNRS))
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        per_rank = B * args.steps / dt
        e2e = {'value': world * per_rank, 'unit': UNIT, 'h2d_bytes_per_step': B * N_ANT * 16,
               'd2h_bytes_per_step': B * N_ANT * 16, 'api': 'qce_estimate_host (Gmm_nbit.estimate_from_y on host arrays)',
               'host_buffers': 'pinned', 'pcie_gbs_measured': pcie_all,
               'pcie_frac': world * per_rank * 2 * N_ANT * 16 / 1e9 / pcie_all, 'numa': numa,
               'pcie_note': 'pcie_gbs_measured: pinned H2D + D2H copies running concurrently on every rank at the same time (cudaMemcpyAsync '
                            'only, sum over directions and ranks) -- the host-side ceiling of this box for N ranks; pcie_frac: the share of it '
                            'the e2e path moves (2 KiB per estimate: complex128 in and out, the reference dtype)'}
        # the same call with the compact transfer formats (uint8 level codes in, complex64 estimates out: 128 + 512 B per pilot)
        if tc_used:
            _, codes_dev = quant.quantize(torch.view_as_complex(torch.view_as_real(r)), want_codes=True)      # r is on the 1-bit grid: Q(r) = r
            codes_host = torch.empty((B, N_ANT, 2), dtype=torch.uint8).pin_memory()
            codes_host.copy_(codes_dev.cpu())
            out32 = torch.empty((B, N_ANT), dtype=torch.complex64).pin_memory()
            del codes_dev

            def codes_step(j):
                _lib.check(lib.qce_estimate_host_codes(models[j].handle, quant.handle, C.c_void_p(codes_host.data_ptr()), B, mode, n_top, rho, prec,
                                                       C.c_void_p(out32.data_ptr()), 1))
            for i in range(2):
                codes_step(i % len(SNRS))
            barrier()
            t0 = time.perf_counter()
            for i in range(args.steps):
                codes_step(i % len(SNRS))
            torch.cuda.synchronize()
            dtc = max_over_ranks(time.perf_counter() - t0)
            # the complex64 estimates equal the complex128 ones narrowed
            chk = float((out32[:4096].to(torch.complex128) - out_host[:4096]).abs().max()) if (args.steps - 1) % len(SNRS) == (args.steps - 1) % len(SNRS) else None
            e2e['codes_c64'] = {'value': world * B * args.steps / dtc, 'unit': UNIT, 'h2d_bytes_per_step': B * N_ANT * 2, 'd2h_bytes_per_step': B * N_ANT * 8,
                                'api': 'qce_estimate_host_codes (uint8 level codes in, complex64 estimates out)', 'max_abs_diff_vs_c128_path': chk,
                                'pcie_frac_d2h': (B * args.steps / dtc) * N_ANT * 8 / 1e9 / (pcie / 2)}
            del codes_host, out32
        del r_host, out_host
    del r
    clk = clocks.stop() if rank == 0 else None

    # --- config 5 (BASELINE configs[4]): K = 256, a fixed global batch sharded over the ranks, one NMSE all-reduce per sweep
    c5 = None
    if not args.no_config5:
        c5 = run_config5(torch, dist, qce, engine, _lib, dev, world, rank, args, barrier, max_over_ranks)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_subprocess()

    if args.dump_outputs and rank == 0:
        j = (args.steps - 1) % len(SNRS)
        dump_outputs(args.dump_outputs, torch, models[j], quant, h, noise, SNRS[j], args.precision)

    if rank == 0:
        nmse = {str(s): float(a[0] / max(a[2], 1) / N_ANT) for s, a in zip(SNRS, accs) if a[2] > 0}
        line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f16x2-split/f32-acc' if tc_used else 'f64', 'data': 'synthetic',
                'config': {'workload': WORKLOAD,
                           'batch_per_gpu_per_step': B, 'global_batch': world * B, 'parallelism': f'dp{world}',
                           'l2': 'inputs larger than L2 (h 512 MiB c64 + noise 1 GiB c128 per step), no flush needed',
                           'params': 'random-PSD GMM seed 0 (SURVEY 8d P-rand)'},
                'roofline': roofline, 'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clk,
                'nmse_per_snr': nmse, 'config5': c5}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_config5(torch, dist, qce, engine, _lib, dev, world, rank, args, barrier, max_over_ranks):
    """Strong scaling: C5_GLOBAL observations per step in chunks of 2^20 generated from the GLOBAL chunk index (so the data, and with
    it the NMSE per SNR, do not depend on the number of ranks); rank g owns the chunks [g C / G, (g + 1) C / G)."""
    K = C5_COMP
    chunk = 1 << 20
    n_chunks = C5_GLOBAL // chunk
    if n_chunks % world:
        return {'skipped': f'{n_chunks} chunks do not split over {world} ranks'}
    means, covs, w = make_params(K)
    m = qce.Gmm_nbit(n_components=K, covariance_type='full').set_parameters(means, covs, w, zero_mean=True)
    m.precision = args.precision
    eye = np.eye(N_ANT, dtype=complex)
    models = [m._prepared(eye, s, N_BITS, 'uniform', None) for s in SNRS]
    quant = engine.Quantizer.get(N_BITS)
    Lc = torch.linalg.cholesky(torch.as_tensor(covs, device=dev))
    w_t = torch.as_tensor(w, device=dev)
    mine = range(rank * n_chunks // world, (rank + 1) * n_chunks // world)
    data = []
    for c in mine:
        gen = torch.Generator(device=dev).manual_seed(900000 + c)
        data.append(synth_channels(torch, Lc, w_t, chunk, gen, dev))
    del Lc
    acc = torch.zeros((len(SNRS), 3), dtype=torch.float64, device=dev)
    total = torch.zeros_like(acc)

    def step(i):
        j = i % len(SNRS)
        for h, noise in data:
            models[j].pipeline(quant, h, noise, 10 ** (-SNRS[j] / 20), 'all', args.precision, acc=acc[j])
        if j == len(SNRS) - 1:
            flush()

    def flush():
        if world > 1:
            dist.all_reduce(acc)
        total.add_(acc)
        acc.zero_()
    for i in range(len(SNRS)):
        step(i)
    barrier()
    acc.zero_()
    total.zero_()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = _lib.launch_count()
    ev0.record()
    for i in range(args.steps):
        step(i)
    flush()
    ev1.record()
    barrier()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    t = total.cpu().numpy()
    return {'metric': 'Bussgang-GMM estimates/sec (M=64,K=256,1-bit), sample-sharded', 'value': C5_GLOBAL * args.steps / (ms * 1e-3),
            'unit': UNIT, 'scaling': 'strong', 'n_gpus': world, 'ms_per_step': ms / args.steps, 'global_batch_per_step': C5_GLOBAL,
            'fraction_of_1e8_observations': C5_GLOBAL / 1e8, 'chunks_per_rank': len(data), 'gpu_launches': int(_lib.launch_count() - l0),
            'algorithmic_tflops': 16 * K * N_ANT * N_ANT * C5_GLOBAL * args.steps / (ms * 1e-3) / 1e12,
            'collective': 'one all-reduce of the [9, 3] float64 NMSE accumulators per SNR sweep (NCCL)',
            'nmse_per_snr': {str(s): float(a[0] / max(a[2], 1) / N_ANT) for s, a in zip(SNRS, t) if a[2] > 0},
            'pilots_per_snr': {str(s): int(a[2]) for s, a in zip(SNRS, t) if a[2] > 0}}


if __name__ == '__main__':
    main()
