#!/usr/bin/env python
"""bench.py -- EM iterations/s of the cACGMM hot path (BASELINE.json metric).

Workload (config.workload = "C2"): cACGMM, F=513 bins, T=500 frames, D=8
channels, K=3 classes, 100 EM iterations per fit, synthetic complex128 STFT
(iid complex Gaussian, seed 0) and an explicit seeded initialisation.
One "step" = one complete fit (100 EM iterations) of one utterance.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

N > 1 (torchrun, one rank per GPU): every rank fits its own utterance of the
same shape (the path shards over independent utterances / bins without any
data-path collective) -> "scaling": "weak"; value is the whole-job aggregate.

Keys beyond the base contract: `roofline` (dominant kernel vs the measured HBM peak, plus the fp64-pipe
fractions that actually bound it), `cpu_baseline` (the reference -- oracle/_ref, else the NumPy port -- timed on this
host, rank 0, N=1), `e2e` (same metric through the public API with pinned HOST tensors, H2D/D2H inside the timed
region), `e2e_numpy` (the drop-in call: NumPy arrays in, NumPy model out, pageable copies inside the timed region),
`c3_bin_sharded` (BASELINE.json config 3: ONE utterance, bins sharded over the N ranks, fit + predict + all-gather +
DHTV + PSD + GEV + apply, per-stage device times), `frames_bins_per_s`, `clocks`, `gpu_launches`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

F, T, D, K, ITERS = 513, 500, 8, 3, 100
METRIC = 'EM iterations/s, cACGMM F=513 T=500 D=8 K=3 (100-iteration fit)'


def _config(n_gpus):
    return {
        'workload': 'C2: cACGMM fit F=513 T=500 D=8 K=3, 100 EM iterations, complex128',
        'F': F, 'T': T, 'D': D, 'K': K, 'iterations_per_step': ITERS,
        'input': 'iid complex Gaussian STFT, RandomState(0); init RandomState(7) uniform normalised over K',
        'parallelism': f'{n_gpus} independent utterance(s), one per GPU, no collective',
        'sync': 'resident steps are enqueued back to back inside pb_bss_b200.deferred_status(): the status words of the '
                'K fits are read once after the timed loop; e2e legs synchronise per call',
        'l2': 'a 256 MiB buffer is overwritten between timed steps (L2 flush); within a step the '
              '32.8 MB observation is re-read every EM iteration and stays L2 resident by design',
    }


def _inputs(rank):
    from oracle import synth
    y = synth.noise_stft(F, T, D, seed=rank)
    init = synth.init_affiliation(F, K, T, seed=7 + rank)
    return y, init


# --------------------------------------------------------------------------
# clocks sampler (nvidia-smi in a background thread during the timed region)
# --------------------------------------------------------------------------
class ClockSampler:
    """Streams `nvidia-smi -lms 10` for one GPU while the timed region runs."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap,power.draw')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        self.head = b''
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                 '--format=csv,noheader,nounits', '-lms', '10'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, bufsize=0)
            # the sampler is running before the timed region starts: wait for its first line (nvidia-smi takes a
            # few hundred ms to come up, longer when eight ranks start one each)
            import select
            ready, _, _ = select.select([self.proc.stdout], [], [], 5.0)
            if ready:
                self.head = os.read(self.proc.stdout.fileno(), 65536)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is None:
            return
        time.sleep(0.03)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = b''
        text = (self.head + (out or b'')).decode(errors='replace')
        self.rows = [[c.strip() for c in line.split(',')] for line in text.strip().splitlines() if line.strip()]

    def summary(self):
        def num(x):
            try:
                return float(x)
            except ValueError:
                return None
        rows = [r for r in self.rows if len(r) >= 6 and num(r[0]) is not None]
        sm = [num(r[0]) for r in rows]
        mx = [num(r[1]) for r in rows if num(r[1]) is not None]
        # "under load": samples within 25% of the highest clock seen (idle samples bracket the region)
        load = [v for v in sm if v >= 0.75 * max(sm)] if sm else []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in rows for i in range(4) if r[2 + i].lower().startswith('active')})
        pw = [num(r[6]) for r in rows if len(r) > 6 and num(r[6]) is not None]
        return {'sm_mhz': float(np.median(load)) if load else None,
                'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm), 'power_w_max': max(pw) if pw else None}


# --------------------------------------------------------------------------
# CPU baseline: the unmodified reference (oracle/_ref, see oracle/build_ref.py) when it travelled with the
# repository, else the NumPy oracle port (same einsums as the reference)
# --------------------------------------------------------------------------
def _cpu_fit_fn():
    """Returns (fit(y, init, iterations), kind, description)."""
    try:
        from oracle import ref_shim
        if ref_shim.available():
            ref = ref_shim.load()
            trainer = ref.distribution.CACGMMTrainer()
            return (lambda y, init, it: trainer.fit(y, initialization=init, iterations=it),
                    'reference', 'pb_bss.distribution.CACGMMTrainer.fit of the unmodified reference (oracle/_ref)')
    except Exception:
        pass
    from oracle import pb_bss_oracle as O
    return (lambda y, init, it: O.cacgmm_fit(y, init, it)), 'port', 'oracle/pb_bss_oracle.cacgmm_fit (NumPy port)'


def cpu_baseline_single(iters=40):
    """As shipped: one process (the hot einsums are single threaded)."""
    fit, kind, what = _cpu_fit_fn()
    y, init = _inputs(0)
    fit(y[:32], init[:32], 2)  # warm-up (imports, einsum paths)
    t0 = time.perf_counter()
    fit(y, init, iters)
    dt = time.perf_counter() - t0
    return {'value': iters / dt, 'unit': 'EM iterations/s', 'cores': 1, 'kind': kind,
            'sample': f'{iters} EM iterations of the full C2 problem in {dt:.1f} s, {what}, 1 process'}


def _ref_worker(idx, cpu, lo, hi, conn):
    """Persistent worker of the reference arm: owns bins [lo, hi) for the whole run (nothing is pickled per step),
    pinned to one core, one BLAS thread."""
    try:
        os.sched_setaffinity(0, {cpu})
    except Exception:
        pass
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    fit, kind, what = _cpu_fit_fn()
    y, init = _inputs(0)
    y, init = np.ascontiguousarray(y[lo:hi]), np.ascontiguousarray(init[lo:hi])
    conn.send((kind, what))
    while True:
        iters = conn.recv()
        if iters is None:
            break
        t0 = time.perf_counter()
        fit(y, init, iters)
        conn.send(time.perf_counter() - t0)


def reference_arm(args):
    """--impl reference: the reference's CPU implementation with all host cores.  The bins are independent, so they
    are sharded over one persistent worker process per core; a step is one fit of the whole C2 problem (wall time of
    the slowest worker), 100 EM iterations when the run then still ends within a few minutes, else a bounded sample."""
    import multiprocessing as mp
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except Exception:
        cpus = list(range(os.cpu_count() or 1))
    workers = max(1, min(len(cpus), F))
    bounds = np.linspace(0, F, workers + 1).astype(int)
    ctx = mp.get_context('fork')
    procs = []
    for i, (lo, hi) in enumerate(zip(bounds[:-1], bounds[1:])):
        if hi <= lo:
            continue
        pc, cc = ctx.Pipe()
        p = ctx.Process(target=_ref_worker, args=(i, cpus[i % len(cpus)], int(lo), int(hi), cc), daemon=True)
        p.start()
        procs.append((p, pc))
    kind, what = procs[0][1].recv()
    for _, pc in procs[1:]:
        pc.recv()

    def step(iters):
        t0 = time.perf_counter()
        for _, pc in procs:
            pc.send(iters)
        for _, pc in procs:
            pc.recv()
        return time.perf_counter() - t0

    step(2)
    t_it = step(4) / 4  # seconds per EM iteration of the whole problem
    budget = 150.0
    iters = ITERS if (args.steps + max(1, args.warmup)) * ITERS * t_it <= budget else \
        max(4, int(budget / ((args.steps + max(1, args.warmup)) * t_it)))
    for _ in range(max(1, args.warmup)):
        step(iters)
    ts = [step(iters) for _ in range(args.steps)]
    for p, pc in procs:
        pc.send(None)
    for p, _ in procs:
        p.join(timeout=5)
    dt = sum(ts)
    value = args.steps * iters / dt
    cfg = _config(args.gpus)
    cfg['iterations_per_step'] = iters
    cfg['parallelism'] = f'{len(procs)} worker processes, one per host core, bins sharded, no communication'
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'EM iterations/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': max(1, args.warmup),
        'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': cfg, 'frames_bins_per_s': value * F * T,
        'step_spread': {'min_ms': min(ts) * 1e3, 'max_ms': max(ts) * 1e3},
        'cpu_baseline': {'value': value, 'unit': 'EM iterations/s', 'cores': len(procs), 'kind': kind,
                         'sample': f'{iters} EM iterations per step of the full C2 problem (F=513 bins sharded over '
                                   f'{len(procs)} persistent worker processes pinned to one core each), {what}'},
        'e2e': {'value': value, 'unit': 'EM iterations/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------
# BASELINE.json config 3: one utterance, bins sharded over the ranks
# --------------------------------------------------------------------------
def c3_bin_sharded_block(world, rank, barrier, reps=5):
    """fit (100 it) + predict + all-gather + DHTV + PSD + GEV + apply on ONE utterance whose 513 bins are sharded
    over the `world` ranks (pb_bss_b200.parallel.sharded_separation).  Device-timed with CUDA events per stage, max
    over ranks; rank 0 also runs the whole utterance alone in the same job, which gives the speed-up."""
    import torch
    import torch.distributed as dist
    from oracle import synth
    from pb_bss_b200 import parallel
    y, _ = synth.structured_stft(F, T, D, K, seed=5)
    init = synth.init_affiliation(F, K, T, seed=7)
    lo, hi = parallel.bin_shards(F, world)[rank]
    yl, il = torch.from_numpy(y[lo:hi]).cuda(), torch.from_numpy(init[lo:hi]).cuda()

    def run(y_, i_, alone):
        saved = parallel.world
        if alone:
            parallel.world = lambda group=None: (0, 1)
        try:
            best = None
            for rep in range(reps + 2):
                if not alone:
                    barrier()
                else:
                    torch.cuda.synchronize()
                tm = parallel.StageTimer()
                parallel.sharded_separation(y_, i_, F, iterations=ITERS, timer=tm)
                torch.cuda.synchronize()
                ms = tm.ms()
                ms['total'] = sum(ms.values())
                if rep >= 2 and (best is None or ms['total'] < best['total']):
                    best = ms
            return best
        finally:
            parallel.world = saved

    stages = run(yl, il, alone=False)
    names = list(stages)
    t = torch.tensor([stages[n] for n in names], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    stages = dict(zip(names, t.tolist()))
    single = None
    if rank == 0:
        single = stages if world == 1 else run(torch.from_numpy(y).cuda(), torch.from_numpy(init).cuda(), alone=True)
    if world > 1:
        barrier()
    if rank != 0:
        return None
    return {
        'workload': 'C3: one utterance F=513 T=500 D=8 K=3 (structured mixture), bins sharded over the ranks; '
                    'cACGMM fit 100 iterations + predict + NCCL all-gather of the affiliations + DHTV permutation '
                    'alignment (replicated) + PSD + GEV + apply',
        'n_gpus': world, 'bins_per_rank': [h - l for l, h in parallel.bin_shards(F, world)],
        'ms_per_pipeline': stages['total'], 'stage_ms': {k: v for k, v in stages.items() if k != 'total'},
        'single_gpu_ms_same_run': single['total'], 'single_gpu_stage_ms': {k: v for k, v in single.items() if k != 'total'},
        'speedup_vs_single_gpu': single['total'] / stages['total'],
        'timing': 'CUDA events on the launching stream, best of %d repetitions after 2 warm-ups, max over ranks per '
                  'stage' % reps,
    }


def dump_outputs(model, out_dir):
    """Writes the model of one timed step, as a caller of CACGMMTrainer.fit receives it, to out_dir/<name>.npy in
    float64 (3.3 MB for C2).  Complex arrays get a trailing (real, imag) axis.  The eigenvectors carry an arbitrary
    phase per column; the covariance V diag(lambda) V^H does not, so two builds can be compared on it."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {
        'weight': model.weight,                                                    # (F, K, 1)
        'covariance_eigenvalues': model.cacg.covariance_eigenvalues,               # (F, K, D)
        'covariance_eigenvectors': model.cacg.covariance_eigenvectors,             # (F, K, D, D, 2)
        'covariance': model.cacg.covariance,                                       # (F, K, D, D, 2)
    }
    for name, t in arrays.items():
        if t.is_complex():
            t = torch.view_as_real(t)
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy().astype(np.float64, copy=False))


# --------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------
def b200_arm(args):
    import torch
    import torch.distributed as dist
    import pb_bss_b200
    from pb_bss_b200 import _lib
    from pb_bss_b200.distribution import CACGMMTrainer

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    lib = _lib.load()

    y_host, init_host = _inputs(rank)
    y_pin = torch.from_numpy(y_host).pin_memory()
    init_pin = torch.from_numpy(init_host).pin_memory()
    y_dev, init_dev = y_pin.cuda(), init_pin.cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    trainer = CACGMMTrainer()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        return trainer.fit(y_dev, initialization=init_dev, iterations=ITERS)

    def step_e2e():
        # host buffers in, host model out: every byte crosses PCIe inside this call
        m = trainer.fit(y_pin, initialization=init_pin, iterations=ITERS)
        out = (m.weight.cpu(), m.cacg.covariance_eigenvectors.cpu(), m.cacg.covariance_eigenvalues.cpu())
        assert not out[1].is_cuda
        return out

    def step_numpy():
        # the drop-in call of the reference's API: NumPy arrays in, NumPy model out (pageable host memory)
        m = trainer.fit(y_host, initialization=init_host, iterations=ITERS)
        assert isinstance(m.cacg.covariance_eigenvectors, np.ndarray)
        return m

    for _ in range(max(3, args.warmup)):
        step_resident()
    barrier()
    lib.pbb_profile_reset()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with ClockSampler(local) as clocks:
        barrier()
        launches0 = lib.pbb_launch_count()
        # The K resident steps are enqueued back to back: inside deferred_status() a fit does not read its 4-byte
        # device status word back (a host synchronisation) after every call but once, when the block ends, so the
        # events bracket GPU work only and the number does not depend on the speed of the host's Python.  (The e2e
        # legs below keep the per-call synchronisation of the plain API.)
        with pb_bss_b200.deferred_status():
            for e0, e1 in evs:
                flush.fill_(1)
                e0.record()
                model = step_resident()
                e1.record()
        barrier()
        launches = lib.pbb_launch_count() - launches0
    t_dev = sum(e0.elapsed_time(e1) for e0, e1 in evs) * 1e-3
    if args.dump_outputs and rank == 0:
        dump_outputs(model, args.dump_outputs)
    # end to end through the public API with host buffers
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    barrier()
    step_numpy()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_numpy()
    torch.cuda.synchronize()
    t_np = time.perf_counter() - t0
    barrier()
    c3 = c3_bin_sharded_block(world, rank, barrier)
    # the end-to-end path must produce the resident path's model (checked outside the timed regions)
    m_res = step_resident()
    out_e2e = step_e2e()
    e2e_identical = bool(torch.equal(out_e2e[2], m_res.cacg.covariance_eigenvalues.cpu())
                         and torch.equal(out_e2e[1], m_res.cacg.covariance_eigenvectors.cpu()))
    # dominant-kernel timing: an extra, event-instrumented fit right after the timed region
    prof = None
    if rank == 0:
        lib.pbb_profile_enable(1)
        step_resident()
        torch.cuda.synchronize()
        import ctypes
        ms = ctypes.c_double()
        n = ctypes.c_int()
        name = ctypes.create_string_buffer(128)
        lib.pbb_profile_dominant(name, 128, ctypes.byref(ms), ctypes.byref(n))
        lib.pbb_profile_enable(0)
        prof = {'kernel': name.value.decode(), 'ms_total': ms.value, 'launches': n.value}

    times = torch.tensor([t_dev, t_e2e, t_np], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    t_dev, t_e2e, t_np = times.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * args.steps * ITERS / t_dev
    e2e = world * args.steps * ITERS / t_e2e
    e2e_np = world * args.steps * ITERS / t_np
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s'
    # algorithmic bytes of one EM iteration (SURVEY.md 8d, complex128):
    # F*T*D*16 + 2*F*K*(D*D*16 + D*8 + 8)
    b_iter = F * T * D * 16 + 2 * F * K * (D * D * 16 + D * 8 + 8)
    line_clocks = clocks.summary()
    roofline = None
    traffic = None
    try:  # DRAM bytes of the same kernel + workload from the committed `ncu --set full` capture
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'em_kernel_metrics.json')))['traffic_bytes_per_launch']
    except Exception:
        pass
    if prof and prof['ms_total'] > 0:
        iters_covered = ITERS  # the dominant kernel(s) of one fit cover all EM iterations
        achieved = b_iter * iters_covered / (prof['ms_total'] * 1e-3) / 1e9
        roofline = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                    'frac': achieved / peak, 'traffic': traffic, 'peak_source': peak_src,
                    'traffic_source': 'profiles/em_kernel_metrics.json (dram__bytes_read.sum + dram__bytes_write.sum, one launch = 100 EM iterations)',
                    'algorithmic_bytes_per_launch': b_iter * iters_covered,
                    'kernel': prof['kernel'], 'kernel_launches_per_fit': prof['launches'],
                    'kernel_ms_per_fit': prof['ms_total'],
                    'algorithmic_bytes_per_em_iteration': b_iter,
                    'note': 'fp64 CUDA-core bound: the observation is L2 resident after the first iteration, so DRAM '
                            'traffic is far below the algorithmic bytes; the fp64 figures below are the binding ones'}
        # fp64 pipe: 560 pipe operations per frame x bin x iteration (512 slot-form E/M operations + posterior),
        # DESIGN.md section 4.  Two denominators: the nominal DFMA rate (64 lanes/clk/SM: fma(a, x, y) with two
        # operands held in the reuse cache, scripts/microbench/fp64_rate.cu) and the rate of a DFMA that reads three
        # different 64-bit registers, which is what acc = fma(w, psi, acc) is (42.7 lanes/clk/SM measured,
        # scripts/microbench/fp64_operands.cu, profiles/fp64_operands_r2.txt).
        clk = (line_clocks or {}).get('sm_mhz') or 1965.0
        ops = 560.0 * F * ((T + 31) // 32 * 32) * ITERS
        t_k = prof['ms_total'] * 1e-3
        nominal = 148 * 64 * clk * 1e6
        roofline['fp64'] = {
            'pipe_ops_per_launch': ops, 'achieved_lane_ops_per_s': ops / t_k,
            'peak_nominal_lane_ops_per_s': nominal, 'frac_of_nominal_dfma_peak': ops / t_k / nominal,
            'peak_three_register_dfma_lane_ops_per_s': nominal * 42.7 / 64,
            'frac_of_three_register_dfma_peak': ops / t_k / (nominal * 42.7 / 64),
            'sm_mhz': clk,
            'chain_bound': 'one bin-iteration (task -> class update -> publish -> next model) has a latency of ~17 us '
                           'on an otherwise idle GPU (profiles/chain_latency_r2.txt), which alone bounds a '
                           '100-iteration fit at 1.7 ms whatever the arithmetic rate'}
    cpu = None
    if world == 1 and not args.no_cpu:
        cpu = cpu_baseline_single()
    line = {
        'metric': METRIC, 'value': value, 'unit': 'EM iterations/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': max(3, args.warmup), 'ms_per_step': t_dev / args.steps * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic', 'config': _config(world),
        'frames_bins_per_s': value * F * T,
        'e2e': {'value': e2e, 'unit': 'EM iterations/s',
                'h2d_bytes_per_step': int(y_host.nbytes + init_host.nbytes),
                'd2h_bytes_per_step': int(F * K * (D * D * 16 + D * 8 + 8)),
                'frames_bins_per_s': e2e * F * T,
                'model_identical_to_resident_path': e2e_identical,
                'transfer': 'CACGMMTrainer.fit on pinned host tensors: observation + initial affiliations are '
                            'read over PCIe by a loader kernel that overlaps the EM kernel, the model is '
                            'written to pinned host memory by the final update kernel; timed with the host '
                            'clock around K calls, each synchronised'},
        'e2e_numpy': {'value': e2e_np, 'unit': 'EM iterations/s', 'ms_per_step': t_np / args.steps * 1e3,
                      'h2d_bytes_per_step': int(y_host.nbytes + init_host.nbytes),
                      'd2h_bytes_per_step': int(F * K * (D * D * 16 + D * 8 + 8)),
                      'transfer': 'CACGMMTrainer.fit(numpy, initialization=numpy) -> model of NumPy arrays: pageable '
                                  'host -> device copies, fit, device -> host copies, all inside the timed region'},
        'c3_bin_sharded': c3,
        'gpu_launches': int(launches),
        'roofline': roofline, 'cpu_baseline': cpu, 'clocks': line_clocks,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the model fitted in the last timed step to DIR/<name>.npy (float64, rank 0); the '
                         'inputs are seeded, so runs with the same arguments can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200 (the reference arm keeps its models in the worker processes)')
    if args.impl == 'reference':
        reference_arm(args)
    else:
        b200_arm(args)


if __name__ == '__main__':
    main()
