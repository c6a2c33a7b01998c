#!/usr/bin/env python
"""bench.py -- GP predictions/sec (N train x horizon test, fp64) on B200s.

One "step" = one pass of the hot path over one horizon batch: H test points evaluated
for ALL Ny outputs (mean, variance, Jacobian, first-order Taylor covariance, method
'TA'), model resident on the device(s).  Default workload = BASELINE.json's 1/2/4/8-GPU
configuration C5 (N=16384, Nx=10, Ny=8, H=50): the Ny independent GPs are sharded over
the ranks (all 8 on one GPU at --gpus 1, one per GPU at --gpus 8: strong scaling), one
NCCL all-gather of H*(2+Nx) doubles per output reassembles state/covariance.

  python bench.py [--gpus N --steps K --warmup W] [--workload c5|c3|c2] [--impl reference]
                  [--dump-outputs DIR]

--dump-outputs writes the arrays the timed path returned in its last timed step as
DIR/<name>.npy (float64); the inputs are seeded, so two builds run with the same arguments
can be compared output for output.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events on the
engine's stream, max over ranks); `e2e` = the same metric through the host C-ABI call
(host buffers, H2D/D2H inside); `roofline` = the dominant kernel (the v = L^-1 ks
tensor-core product) against the measured fp64 GEMM peak; `cpu_baseline` = the oracle
port of the reference's predict path on the box's host cores (bounded sample).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the source tree

WORKLOADS = {
    'c5': dict(N=16384, Nx=10, Ny=8, H=50, cfg=5, name='C5: N=16384 Nx=10 Ny=8 H=50 TA, outputs sharded over GPUs'),
    'c3': dict(N=4096, Nx=8, Ny=6, H=30, cfg=3, name='C3: N=4096 Nx=8 Ny=6 H=30 TA'),
    'c2': dict(N=1000, Nx=8, Ny=6, H=30, cfg=2, name='C2: N=1000 Nx=8 Ny=6 H=30 TA'),
}
METRIC = 'GP predictions/sec (N train x horizon test, fp64)'
PREDICT_KERNEL_NAME = ('predict_streamk_kernel<BM> (v = Linv ks: persistent stream-K DMMA product fed by TMA tensor maps, '
                       'fused squared-norm reduction / finalize / peer store / covariance assembly)')


def make_workload(N, Nx, Ny, cfg, H):
    """Seeded synthetic inputs of SURVEY.md 8(d) (same generator as the oracle's
    synthetic_problem; tests assert they agree)."""
    rng = np.random.default_rng(1234 + cfg)
    X = rng.standard_normal((N, Nx))
    W = rng.standard_normal((Nx, Ny)) / np.sqrt(Nx)
    F = np.sin(X @ W) + 0.1 * (X @ W) ** 2
    Y = F + 1e-2 * rng.standard_normal((N, Ny))
    Y = (Y - Y.mean(0)) / Y.std(0)
    hyper = np.zeros((Ny, Nx + 2))
    hyper[:, :Nx] = rng.uniform(2.0, 6.0, size=(Ny, Nx))
    hyper[:, Nx] = 1.0
    hyper[:, Nx + 1] = 1e-2
    rt = np.random.default_rng(7)
    Z = 0.5 * rt.standard_normal((H, Nx))
    A = rt.standard_normal((Nx, Nx))
    Sigma = 1e-4 * np.eye(Nx) + 1e-5 * A @ A.T
    return dict(X=X, Y=Y, hyper=hyper, Z=Z, Sigma=Sigma)


def dump_outputs(dirname, **arrays):
    """--dump-outputs: each array as dirname/<name>.npy in float64."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + '.npy'), np.ascontiguousarray(a, dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, device):
        self.device = device
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(self.device), '--query-gpu=' + self.Q,
                                       '--format=csv,noheader,nounits', '-lms', '100'],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
            return
        t0 = time.time()          # nvidia-smi needs ~0.5 s to emit its first sample
        while time.time() - t0 < 4.0 and os.path.getsize(self.f.name) == 0:
            time.sleep(0.05)

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(',') for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[5 + k].strip().lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def cpu_predict_port(orc, X, hyper_a, alpha_a, L_a, Z):
    """The reference's numeric predict for ONE output on the CPU (oracle port of
    gp_functions.py:111-147 / GP.covar gp_class.py:353-381): ks, mean, v = L\\ks (true
    triangular solve -- cheaper than the reference's LU np.linalg.solve, so conservative),
    var, Jacobian."""
    from scipy.linalg import solve_triangular
    Nx = X.shape[1]
    ell = hyper_a[:Nx]; sf2 = hyper_a[Nx] ** 2
    ks = orc.covSEard(X, Z, ell, sf2)
    mean = ks.T @ alpha_a
    v = solve_triangular(L_a, ks, lower=True, check_finite=False)
    var = sf2 - np.sum(v * v, 0)
    w = ks * alpha_a[:, None]
    J = np.stack([(w * (X[:, d][:, None] - Z[:, d][None, :])).sum(0) / ell[d] ** 2 for d in range(Nx)], 1)
    return mean, var, J


def all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs (reference arm, oracle parity) are meant to use every
    host core, so lift the BLAS/OpenMP limits at run time."""
    try:
        from threadpoolctl import threadpool_limits
        return threadpool_limits(limits=os.cpu_count())
    except Exception:
        import contextlib
        return contextlib.nullcontext()


def run_reference(args, wl, rank):
    """--impl reference: the reference's own CPU path for this metric (oracle port; the
    reference is pure Python on numpy/CasADi, CasADi is not installable here) on all host
    threads, at the SAME configuration as the GPU arm: every one of the Ny outputs is
    factorised on the CPU (set-up, not timed -- as in the GPU arm) and every timed step
    predicts all H points for all Ny outputs (ks, mean, L\\ks, var, Jacobian, TA covariance).
    When all Ny outputs do not fit the ~150 s budget (N=16384: ~25 s of CPU set-up and ~1.3 s per predict pass
    per output on 128 cores) a stated subset of the outputs is run at FULL N and H and the step time is scaled by
    Ny / n (outputs are independent and cost the same): no extrapolation in N."""
    if rank != 0:
        return
    from oracle import gp_oracle as orc
    _limits = all_host_threads()
    _limits.__enter__()
    N, Nx, Ny, H = wl['N'], wl['Nx'], wl['Ny'], wl['H']
    w = make_workload(N, Nx, Ny, wl['cfg'], H)
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64e9
    # bounded sample (the whole run must end within a few minutes): as many of the Ny outputs as fit a ~150 s
    # budget, measured on the first one -- CPU factorisation (set-up, not timed) + (warmup + steps) predict passes
    budget_s = float(os.environ.get('GPMPC_REF_BUDGET_S', '150'))
    facs = []
    t0 = time.perf_counter()
    facs.append(orc.factor_large(w['X'], w['Y'][:, 0], w['hyper'][0]))
    t_fac1 = time.perf_counter() - t0
    t1 = time.perf_counter()
    cpu_predict_port(orc, w['X'], w['hyper'][0], facs[0]['alpha'], facs[0]['chol'], w['Z'])
    t_pred1 = time.perf_counter() - t1
    per_output = t_fac1 + (args.warmup + args.steps) * t_pred1
    n_fac = int(max(1, min(Ny, budget_s // max(per_output, 1e-9), (avail // (8.0 * N * N)) - 3)))
    for a in range(1, n_fac):
        facs.append(orc.factor_large(w['X'], w['Y'][:, a], w['hyper'][a]))
    t_setup = time.perf_counter() - t0

    def step():
        mean = np.zeros((H, n_fac)); var = np.zeros((H, n_fac)); J = np.zeros((H, n_fac, Nx))
        for a in range(n_fac):
            mean[:, a], var[:, a], J[:, a] = cpu_predict_port(orc, w['X'], w['hyper'][a], facs[a]['alpha'], facs[a]['chol'], w['Z'])
        return dict(mean=mean, var=var, cov=orc.ta_cov(var, J, w['Sigma']), jac=J)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step()
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, **out)
    t_step = dt * (Ny / n_fac)
    val = H / t_step
    if n_fac == Ny:
        sample = ('full configuration: all %d outputs at N=%d, H=%d per step; CPU set-up (K + potrf + alpha, %d outputs) '
                  '%.1f s not timed' % (Ny, N, H, Ny, t_setup))
    else:
        sample = ('%d of %d outputs at full N=%d, H=%d; per-step time x %g (outputs are independent); CPU set-up %.1f s '
                  'not timed' % (n_fac, Ny, N, H, Ny / n_fac, t_setup))
    line = {'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'predictions/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': t_step * 1e3, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': wl['name'], 'method': 'TA', 'N': N, 'Nx': Nx, 'Ny': Ny, 'H': H},
            'cpu_baseline': {'value': val, 'unit': 'predictions/s', 'cores': os.cpu_count(), 'kind': 'port',
                             'sample': sample},
            'e2e': {'value': val, 'unit': 'predictions/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c5', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="write the last timed step's mean, var, cov and jac to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else max(args.warmup, 1)
    wl = dict(WORKLOADS[args.workload])
    if os.environ.get('GPMPC_BENCH_NY'):          # diagnostics: e.g. one output per GPU on fewer GPUs
        wl['Ny'] = int(os.environ['GPMPC_BENCH_NY']); wl['name'] += ' [Ny=%d override]' % wl['Ny']
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))

    if args.impl == 'reference':
        run_reference(args, wl, rank)
        return

    import torch
    import torch.distributed as dist
    import gp_mpc_b200
    from gp_mpc_b200 import _lib as L
    from gp_mpc_b200.partition import output_block

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the engine has no CPU path')
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    N, Nx, Ny, H = wl['N'], wl['Nx'], wl['Ny'], wl['H']
    w = make_workload(N, Nx, Ny, wl['cfg'], H)

    # ---- model set-up (not timed): data -> K -> Cholesky -> L^-1 -> alpha on the GPU ----
    b, n = output_block(Ny, rank, world)
    if n == 0:
        raise SystemExit('workload %s has fewer outputs than ranks' % args.workload)
    t0 = time.perf_counter()
    eng = gp_mpc_b200.Engine(N, Nx, Ny, b, n, device=local_rank)
    for kv in filter(None, os.environ.get('GPMPC_OPTS', '').split(',')):     # e.g. tri_variant=0,gemm_variant=1
        k, v = kv.split('=')
        eng.set_option(k, float(v))
    eng.set_data(w['X'], w['Y'])
    eng.set_hyper(w['hyper'])
    if world > 1:
        box = [eng.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        eng.comm_init(box[0], rank, world)
        peer_mode = False
        if os.environ.get('GPMPC_NO_PEER', '0') != '1':     # fused epilogue + all-gather over peer memory
            try:
                mine = eng.peer_export(max(64, H))
            except Exception:
                mine = None
            hs = [None] * world
            dist.all_gather_object(hs, mine)
            ok = all(x is not None for x in hs)
            if ok:
                try:
                    eng.peer_attach(hs)
                except Exception:
                    ok = False
            oks = [None] * world
            dist.all_gather_object(oks, ok)
            peer_mode = all(oks)
            if not peer_mode:                                # collective fallback to the NCCL gather
                eng.set_option('peer', 0)
    else:
        peer_mode = False
    # north-star kernel targets, timed with CUDA events inside the library on this engine's slabs
    # (they are scratch until factorize): K build, the top-level trailing update, potrf+trtri
    sec = {}
    if os.environ.get('GPMPC_BENCH_SECONDARY', '1') == '1':
        sec['kbuild_full_ms'] = eng.profile(L.PROF_KBUILD_FULL, reps=10)
        sec['kbuild_lower_ms'] = eng.profile(L.PROF_KBUILD_LOWER, reps=10)
        sec['syrk_ms'] = eng.profile(L.PROF_SYRK, n=0, reps=3)
        sec['factorize_ms'] = eng.profile(L.PROF_FACTORIZE, reps=2)
    eng.factorize()
    t_setup = time.perf_counter() - t0

    st = torch.cuda.ExternalStream(eng.stream())
    dZ = torch.from_numpy(w['Z']).cuda(); dS = torch.from_numpy(w['Sigma']).cuda()
    d_mean = torch.empty(H, Ny, dtype=torch.float64, device='cuda')
    d_var = torch.empty_like(d_mean)
    d_cov = torch.empty(H, Ny, Ny, dtype=torch.float64, device='cuda')
    d_jac = torch.empty(H, Ny, Nx, dtype=torch.float64, device='cuda')
    torch.cuda.synchronize()

    def step_dev():
        eng.predict_device(L.METHOD_TA, H, dZ.data_ptr(), dS.data_ptr(), 0, d_mean.data_ptr(), d_var.data_ptr(),
                           d_cov.data_ptr(), d_jac.data_ptr(), sync=False)

    # model bytes touched per step on this rank: L^-1 lower triangles; larger than L2 => no flush
    model_bytes = n * 4 * N * N
    flush = model_bytes < 4 * 126e6
    fl = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device='cuda') if flush else None   # 256 MB

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step_dev()
    eng.synchronize()
    barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    with torch.cuda.stream(st):
        for e0, e1 in evs:
            if flush:
                fl.zero_()
            e0.record(st)
            step_dev()
            e1.record(st)
    eng.synchronize()
    barrier()
    if args.dump_outputs and rank == 0:       # every rank holds all Ny outputs after the gather
        dump_outputs(args.dump_outputs, mean=d_mean.cpu(), var=d_var.cpu(), cov=d_cov.cpu(), jac=d_jac.cpu())
    ms_total = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    clocks = sampler.stop()
    tm = torch.tensor([ms_total], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_step = float(tm.item()) / args.steps
    value = H / (ms_step * 1e-3)

    # ---- e2e through the host C-ABI call (host buffers, H2D + D2H inside the timed region) ----
    for _ in range(2):
        eng.predict(w['Z'], w['Sigma'], L.METHOD_TA)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        mean, var, cov, jac = eng.predict(w['Z'], w['Sigma'], L.METHOD_TA)
    barrier()
    te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = H * args.steps / float(te.item())
    h2d = (H * Nx + Nx * Nx) * 8
    d2h = (2 * H * Ny + H * Ny * Nx + H * Ny * Ny) * 8

    # ---- roofline of the dominant kernel: v = L^-1 ks on the fp64 tensor pipe -----------------
    # algorithmic work per launch (DESIGN.md): flops = n_local * H * N^2, bytes = n_local * 4 N^2
    ms_tri = eng.profile(L.PROF_TRIGEMM, n=H, reps=max(5, args.steps))
    flops = n * H * float(N) * N
    achieved = flops / (ms_tri * 1e-3) / 1e12
    # fp64 tensor peak is not in MEASURED_PEAKS.json (bf16 only): measure cuBLAS DGEMM here, as a
    # burst (best of 4, for kernels timed alone) and sustained (back to back for ~4 s, clocks sampled)
    a = torch.randn(8192, 8192, dtype=torch.float64, device='cuda'); bmat = torch.randn_like(a)
    best = 1e9
    for _ in range(4):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, bmat); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    dgemm_tf = 2 * 8192.0 ** 3 / (best * 1e-3) / 1e12
    sustained = None
    if rank == 0 and os.environ.get('GPMPC_BENCH_SUSTAINED', '1') == '1':
        n_it = max(8, int(4000.0 / best))
        smp = ClockSampler(local_rank); smp.start()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_it):
            torch.matmul(a, bmat)
        e1.record(); torch.cuda.synchronize()
        ck = smp.stop()
        sustained = {'tflops': 2 * 8192.0 ** 3 * n_it / (e0.elapsed_time(e1) * 1e-3) / 1e12, 'iters': n_it,
                     'seconds': e0.elapsed_time(e1) * 1e-3, 'clocks': ck}
    del a, bmat
    # write-only HBM bandwidth (the K build only writes): best of 5 fills of a 2 GiB buffer, for context beside the
    # copy-bandwidth denominator of MEASURED_PEAKS.json
    wbuf = torch.empty(1 << 28, dtype=torch.float64, device='cuda')
    wbest = 1e9
    for _ in range(5):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); wbuf.fill_(1.0); e1.record(); torch.cuda.synchronize()
        wbest = min(wbest, e0.elapsed_time(e1))
    hbm_write_gbs = wbuf.numel() * 8 / wbest / 1e6
    del wbuf
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    hbm_src = 'MEASURED_PEAKS.json (measured)' if peaks else 'fallback 6650 GB/s'
    traffic = None
    tj = {}
    try:      # per-launch DRAM bytes from the committed ncu capture (profiles/), same workload only
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json')))
        if N == 16384 and H == 50:
            traffic = n * tj['trigemm_N16384_H50_per_output_bytes']
    except Exception:
        pass
    roofline = {'bound': 'tensor', 'kernel': PREDICT_KERNEL_NAME,
                'achieved': achieved, 'peak': dgemm_tf, 'unit': 'TFLOP/s', 'frac': achieved / dgemm_tf,
                'peak_source': 'cuBLAS DGEMM 8192^3 burst (best of 4) measured in this run; fp64 is absent from MEASURED_PEAKS.json',
                'peak_sustained': sustained, 'frac_vs_sustained': (achieved / sustained['tflops']) if sustained else None,
                'ms_per_launch': ms_tri, 'traffic': traffic, 'algorithmic_bytes': n * 4.0 * N * N,
                'hbm_view': {'algorithmic_gbs': n * 4.0 * N * N / (ms_tri * 1e-3) / 1e9, 'peak_gbs': hbm_peak,
                             'peak_source': hbm_src}}
    # secondary kernels (BASELINE north_star targets: >=0.70 HBM on the K build, >=0.80 tensor on the
    # Cholesky trailing update), one output at this N; algorithmic work per DESIGN.md section 4
    secondary = None
    if sec:
        Np = (N + 127) // 128 * 128
        n1 = (Np // 128 // 2) * 128; n2 = Np - n1
        syrk_flops = float(n2) * (n2 + 1) * n1                # lower triangle incl. the diagonal, 2 flops per multiply-add
        secondary = {
            'kbuild_full': {'ms': sec['kbuild_full_ms'], 'gbs': 8.0 * Np * Np / sec['kbuild_full_ms'] / 1e6,
                            'frac': 8.0 * Np * Np / sec['kbuild_full_ms'] / 1e6 / hbm_peak, 'bound': 'hbm',
                            'algorithmic_bytes': 8.0 * Np * Np, 'traffic': tj.get('kbuild_full_N16384_bytes') if N == 16384 else None,
                            'write_only_peak_gbs': hbm_write_gbs, 'frac_of_write_only_peak': 8.0 * Np * Np / sec['kbuild_full_ms'] / 1e6 / hbm_write_gbs,
                            'peak_source': hbm_src},
            'kbuild_lower': {'ms': sec['kbuild_lower_ms'], 'gbs': 4.0 * Np * (Np + 1) / sec['kbuild_lower_ms'] / 1e6,
                             'frac': 4.0 * Np * (Np + 1) / sec['kbuild_lower_ms'] / 1e6 / hbm_peak, 'bound': 'hbm',
                             'algorithmic_bytes': 4.0 * Np * (Np + 1)},
            'syrk_trailing_update': {'ms': sec['syrk_ms'], 'tflops': syrk_flops / sec['syrk_ms'] / 1e9,
                                     'frac': syrk_flops / sec['syrk_ms'] / 1e9 / dgemm_tf, 'bound': 'tensor',
                                     'shape': 'C(%d x %d lower) -= P P^T, K=%d' % (n2, n2, n1),
                                     'traffic': tj.get('syrk_8192x8192_K8192_bytes') if N == 16384 else None},
            'factorize_potrf_trtri': {'ms': sec['factorize_ms'], 'tflops': (2.0 / 3.0) * float(Np) ** 3 / sec['factorize_ms'] / 1e9,
                                      'frac': (2.0 / 3.0) * float(Np) ** 3 / sec['factorize_ms'] / 1e9 / dgemm_tf, 'bound': 'tensor',
                                      'note': 'K build + potrf + explicit L^-1 of one output, 2N^3/3 flops'},
        }
        if rank == 0 and world == 1:
            # sequential H=1 predicts (examples/van_der_pol.py:34-38: 2000 gp.predict calls in a Python loop): the
            # HBM-bound regime -- every step streams the lower triangle of every output's L^-1 once
            z1 = np.ascontiguousarray(w['Z'][:1])
            for _ in range(3):
                eng.predict(z1, None, L.METHOD_ME, want_jac=False)
            t1 = time.perf_counter(); n1 = 50
            for _ in range(n1):
                eng.predict(z1, None, L.METHOD_ME, want_jac=False)
            ms1 = (time.perf_counter() - t1) / n1 * 1e3
            secondary['sequential_h1'] = {'ms_per_call_e2e': ms1, 'calls_per_s': 1e3 / ms1, 'bound': 'hbm',
                                          'algorithmic_bytes': n * 4.0 * Np * (Np + 1), 'gbs': n * 4.0 * Np * (Np + 1) / ms1 / 1e6,
                                          'frac': n * 4.0 * Np * (Np + 1) / ms1 / 1e6 / hbm_peak,
                                          'note': 'host C-ABI call per step (H2D + 2 launches + D2H + sync inside), method ME, N=%d, %d outputs' % (N, n)}
        if rank == 0 and world == 1 and os.environ.get('GPMPC_BENCH_NLML', '1') == '1':
            # BASELINE config C4: NLML + analytic gradient at N=8192, Nx=8 (one output) through the C ABI
            w4 = make_workload(8192, 8, 1, 4, 1)
            e4 = gp_mpc_b200.Engine(8192, 8, 1, 0, 1, device=local_rank)
            e4.set_data(w4['X'], w4['Y'])
            e4.nlml(0, w4['hyper'][0], grad=True)
            t1 = time.perf_counter()
            for _ in range(3):
                e4.nlml(0, w4['hyper'][0], grad=True)
            ms_g = (time.perf_counter() - t1) / 3 * 1e3
            t1 = time.perf_counter()
            for _ in range(3):
                e4.nlml(0, w4['hyper'][0], grad=False)
            ms_v = (time.perf_counter() - t1) / 3 * 1e3
            e4.close()
            secondary['nlml_c4'] = {'ms_value_and_grad': ms_g, 'ms_value_only': ms_v, 'N': 8192, 'Nx': 8,
                                    'tflops': 8192.0 ** 3 / ms_g / 1e9, 'frac': 8192.0 ** 3 / ms_g / 1e9 / dgemm_tf,
                                    'note': 'host-timed C-ABI call (sync inside); N^3 flops = potrf N^3/3 + trtri N^3/3 + K^-1 N^3/3'}

    # ---- parity against an INDEPENDENT CPU factor (rank 0, every N) + CPU baseline (N=1) --------
    cpu = None
    parity = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import gp_oracle as orc
        _limits = all_host_threads()
        _limits.__enter__()
        outs = sorted({0, Ny - 1})          # rank 0's own first output and the last rank's last output
        ref = {}
        t_fac = 0.0
        for a_o in outs:
            t1 = time.perf_counter()
            f = orc.factor_large(w['X'], w['Y'][:, a_o], w['hyper'][a_o])
            t_fac += time.perf_counter() - t1
            ref[a_o] = (f,) + tuple(orc.predict_large(w['X'], w['hyper'][a_o], f['alpha'], f['chol'], w['Z']))
        def rel(x, y):
            return float(np.abs(x - y).max() / max(np.abs(y).max(), 1e-300))
        pm = max(rel(mean[:, a_o], ref[a_o][1]) for a_o in outs)
        pv = max(rel(var[:, a_o], ref[a_o][2]) for a_o in outs)
        pj = max(rel(jac[:, a_o], ref[a_o][3]) for a_o in outs)
        vo = np.stack([ref[a_o][2] for a_o in outs], 1); Jo = np.stack([ref[a_o][3] for a_o in outs], 1)
        co = orc.ta_cov(vo, Jo, w['Sigma'])
        pc = rel(cov[:, outs][:, :, outs], co)
        parity = {'mean': pm, 'var': pv, 'jac': pj, 'cov': pc, 'max': max(pm, pv, pj, pc), 'tol': 1e-6,
                  'ok': bool(max(pm, pv, pj, pc) < 1e-6), 'outputs_checked': outs,
                  'how': 'independent CPU factor (np.linalg.cholesky of the expansion-form K, triangular solves) of outputs '
                         '%s at full N=%d; gathered GPU result of the e2e call compared, batch-inf-norm relative' % (outs, N)}
        if world == 1:
            f0 = ref[0][0]
            reps = 0; tt = 0.0
            while tt < 10.0 and reps < 5:
                t1 = time.perf_counter()
                cpu_predict_port(orc, w['X'], w['hyper'][0], f0['alpha'], f0['chol'], w['Z'])
                tt += time.perf_counter() - t1; reps += 1
            t_one = tt / reps
            cpu = {'value': H / (t_one * Ny), 'unit': 'predictions/s', 'cores': os.cpu_count(), 'kind': 'port',
                   'sample': 'oracle port of the numeric predict (ks, mean, L\\ks triangular solve, var, Jacobian) for 1 of '
                             '%d outputs at full N=%d, H=%d, %d reps, time x Ny; CPU factor (%.1f s per output) not timed'
                             % (Ny, N, H, reps, t_fac / len(outs))}
        del ref

    if rank == 0:
        line = {'metric': METRIC, 'value': value, 'unit': 'predictions/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong',
                'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': {'workload': wl['name'], 'method': 'TA', 'N': N, 'Nx': Nx, 'Ny': Ny, 'H': H,
                           'parallelism': 'outputs sharded %d/GPU, %s' % (n, 'single GPU' if world == 1 else (
                               'epilogue stores to NVLink peer buffers (fused all-gather)' if peer_mode else 'NCCL all-gather')),
                           'l2': 'flush 256MB between steps' if flush else 'model %.1f GB/rank > L2, no flush' % (model_bytes / 1e9),
                           'setup_s': t_setup},
                'clocks': clocks,
                'e2e': {'value': e2e_val, 'unit': 'predictions/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h},
                # per 64-point chunk: ks_mean_jac_kernel + predict_streamk_kernel (the latter also reduces, finalizes,
                # stores to the peers and assembles); a separate assemble_kernel only for H > 64 or the NCCL fallback
                'gpu_launches': args.steps * (2 * ((H + 63) // 64) + (1 if (H > 64 or (world > 1 and not peer_mode)) else 0)),
                'roofline': roofline, 'roofline_secondary': secondary, 'parity_vs_oracle': parity, 'cpu_baseline': cpu}
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
