"""Time predict, predict_grad and predict_hess ('TA', one GPU) at C2 / C3 / C5 and rate the W = L^-1 dks product.

    python tools/bench_hess.py [--reps R] [--warmup W] [--out profiles/bench_hess.json]

Call times: host clock around the synchronous C-ABI calls (each ends in a stream synchronise), median of R after W
warm-up calls of the same shape.  W-product time: a torch.profiler run per workload (separate from the timed calls)
sums the predict_streamk_kernel time of one predict_hess call and subtracts that of one predict_grad call on the same
inputs (predict_hess runs the same v and beta products, then the W passes on the same kernel).  Its rate is
n_loc * Nx * H * N^2 flop (H*Nx right-hand sides of a triangular product per output) over that time, reported
against the cuBLAS DGEMM rate (torch.matmul, fp64, 8192^3, CUDA events) measured in the same run.  The GPU name and
power limit are recorded with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np

CONFIGS = [('C2', 1000, 8, 6, 30, 2), ('C3', 4096, 8, 6, 30, 3), ('C5', 16384, 10, 8, 50, 5)]


def gpu_info():
    import torch
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def dgemm_rate(n=8192, reps=10):
    import torch
    a = torch.randn(n, n, dtype=torch.float64, device='cuda'); b = torch.randn(n, n, dtype=torch.float64, device='cuda')
    for _ in range(3):
        torch.matmul(a, b)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch.matmul(a, b)
    e1.record(); torch.cuda.synchronize()
    return 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) * 1e-3)


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), float(np.min(ts))


def streamk_us(fn):
    """predict_streamk_kernel device time (us) of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    tot = 0.0
    for ev in prof.events():
        if ev.device_type.name == 'CUDA' and 'predict_streamk_kernel' in ev.name:
            tot += ev.device_time if hasattr(ev, 'device_time') else ev.cuda_time
    return tot


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'bench_hess.json'))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_hess: needs a CUDA device')
    import gp_mpc_b200
    from gp_mpc_b200 import _lib as L
    from bench import make_workload
    info = gpu_info()
    gemm = dgemm_rate()
    res = dict(gpu=info, dgemm_flops=gemm, reps=a.reps, warmup=a.warmup, configs=[])
    for name, N, Nx, Ny, H, cfg in CONFIGS:
        w = make_workload(N, Nx, Ny, cfg, H)
        eng = gp_mpc_b200.Engine(N, Nx, Ny, device=0)
        eng.set_data(w['X'], w['Y']); eng.set_hyper(w['hyper']); eng.factorize()
        Z, S = w['Z'], w['Sigma']
        row = dict(name=name, N=N, Nx=Nx, Ny=Ny, H=H)
        for key, fn in (('predict', lambda: eng.predict(Z, S, L.METHOD_TA)),
                        ('predict_grad', lambda: eng.predict_grad(Z, S, L.METHOD_TA, want_hess=True)),
                        ('predict_hess', lambda: eng.predict_hess(Z, S, L.METHOD_TA))):
            med, mn = timed(fn, a.reps, a.warmup)
            row[key + '_ms'] = 1e3 * med
            row[key + '_min_ms'] = 1e3 * mn
        sk_grad = streamk_us(lambda: eng.predict_grad(Z, S, L.METHOD_TA, want_hess=True))
        sk_hess = streamk_us(lambda: eng.predict_hess(Z, S, L.METHOD_TA))
        w_us = sk_hess - sk_grad
        flops = float(Ny) * Nx * H * float(N) ** 2
        row.update(streamk_grad_us=sk_grad, streamk_hess_us=sk_hess, w_product_us=w_us, w_flop=flops,
                   w_flops=flops / (w_us * 1e-6) if w_us > 0 else None)
        row['w_vs_dgemm'] = row['w_flops'] / gemm if row['w_flops'] else None
        print(json.dumps(row), flush=True)
        res['configs'].append(row)
        eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=info, dgemm_tflops=gemm / 1e12)))


if __name__ == '__main__':
    main()
