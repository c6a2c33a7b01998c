"""Time the FITC sparse build (gpmpc_fitc) and the predict step on a sparse handle (one GPU).

    python tools/bench_sparse.py [--reps R] [--warmup W] [--out profiles/bench_sparse.json]

Workloads (N, M, Ny) in {(16384, 2048, 8), (262144, 2048, 8), (1048576, 4096, 1)}, Nx = 10, synthetic data (sn = 0.1).
Per workload:
  * build time (host clock around the synchronous call) and its split from CUDA events inside the build
    (gpmpc_fitc_timings): Kuf build, V = Luu^-1 Kuf product, column pass, SYRK, M-sized factorisations;
  * the V product and the SYRK rated at Ny * Mpad^2 * Nq flop each (Nq = N rounded up to whole panels; the product
    skips the zero upper triangle of Luu^-1, the SYRK computes the lower tiles only, so both do about half of 2 M^2 N)
    against cuBLAS DGEMM (torch.matmul, fp64, 8192^3, CUDA events) measured in the same run;
  * the Kuf build's write rate, Ny * Mpad * Nq * 8 bytes, against device copy bandwidth (torch copy_, 2 GiB, read+write);
  * the predict step (H = 50, 'TA', median of R calls after W warm-up calls) on the sparse handle, next to a dense
    N = 16384 handle's step (Ny = 8) from the same run;
  * at the two smaller sizes a parity field: batch-inf-norm relative error of mean and var of output 0 at 16 test points
    against the Woodbury form of tests/_fitc_oracle.py (CPU, float64).
The GPU name and power limit are recorded with the numbers."""
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

WORKLOADS = [(16384, 2048, 8), (262144, 2048, 8), (1048576, 4096, 1)]
NX, H = 10, 50


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


def copy_bandwidth(nbytes=2 << 30, reps=10):
    import torch
    a = torch.empty(nbytes // 8, dtype=torch.float64, device='cuda').fill_(1.0); b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record(); torch.cuda.synchronize()
    return 2.0 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3)


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def synthetic(N, Ny, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, NX))
    W = rng.standard_normal((NX, Ny)) / np.sqrt(NX)
    Y = np.sin(X @ W) + 0.1 * rng.standard_normal((N, Ny))
    hyper = np.column_stack([rng.uniform(1.5, 3.0, (Ny, NX)), np.ones(Ny), np.full(Ny, 0.1)])
    return X, Y, hyper


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'bench_sparse.json'))
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_sparse: needs a CUDA device')
    import gp_mpc_b200
    from gp_mpc_b200 import _lib as L
    from tests import _fitc_oracle as fo
    info = gpu_info()
    gemm, bw = dgemm_rate(), copy_bandwidth()
    res = dict(gpu=info, dgemm_flops=gemm, copy_bytes_per_s=bw, reps=a.reps, warmup=a.warmup, H=H, Nx=NX, workloads=[])
    rng = np.random.default_rng(9)
    Z = 0.5 * rng.standard_normal((H, NX))
    S = 1e-4 * np.eye(NX)
    # dense N = 16384 reference step (Ny = 8)
    Xd, Yd, hd = synthetic(16384, 8, 16384)
    dense = gp_mpc_b200.Engine(16384, NX, 8, device=0)
    dense.set_data(Xd, Yd); dense.set_hyper(hd); dense.factorize()
    res['dense_16384_predict_ms'] = 1e3 * timed(lambda: dense.predict(Z, S, L.METHOD_TA), a.reps, a.warmup)
    dense.close()
    del Xd, Yd
    for N, M, Ny in WORKLOADS:
        X, Y, hyper = synthetic(N, Ny, N)
        U = X[fo.seeded_subset(N, M)]
        eng = gp_mpc_b200.Engine(M, NX, Ny, device=0)
        eng.set_data(U, np.zeros((M, Ny))); eng.set_hyper(hyper)
        eng.fitc(X, Y)                                              # warm-up (module load, attributes, tensor maps)
        t0 = time.perf_counter(); info_, nll = eng.fitc(X, Y); t_build = time.perf_counter() - t0
        ph = eng.fitc_timings()
        mp = (M + 127) // 128 * 128
        nq = (N + 4095) // 4096 * 4096
        fl = float(Ny) * mp * mp * nq
        kuf_bytes = float(Ny) * mp * nq * 8
        row = dict(N=N, M=M, Ny=Ny, build_ms=1e3 * t_build, phases_ms=ph, shifted=int(np.sum(info_)),
                   v_product_flops=fl / (ph['v_product'] * 1e-3), syrk_flops=fl / (ph['syrk'] * 1e-3),
                   kuf_bytes_per_s=kuf_bytes / (ph['kuf'] * 1e-3))
        row['v_product_vs_dgemm'] = row['v_product_flops'] / gemm
        row['syrk_vs_dgemm'] = row['syrk_flops'] / gemm
        row['kuf_vs_copy'] = row['kuf_bytes_per_s'] / bw
        row['predict_ms'] = 1e3 * timed(lambda: eng.predict(Z, S, L.METHOD_TA), a.reps, a.warmup)
        if N <= 262144:
            Zp = Z[:16]
            mw, vw, nw = fo.predict('woodbury', U, X, Y[:, :1], hyper[:1], Zp)
            mean, var, _, _ = eng.predict(Zp, None, L.METHOD_ME, want_cov=False, want_jac=False)
            row['parity_woodbury'] = dict(mean=float(np.abs(mean[:, 0] - mw[:, 0]).max() / np.abs(mw).max()),
                                          var=float(np.abs(var[:, 0] - vw[:, 0]).max() / np.abs(vw).max()),
                                          nll=float(abs(nll[0] - nw[0]) / abs(nw[0])))
        print(json.dumps(row), flush=True)
        res['workloads'].append(row)
        eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=info, dgemm_tflops=gemm / 1e12, copy_tb_per_s=bw / 1e12,
                          dense_16384_predict_ms=res['dense_16384_predict_ms'])))


if __name__ == '__main__':
    main()
