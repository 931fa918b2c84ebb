"""Sweeps/s at C2 (4096 x 1024 x 64, 3 replicates, K = 16, 20 % NaN) of the Gaussian sampler in three modes, timed
alternately in one process so that clock and power drift hit them alike:
  scalar        scalar nu2, default route (integer statistics path where it applies)
  scalar_fp64   scalar nu2 with BTF_STATS_NO_I8=1 (FP64 statistics with count weights)
  per_cell      known per-cell variances (btf_set_nu2_cells): FP64 statistics with f64 weights, no nu2 step
The data and the variances are generated on the device.  Prints the card name and power limit beside the numbers.
usage: python tools/nu2_cells_bench.py [--rounds 3] [--steps 20]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

N, M, T, R, K = 4096, 1024, 64, 3, 16


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--steps', type=int, default=20)
    args = ap.parse_args()
    import torch
    from functionalmf_b200 import _lib as L
    from functionalmf_b200.engine import Engine
    dev = torch.device('cuda', 0)
    modes = ['scalar', 'scalar_fp64', 'per_cell']
    engines = {}
    for name in modes:
        if name == 'scalar_fp64':
            os.environ['BTF_STATS_NO_I8'] = '1'      # read when the engine is created
        engines[name] = Engine(N, M, T, nembeds=K, tf_order=2, seed=11)
        os.environ.pop('BTF_STATS_NO_I8', None)
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    V0 = (torch.randn(M, T, K, generator=g, device=dev, dtype=torch.float64) * 0.3).cumsum(1)
    for i, a in enumerate(range(0, N, 256)):
        W = torch.randn(256, K, generator=g, device=dev, dtype=torch.float64)
        Y = (W @ V0.reshape(M * T, K).T).reshape(256, M, T, 1) + \
            torch.randn(256, M, T, R, generator=g, device=dev, dtype=torch.float64)
        Y[torch.rand(Y.shape, generator=g, device=dev) < 0.2] = float('nan')
        torch.cuda.synchronize()
        for eng in engines.values():
            eng.set_data_gaussian_rows_device(Y.data_ptr(), a, 256, R, i == 0)
        del Y
    nu2 = torch.rand(N, M, T, generator=g, device=dev, dtype=torch.float64) + 0.5
    torch.cuda.synchronize()
    pc = engines['per_cell']
    L.check(pc.lib.btf_set_nu2_cells(pc._h, C.c_void_p(nu2.data_ptr())))
    del nu2
    for name, eng in engines.items():
        eng.init_state(127)
        if name == 'per_cell':
            eng.set_sample_mask(127 & ~L.SAMPLE_NU2)
        eng.sweep(5)
    ms = {name: [] for name in modes}
    for _ in range(args.rounds):
        for name in modes:
            ms[name].append(engines[name].sweep_timed(args.steps) / args.steps)
    out = {'card': card(), 'shape': [N, M, T, R, K], 'steps': args.steps,
           'i8_route': {name: list(engines[name].diag('i8_route')) for name in modes}}
    for name in modes:
        out[name] = {'sweeps_per_s': [round(1e3 / x, 2) for x in ms[name]], 'best_ms': round(min(ms[name]), 4)}
    print(json.dumps(out))


if __name__ == '__main__':
    main()
