"""float32 vs float64 storage of Y on one GPU: step and kernel times, memory peaks, and the largest n that fits.

    python tools/bench_y32.py --out DIR [--iters 20] [--warmup 3] [--rounds 5]

1. config 4 (n = 8192, T = 128, r = 8, 'good', lr 0.01) with float32 Y from generate_data_device(dtype=torch.float32),
   then the same configuration with float64 Y in the same process: ms per iteration, k_sweep / ELBO-pass ms
   (tame_last_timing), the fraction of the measured HBM copy bandwidth at 16 algorithmic bytes per dyad-timestep, and
   torch.cuda.max_memory_allocated of each run.
2. A/B at n = 6144, T = 128, r = 8 with both copies of Y resident: float32 and float64 handles alternate for --rounds
   rounds; per-round ms per iteration and the spread.
3. capacity: n = 12288, T = 128, r = 8 with float32 Y for a few sweeps, stepping n down by 512 until it fits; node-level
   parity of the last sweep against the oracle's update_node at spot nodes (as tests/test_gpu_scale.py does).
Prints one JSON object per section and writes them to DIR/bench_y32.jsonl."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "python-temporal-ame-svi_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import tame_oracle as orc  # noqa: E402
from tame_b200 import TemporalAMEModel, _lib  # noqa: E402
from tame_b200.inference import _bind_Y, _fit_config  # noqa: E402

DEV = torch.device("cuda", 0)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[1] if len(q) > 1 else "unknown"


def hbm_peak_gbs(gib=8, reps=10):
    """device-to-device copy bandwidth (read + write bytes / time), best of `reps`"""
    a = torch.empty(gib << 28, dtype=torch.float32, device=DEV)
    b = torch.empty_like(a)
    best = 0.0
    for _ in range(reps + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


class Fit:
    """one handle over a model's Y (float32 or float64) with a seeded random start state on the device"""

    def __init__(self, model, Y, lr=0.01, mode=_lib.MODE_GOOD, seed=1):
        self.lib = _lib.load()
        n, T, r, d = model.n, model.T, model.r, model.d
        vi = types.SimpleNamespace(model=model, n=n, T=T, r=r, d=d, _mode=mode, lr=lr)
        self.cfg, self._keep = _fit_config(vi, DEV.index)
        g = torch.Generator(device=DEV).manual_seed(seed)
        self.Y = Y
        self.Xm = 0.1 * torch.randn(n, T, d, generator=g, dtype=torch.float64, device=DEV)
        B = 0.1 * torch.randn(n, T, d, 2, generator=g, dtype=torch.float64, device=DEV)
        self.Xc = (0.5 * torch.eye(d, dtype=torch.float64, device=DEV) + B @ B.transpose(-1, -2)).contiguous()
        del B
        torch.cuda.synchronize()
        self.h = C.c_void_p()
        _lib.check(self.lib.tame_create(C.byref(self.cfg), C.byref(self.h)))
        _lib.check(_bind_Y(self.lib, self.h, Y))
        _lib.check(self.lib.tame_bind_state(self.h, self.Xm.data_ptr(), self.Xc.data_ptr()))
        _lib.check(self.lib.tame_set_timing(self.h, 1))
        self.out = (C.c_double * 6)()

    def iterate(self, k):
        """k iterations; returns per-iteration (ms, sweep_ms, k_sweep_ms, elbo_ms, llmse_ms)"""
        rows = []
        for _ in range(k):
            t0 = time.perf_counter()
            _lib.check(self.lib.tame_iterate(self.h, self.out))
            ms = (time.perf_counter() - t0) * 1e3
            v = [C.c_double() for _ in range(5)]
            _lib.check(self.lib.tame_last_timing(self.h, *[C.byref(x) for x in v]))
            sweep, elbo, _contract, chain, llmse = (x.value for x in v)
            rows.append((ms, sweep, chain, elbo, llmse))
        return np.array(rows)

    def close(self):
        if self.h:
            self.lib.tame_destroy(self.h)
            self.h = C.c_void_p()


def model_of(n, T=128, r=8, seed=42):
    return TemporalAMEModel(n_nodes=n, n_time=T, latent_dim=r, ar_coefficient=0.8, rho_dyadic=0.5, seed=seed)


def config4(dtype, args, peak):
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats(DEV)
    m = model_of(8192)
    Y = m.generate_data_device(device=DEV, dtype=dtype, seed=11)
    f = Fit(m, Y)
    try:
        f.iterate(args.warmup)
        t = f.iterate(args.iters)
        med = np.median(t, axis=0)
        n, T = m.n, m.T
        return dict(section="config4", y_dtype=str(dtype).replace("torch.", ""), n=n, T=T, r=m.r, iters=args.iters,
                    ms_per_iter_median=med[0], ms_per_iter_min=float(t[:, 0].min()), sweep_ms=med[1], k_sweep_ms=med[2],
                    elbo_ms=med[3], k_llmse_ms=med[4], elbo=float(f.out[0]),
                    frac_hbm_peak_at_16B=16.0 * n * n * T / (med[0] * 1e-3) / 1e9 / peak,
                    max_memory_allocated_GB=torch.cuda.max_memory_allocated(DEV) / 1e9,
                    device_used_GB=(torch.cuda.mem_get_info(DEV)[1] - torch.cuda.mem_get_info(DEV)[0]) / 1e9)
    finally:
        f.close()
        del f, Y, m
        torch.cuda.empty_cache()


def ab(args):
    torch.cuda.empty_cache()
    m = model_of(6144)
    Y64 = m.generate_data_device(device=DEV, dtype=torch.float64, seed=12)
    Y32 = Y64.float()
    f32, f64 = Fit(m, Y32), Fit(m, Y64)
    try:
        f32.iterate(args.warmup), f64.iterate(args.warmup)
        per = {"float32": [], "float64": []}
        for _ in range(args.rounds):
            for name, f in (("float32", f32), ("float64", f64)):
                per[name].append(float(np.median(f.iterate(5)[:, 0])))
        res = dict(section="ab_n6144", n=6144, T=128, r=8, rounds=args.rounds, iters_per_round=5)
        for name, v in per.items():
            v = np.array(v)
            res[name] = dict(ms_rounds=v.round(3).tolist(), median=float(np.median(v)), min=float(v.min()), max=float(v.max()))
        res["f32_over_f64_per_round"] = (np.array(per["float32"]) / np.array(per["float64"])).round(4).tolist()
        return res
    finally:
        f32.close(), f64.close()
        del f32, f64, Y32, Y64
        torch.cuda.empty_cache()


class _OneRow:
    def __init__(self, i, rows):
        self.i, self.rows = i, rows

    def __getitem__(self, k):
        return self.rows[k[1]]

    def __setitem__(self, k, v):
        self.rows[k[1]] = v


def capacity(args):
    n = 12288
    while n >= 8192:
        torch.cuda.empty_cache()
        f = Y = None
        try:
            m = model_of(n)
            Y = m.generate_data_device(device=DEV, dtype=torch.float32, seed=13)
            f = Fit(m, Y, lr=0.3)
            f.iterate(2)
            break
        except (torch.OutOfMemoryError, RuntimeError) as e:
            print(f"capacity: n={n} does not fit: {str(e).splitlines()[0][:160]}", flush=True)
            if f is not None:
                f.close()
            f = Y = m = None                 # m.Y holds the generated Y as well
            n -= 512
    if n < 8192:
        return dict(section="capacity", largest_n=None)
    try:
        c = orc.derived_constants(dict(n=n, T=m.T, r=m.r, d=m.d, R=m.R.double().numpy(), R_inv=m.R_inv.double().numpy(),
                                       Sigma=m.Sigma.double().numpy(), Psi=m.Psi.double().numpy(),
                                       Phi=m.Phi.double().numpy(), Q=m.Q.double().numpy()))
        rng = np.random.default_rng(n)
        spots = sorted({0, 1, 31, 32, 63, 64, n // 2, n // 2 + 17, n - 33, n - 1, *rng.integers(0, n, 6).tolist()})
        old_m = f.Xm.cpu().numpy()
        old_c = {i: f.Xc[i].cpu().numpy() for i in spots}
        t = f.iterate(1)
        new_m = f.Xm.cpu().numpy()
        worst_m = worst_c = 0.0
        mix = new_m.copy()
        for i in spots:
            mix[:i] = new_m[:i]
            mix[i:] = old_m[i:]
            row = f.Y[i].double().cpu().numpy()[None]
            cov = _OneRow(i, old_c[i].copy())
            orc.update_node(row, mix, cov, i, c, 0.3, orc.GOOD, row=0)
            got_c = f.Xc[i].cpu().numpy()
            worst_m = max(worst_m, float(np.max(np.abs(mix[i] - new_m[i])) / np.max(np.abs(mix[i]))))
            worst_c = max(worst_c, float(np.max(np.abs(cov.rows - got_c)) / np.max(np.abs(cov.rows))))
        free, total = torch.cuda.mem_get_info(DEV)
        return dict(section="capacity", largest_n=n, T=m.T, r=m.r, y_GB=f.Y.numel() * 4 / 1e9, ms_per_iter=float(t[0, 0]),
                    device_used_GB=(total - free) / 1e9, device_total_GB=total / 1e9, spot_nodes=len(spots),
                    worst_rel_err_mean=worst_m, worst_rel_err_cov=worst_c)
    finally:
        f.close()
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--sections", default="config4,ab,capacity")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    lines = [dict(section="gpu", name_power_limit_max_sm_clock=gpu_info())]
    peak = hbm_peak_gbs()
    lines.append(dict(section="hbm", copy_GBs=peak))
    for line in lines:
        print(json.dumps(line), flush=True)
    secs = args.sections.split(",")
    if "config4" in secs:
        for dt in (torch.float32, torch.float64):
            lines.append(config4(dt, args, peak))
            print(json.dumps(lines[-1]), flush=True)
    if "ab" in secs:
        lines.append(ab(args))
        print(json.dumps(lines[-1]), flush=True)
    if "capacity" in secs:
        lines.append(capacity(args))
        print(json.dumps(lines[-1]), flush=True)
    with open(os.path.join(args.out, "bench_y32.jsonl"), "w") as fh:
        for line in lines:
            fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
