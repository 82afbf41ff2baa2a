#!/usr/bin/env python
"""bench.py -- dyad-timesteps/s of the Temporal-AME structured mean-field VI fit loop on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 4|3|n,T,r] [--dump-outputs DIR]

One "step" = one iteration of fit(): a full Gauss-Seidel sweep + ELBO + reconstruction MSE ("good" SMF, FP64),
i.e. n^2 * T dyad-timesteps.  At N GPUs the SAME problem is node-sharded (strong scaling).  Workload: BASELINE
config 4 (n=8192, T=128, r=8; Y = 137.4 GB FP64) when it fits the GPU, else the largest n that does.

Prints ONE JSON line (rank 0).  `value` is measured with inputs resident in HBM; `e2e` goes through the
host-buffer C-ABI entry (tame_fit_host: pinned host Y/state -> device -> fit -> state back) at the SAME n, copies
inside the timed region; `roofline` is the dominant streaming kernel against the measured HBM peak; `cpu_baseline`
is the oracle port timed on the host cores on a FIXED sample (CPU_SAMPLE_NODES nodes of the workload), the same
sample `--impl reference` times, so the two arms describe one configuration.  `extra` carries BASELINE configs 3
(200 sweeps, three reciprocity values) and 5 (512 batched fits).  --impl reference also times the unmodified
reference (copied to oracle/_ref at build time, when present) on BASELINE config 1.

--dump-outputs DIR writes what the last timed step handed back (ELBO, its parts, MSE, the variational state) as
float64 .npy files; the inputs are seeded, so two builds run with the same arguments can be compared file by file.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "python-temporal-ame-svi_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

CONFIGS = {"4": (8192, 128, 8), "3": (1024, 64, 4), "2": (50, 20, 2), "1": (15, 10, 2)}
HYPER = dict(ar_coefficient=0.8, rho_additive=0.5, rho_multiplicative=0.3, rho_dyadic=0.5)
LR = 0.01
METRIC = "SMF-VI dyad-timesteps/sec (N^2*T per sweep; sweep + ELBO + MSE per step)"
UNIT = "dyad-timesteps/s"
PANEL = int(os.environ.get("TAME_PANEL", "64"))    # nodes per ownership panel of the multi-GPU fit (multiple of 64)
CPU_SAMPLE_NODES = 384      # fixed node subsample of the workload timed on the host (cpu_baseline and --impl reference)
DUMP_STATE_BYTES = 60 << 20     # --dump-outputs: state rows kept so that all files together stay under 64 MB


def parse_shape(s):
    if s in CONFIGS:
        return CONFIGS[s]
    n, T, r = (int(x) for x in s.split(","))
    return n, T, r


def kernel_source_hash():
    import hashlib
    h = hashlib.sha256()
    for name in ("tame_kernels.cuh", "tame_ops.cu"):
        with open(os.path.join(PKG, "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def measured_traffic(n, T, r, kernel="k_sweep"):
    """DRAM bytes per launch of the sweep kernel from the committed ncu capture (profiles/r02_traffic.json).  None
    unless the capture was taken at this configuration AND from the kernel sources that are in the tree now."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            t = json.load(f)
        if (t["n"], t["T"], t["r"]) == (n, T, r) and t.get("source_hash") == kernel_source_hash():
            return t[kernel]["dram_bytes"]
    except Exception:
        pass
    return None


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons.  Started before the warm-up (nvidia-smi needs a moment to start); only the
    samples whose wall-clock time falls inside the timed region are reported (all samples if none does)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=None, t1=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = [r for (ts, r) in self.rows if t0 is None or (t0 - 0.02 <= ts <= t1 + 0.08)]
        window = "timed region"
        if not rows:
            rows, window = [r for (_, r) in self.rows], "warm-up + timed region"
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "window": window, "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------
# CPU arm (oracle port)
# ----------------------------------------------------------------------------------------------------------
def cpu_sample_problem(n_s, T, r, seed=42):
    from oracle import tame_oracle as orc
    rng = np.random.default_rng(seed)
    c = orc.model_constants(n_s, T, r, **HYPER)
    d = c["d"]
    L0 = np.linalg.cholesky(c["S0"])
    Lq = np.linalg.cholesky(c["Q"])
    X = np.zeros((n_s, T, d))
    X[:, 0] = rng.standard_normal((n_s, d)) @ L0.T
    for t in range(1, T):
        X[:, t] = X[:, t - 1] @ c["Phi"].T + rng.standard_normal((n_s, d)) @ Lq.T
    Lr = np.linalg.cholesky(c["R"])
    Y = np.zeros((n_s, n_s, T, 2))
    iu = np.triu_indices(n_s, 1)
    for t in range(T):
        mu = orc.compute_mean(X[:, t, :2], X[:, t, 2:], r)
        yt = (mu + rng.standard_normal((n_s, n_s, 2)) @ Lr.T)[iu]
        Y[iu[0], iu[1], t] = yt
        Y[iu[1], iu[0], t, 0] = yt[:, 1]
        Y[iu[1], iu[0], t, 1] = yt[:, 0]
    Xm = rng.standard_normal((n_s, T, d)) * 0.1
    G = rng.standard_normal((n_s, T, d, d)) * 0.01
    Xc = 0.6 * np.eye(d) + 0.5 * (G + np.swapaxes(G, -1, -2))
    return c, Y, Xm, Xc


def cpu_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([p.get("num_threads", 1) for p in threadpool_info()] + [1])
    except Exception:
        return os.cpu_count() or 1


def cpu_arm(shape, steps, warmup):
    """Oracle port (sweep_fast + ELBO + MSE, all host threads NumPy/BLAS uses) on the FIXED sample: the first
    CPU_SAMPLE_NODES nodes' worth of the workload (same T, r, hyper-parameters, distribution)."""
    from oracle import tame_oracle as orc
    n, T, r = shape
    n_s = min(n, CPU_SAMPLE_NODES)
    c, Y, Xm, Xc = cpu_sample_problem(n_s, T, r)
    for _ in range(warmup):
        orc.sweep_fast(Y, Xm, Xc, c, LR, orc.GOOD)
        orc.elbo_mse_fast(Y, Xm, Xc, c, orc.GOOD)
    t0 = time.perf_counter()
    for _ in range(steps):
        orc.sweep_fast(Y, Xm, Xc, c, LR, orc.GOOD)
        orc.elbo_mse_fast(Y, Xm, Xc, c, orc.GOOD)
    dt = time.perf_counter() - t0
    value = (n_s ** 2) * T * steps / dt
    return value, dt / steps * 1e3, (f"oracle port (NumPy, literal Gauss-Seidel order) on a fixed {n_s}-node sample of the n={n} "
                                     f"workload, T={T}, r={r}, {steps} iteration(s) after {warmup} warm-up")


def reference_python_arm(max_iter=3):
    """The UNMODIFIED reference (src/models + src/inference copied to oracle/_ref by build()) on BASELINE config 1
    (demo.py: n=15, T=10, r=2, good SMF, lr 0.01), float64, timed like experiments/utils.py:201-203."""
    ref_root = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "src", "inference")):
        return {"unavailable": "oracle/_ref/src not present (build() copies it when /root/reference exists)"}
    import importlib
    import torch
    saved = {k: v for k, v in sys.modules.items() if k == "src" or k.startswith("src.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, ref_root)
    old = torch.get_default_dtype()
    try:
        torch.set_default_dtype(torch.float64)
        torch.set_num_threads(1)
        models = importlib.import_module("src.models")
        inference = importlib.import_module("src.inference")
        model = models.TemporalAMEModel(n_nodes=15, n_time=10, latent_dim=2, ar_coefficient=0.8, rho_dyadic=0.5, seed=42)
        model.generate_data()
        vi = inference.TemporalAMEStructuredMFVI(model, factorization="good", learning_rate=0.01, seed=42)
        t0 = time.time()
        hist = vi.fit(max_iter=max_iter, tolerance=0.0, verbose=False)
        dt = time.time() - t0
        return {"value": 15 * 15 * 10 * max_iter / dt, "unit": UNIT, "cores": 1, "kind": "reference",
                "sample": f"unmodified reference (oracle/_ref), config 1 (n=15 T=10 r=2, good SMF, lr 0.01), {max_iter} fit iterations, float64, 1 thread",
                "seconds": dt, "elbo_last": float(hist["elbo"][-1])}
    except Exception as e:                      # the reference arm must never take the bench down
        return {"unavailable": f"{type(e).__name__}: {e}"}
    finally:
        torch.set_default_dtype(old)
        sys.path.remove(ref_root)
        for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def config_dict(n, T, r, world, requested_n=None):
    """The `config` object of the JSON line -- ONE function for both arms, so that they describe the same configuration."""
    requested_n = n if requested_n is None else requested_n
    workload = f"good SMF fit iteration, n={n} T={T} r={r}, lr={LR}" + ("" if n == requested_n else f" (n reduced from {requested_n}: HBM)")
    units = float(n) * n * T
    par = f"node-sharded x{world} ({PANEL}-node panels, cyclic" + (")" if world == 1 else (
        ", panel scheduler + NCCL broadcasts)" if os.environ.get("TAME_SWEEP") == "panel" else ", fused sweep with NVLink peer hand-over)"))
    return {"workload": workload, "n": n, "T": T, "r": r, "method": "good", "lr": LR, "parallelism": par,
            "l2": f"inputs larger than L2: each step streams Y twice ({2 * 16.0 * units / world / 1e9:.1f} GB per GPU per step)"}


def run_reference(args, shape):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    value, ms, sample = cpu_arm(shape, args.steps, args.warmup)
    n, T, r = shape
    cores = cpu_threads()
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_dict(n, T, r, max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "reference_python": reference_python_arm(),
        "note": ("the reference is pure Python/torch-CPU (5-13 k dyad-timesteps/s): the line's value is its NumPy port on the "
                 "fixed sample of this workload; `reference_python` is the unmodified reference itself on BASELINE config 1"),
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------
def make_cfg(lib_mod, c, n, T, r, device, world, rank):
    cfg = lib_mod.TameConfig()
    cfg.n, cfg.T, cfg.r, cfg.mode = n, T, r, lib_mod.MODE_GOOD
    cfg.lr = LR
    for k, v in enumerate(np.asarray(c["R_inv"]).reshape(-1)):
        cfg.Rinv[k] = float(v)
    cfg.logdet_R, cfg.logdet_Q, cfg.logdet_S0 = float(c["logdet_R"]), float(c["logdet_Q"]), float(c["logdet_S0"])
    keep = [np.ascontiguousarray(c[k], dtype=np.float64) for k in ("Phi", "Q_inv", "S0_inv")]
    cfg.Phi, cfg.Qinv, cfg.S0inv = (lib_mod.dptr(a) for a in keep)
    cfg.device, cfg.world, cfg.rank, cfg.panel = device, world, rank, PANEL
    return cfg, keep


def hyper_constants(n, T, r, ar=None, rho=None):
    """Same hyper-parameters as TemporalAMEModel builds (static_ame.py:96-127, temporal_ame.py:129-145); computed with
    numpy here so bench.py's GPU arm does not import the oracle."""
    d = 2 + 2 * r

    def eq(dim, corr, var):
        m = np.full((dim, dim), corr * var)
        np.fill_diagonal(m, var)
        return m
    R = eq(2, HYPER["rho_dyadic"] if rho is None else rho, 0.1)
    S0 = np.zeros((d, d))
    S0[:2, :2] = eq(2, HYPER["rho_additive"], 1.0)
    S0[2:2 + r, 2:2 + r] = eq(r, HYPER["rho_multiplicative"], 1.0)
    S0[2 + r:, 2 + r:] = eq(r, HYPER["rho_multiplicative"], 1.0)
    phi = HYPER["ar_coefficient"] if ar is None else ar
    Q = (1 - phi ** 2) * S0 * 0.1
    return dict(n=n, T=T, r=r, d=d, R=R, R_inv=np.linalg.inv(R), S0=S0, S0_inv=np.linalg.inv(S0), Q=Q, Q_inv=np.linalg.inv(Q),
                Phi=np.eye(d) * phi, logdet_R=np.linalg.slogdet(R)[1], logdet_Q=np.linalg.slogdet(Q)[1],
                logdet_S0=np.linalg.slogdet(S0)[1])


def gen_latents(c, seed=42):
    import torch
    g = torch.Generator().manual_seed(seed)
    n, T, d = c["n"], c["T"], c["d"]
    L0 = torch.from_numpy(np.linalg.cholesky(c["S0"]))
    Lq = torch.from_numpy(np.linalg.cholesky(c["Q"]))
    Phi = torch.from_numpy(c["Phi"])
    X = torch.zeros(n, T, d, dtype=torch.float64)
    X[:, 0] = torch.randn(n, d, generator=g, dtype=torch.float64) @ L0.T
    for t in range(1, T):
        X[:, t] = X[:, t - 1] @ Phi.T + torch.randn(n, d, generator=g, dtype=torch.float64) @ Lq.T
    return X


def init_state(n, T, d, dev, seed=42):
    """'good' initialisation (structured_mf.py:77-90) in distribution, vectorised on the device."""
    import torch
    g = torch.Generator(device=dev).manual_seed(seed)
    Xm = torch.randn(n, T, d, generator=g, dtype=torch.float64, device=dev) * 0.1
    Xc = torch.randn(n, T, d, d, generator=g, dtype=torch.float64, device=dev) * 0.01
    Xc = (Xc + Xc.transpose(-1, -2)) / 2
    Xc += torch.eye(d, dtype=torch.float64, device=dev) * 0.6
    return Xm, Xc


def dump_outputs(path, Xm, Xc, out6):
    """What one fit iteration returns to its caller: the ELBO, its four parts (expected log-likelihood, initial prior,
    transition prior, entropy), the reconstruction MSE and the variational state, as float64 .npy files.  X_mean and
    X_cov hold all nodes when they fit DUMP_STATE_BYTES, else a fixed, seeded sample of nodes (every time step of each);
    node_index.npy lists which."""
    import torch
    n, T, d = Xm.shape
    k = min(n, DUMP_STATE_BYTES // (T * d * (d + 1) * 8))
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    sel = torch.from_numpy(idx).to(Xm.device)
    arrays = {"elbo": out6[0], "elbo_parts": out6[1:5], "reconstruction_error": out6[5], "node_index": idx,
              "X_mean": Xm.index_select(0, sel).cpu().numpy(), "X_cov": Xc.index_select(0, sel).cpu().numpy()}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_ours(args, shape):
    import torch
    import torch.distributed as dist
    from tame_b200 import _lib
    from tame_b200.sharding import owned_rows
    lib = _lib.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    n, T, r = shape
    d = 2 + 2 * r
    # fit the workload into HBM: Y rows of this rank + state + scratch, keep 6 GB of slack
    free_b, total_b = torch.cuda.mem_get_info(dev)
    def need(nn):
        return (nn * nn * T * 2 * 8) / world + nn * T * d * d * 8 * 2.4 + nn * T * d * 8 * 4 + 6e9
    requested_n = n
    while need(n) > free_b and n > 256:
        n -= 256
    c = hyper_constants(n, T, r)

    X = gen_latents(c).to(dev)
    rows = owned_rows(n, PANEL, world, rank)
    nloc = sum(b - a for a, b in rows)
    Y = torch.empty(nloc, n, T, 2, dtype=torch.float64, device=dev)
    Rflat = np.ascontiguousarray(c["R"].reshape(4))
    at = 0
    stream = torch.cuda.current_stream(dev).cuda_stream
    for a, b in rows:
        _lib.check(lib.tame_generate_Y(n, T, r, _lib.dptr(Rflat), X.data_ptr(), C.c_uint64(42), a, b,
                                       Y[at:at + (b - a)].data_ptr(), stream))
        at += b - a
    Xm, Xc = init_state(n, T, d, dev)
    torch.cuda.synchronize(dev)

    cfg, keep = make_cfg(_lib, c, n, T, r, local_rank, world, rank)
    h = C.c_void_p()
    _lib.check(lib.tame_create(C.byref(cfg), C.byref(h)))
    if world > 1:
        idbuf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = (C.c_ubyte * 128)()
            _lib.check(lib.tame_comm_unique_id(raw))
            idbuf = torch.tensor(list(raw), dtype=torch.uint8)
        idbuf = idbuf.to(dev)
        dist.broadcast(idbuf, 0)
        raw = (C.c_ubyte * 128)(*idbuf.cpu().tolist())
        _lib.check(lib.tame_comm_init(h, raw))
        if os.environ.get("TAME_SWEEP") != "panel":
            # fused multi-GPU sweep: exchange the CUDA IPC handles of the hand-over buffers
            mine = (C.c_ubyte * 64)()
            _lib.check(lib.tame_ipc_export(h, mine))
            table = [torch.zeros(64, dtype=torch.uint8, device=dev) for _ in range(world)]
            dist.all_gather(table, torch.tensor(list(mine), dtype=torch.uint8, device=dev))
            flat = torch.cat(table).cpu().tolist()
            _lib.check(lib.tame_ipc_import(h, (C.c_ubyte * (64 * world))(*flat)))
            dist.barrier()
    _lib.check(lib.tame_bind_Y(h, Y.data_ptr()))
    _lib.check(lib.tame_bind_state(h, Xm.data_ptr(), Xc.data_ptr()))
    y_sym = bool(lib.tame_y_symmetric(h))
    _lib.check(lib.tame_set_timing(h, 1))
    out6 = (C.c_double * 6)()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        _lib.check(lib.tame_iterate(h, out6))
    launches0 = lib.tame_launch_count()
    barrier()
    wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kt = np.zeros(5)
    e0.record()
    elbos = []
    for _ in range(args.steps):
        _lib.check(lib.tame_iterate(h, out6))
        elbos.append(out6[0])
        tm = [C.c_double() for _ in range(5)]
        lib.tame_last_timing(h, *[C.byref(x) for x in tm])
        kt += np.array([x.value for x in tm])
    e1.record()
    barrier()
    wall1 = time.time()
    if args.dump_outputs:
        _lib.check(lib.tame_gather_state(h))      # N > 1: covariance rows from their owners (nothing to do on one GPU)
        if rank == 0:
            dump_outputs(args.dump_outputs, Xm, Xc, out6)
    probes = (C.c_uint64 * 16)()
    lib.tame_debug_probes(h, probes)
    probes = list(probes)
    if os.environ.get("TAME_TRACE") and rank == 0:
        nsb = (n + 31) // 32
        tr = (C.c_uint64 * (22 * nsb))()
        if lib.tame_debug_trace(h, tr, 22 * nsb) == 0:
            tr = np.array(list(tr), dtype=np.float64)
            t0_ = float(probes[0])
            hw, ut, rl = tr[:2 * nsb].reshape(nsb, 2), tr[2 * nsb:6 * nsb].reshape(nsb, 4), tr[6 * nsb:].reshape(nsb, 16)
            # columns (us since the chain's start): helper starts waiting, helper released | unit claimed, upper done, group-0 urgent, group-0 stamped
            np.save(os.environ.get("TAME_TRACE_OUT", "gpurun_out/trace.npy"), np.concatenate([(hw - t0_) / 1e3, (ut - t0_) / 1e3, (rl - t0_) / 1e3], 1))
    ms = e0.elapsed_time(e1)
    launches = lib.tame_launch_count() - launches0
    if world > 1:
        tms = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    kt /= args.steps   # per-step ms: sweep, elbo, contract, chain, llmse
    units = float(n) * n * T
    value = units * args.steps / (ms * 1e-3)
    peak, peak_src = measured_peak()

    # ---- the step after the fit (SURVEY.md 8f-2): align the fitted means with the true latents on the device
    align = None
    if world == 1 and rank == 0:
        out_al = torch.empty_like(Xm)
        mse_al = C.c_double(0.0)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for rep in range(2 + 5):
            if rep == 2:
                a0.record()
            _lib.check(lib.tame_align_states(n, T, r, Xm.data_ptr(), X.data_ptr(), 1, out_al.data_ptr(), None, None, stream))
        a1.record()
        _lib.check(lib.tame_align_states(n, T, r, Xm.data_ptr(), X.data_ptr(), 1, out_al.data_ptr(), None, C.byref(mse_al), stream))
        al_ms = a0.elapsed_time(a1) / 5
        al_bytes = 5.0 * n * T * d * 8            # X_est and X_true read twice (cross-covariance, apply), aligned written once
        align = {"op": "align_temporal_states + alignment error (src/utils/alignment.py:224-385)", "ms": al_ms,
                 "achieved": al_bytes / (al_ms * 1e-3) / 1e9, "unit": "GB/s", "algorithmic_bytes": al_bytes,
                 "mse_after_alignment": mse_al.value}
        if not args.no_cpu:
            from oracle import align_oracle
            xe_h, xt_h = Xm.cpu().numpy(), X.cpu().numpy()
            t0 = time.time()
            ref_al = align_oracle.align_temporal_states(xe_h, xt_h, r)
            align["cpu_port_ms"] = (time.time() - t0) * 1e3
            align["max_abs_diff_vs_port"] = float(np.max(np.abs(out_al.cpu().numpy() - ref_al)))
            del xe_h, xt_h, ref_al
        del out_al
        # contribution / U'V diagnostics (SURVEY.md 8f-3) on the same arrays
        d_add = torch.empty(T, dtype=torch.float64, device=dev)
        d_mul = torch.empty(T, dtype=torch.float64, device=dev)
        d_cor = torch.empty(T, dtype=torch.float64, device=dev)
        for rep in range(2 + 5):
            if rep == 2:
                a0.record()
            _lib.check(lib.tame_contributions(n, T, r, Xm.data_ptr(), 1, d_add.data_ptr(), d_mul.data_ptr(), stream))
            _lib.check(lib.tame_uv_correlation(n, T, r, Xm.data_ptr(), X.data_ptr(), d_cor.data_ptr(), stream))
        a1.record()
        torch.cuda.synchronize(dev)
        dg_ms = a0.elapsed_time(a1) / 5
        dg_bytes = 7.0 * n * T * d * 8            # contributions: X_est twice; correlation: X_est 3x, X_true 2x (row sums + Grams + cross)
        align["diagnostics"] = {"op": "compute_temporal_contributions + compute_uv_correlation_over_time (diagnostics.py:170-217, multiplicative_strength_comparison.py:46-89)",
                                "ms": dg_ms, "achieved": dg_bytes / (dg_ms * 1e-3) / 1e9, "unit": "GB/s", "algorithmic_bytes": dg_bytes,
                                "uv_corr_t0": float(d_cor[0].item())}
        if not args.no_cpu:
            from oracle import diag_oracle
            ts = [0, T - 1]
            xe_h, xt_h = Xm[:, ts].cpu().numpy(), X[:, ts].cpu().numpy()
            t0 = time.time()
            o_add, o_mul = diag_oracle.temporal_contributions(xe_h, r, True)
            o_cor = diag_oracle.uv_correlation_over_time(xe_h, xt_h, r)
            align["diagnostics"]["cpu_port_ms"] = (time.time() - t0) * 1e3 * T / len(ts)
            align["diagnostics"]["cpu_port_sample"] = f"{len(ts)} of {T} time steps, scaled"
            align["diagnostics"]["max_abs_diff_vs_port"] = float(max(np.max(np.abs(d_add[ts].cpu().numpy() - o_add)),
                                                                       np.max(np.abs(d_mul[ts].cpu().numpy() - o_mul)),
                                                                       np.max(np.abs(d_cor[ts].cpu().numpy() - o_cor))))
            del xe_h, xt_h

    # ---- N > 1: self-check of the sharded sweep (the GPU test box of the driver has one GPU): one more sweep, then spot
    # nodes of rank 0 re-derived with the oracle's update_node from "new means below i, old means from i on" + row i of Y
    parity = None
    if world > 1:
        parity = multi_gpu_parity(lib, _lib, h, c, Y, Xm, Xc, rows, rank, dev)

    # ---- e2e through host buffers (single GPU): pinned host Y/state -> tame_fit_host -> state back, at the SAME n
    e2e = None
    cpu = None
    extra = None
    if world == 1 and rank == 0 and not args.no_e2e:
        lib.tame_destroy(h)
        h = None
        host, n_e, why = None, n, None
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = None
        while avail is not None and n_e * n_e * T * 16 * 1.05 + 6e9 > avail and n_e > 256:
            n_e -= 256
            why = f"host RAM: {avail / 1e9:.0f} GB available, Y at n={n} needs {n * n * T * 16 / 1e9:.0f} GB pinned"
        while host is None:
            if n_e != n:                      # regenerate the smaller problem on the device
                Y = Xm = Xc = X = None
                torch.cuda.empty_cache()
                c_e = hyper_constants(n_e, T, r)
                X = gen_latents(c_e).to(dev)
                Y = torch.empty(n_e, n_e, T, 2, dtype=torch.float64, device=dev)
                _lib.check(lib.tame_generate_Y(n_e, T, r, _lib.dptr(Rflat), X.data_ptr(), C.c_uint64(42), 0, n_e, Y.data_ptr(), stream))
                Xm, Xc = init_state(n_e, T, d, dev)
            try:
                host = {}
                for k, v in (("Y", Y), ("Xm", Xm), ("Xc", Xc)):
                    host[k] = torch.empty(v.shape, dtype=torch.float64, pin_memory=True)
                    host[k].copy_(v)
            except RuntimeError as e:         # pinning that much memory failed: shrink and say so
                host = None
                why = f"pinned allocation failed at n={n_e} ({str(e)[:80]})"
                n_e = max(256, (int(n_e * 0.8) // 256) * 256)
        torch.cuda.synchronize(dev)
        Y = Xm = Xc = X = None
        torch.cuda.empty_cache()
        e2e = run_e2e(lib, _lib, (n_e, T, r), n, host, args.steps, dev, why)
        del host
    if world == 1 and rank == 0:
        torch.cuda.empty_cache()
        if not args.no_extra:
            extra = {}
            for name, fn in (("config3", extra_config3), ("config5", extra_config5)):
                try:
                    extra[name] = fn(lib, _lib, dev)
                except Exception as e:        # a side measurement must not take the headline down
                    extra[name] = {"error": f"{type(e).__name__}: {e}"}
        if not args.no_cpu:
            v, msc, sample = cpu_arm((n, T, r), max(1, min(args.steps, 2)), 1)
            cpu = {"value": v, "unit": UNIT, "cores": cpu_threads(), "kind": "port", "sample": sample}
    if h is not None:
        lib.tame_destroy(h)

    if rank == 0:
        # per-GPU rates: rank 0 streams units/world dyad-timesteps per pass
        fused = kt[2] < 0.01 * kt[3]          # single GPU: the sweep is one persistent kernel (k_sweep)
        sweep_kernel_ms = kt[3] if fused else kt[2]
        contract_gbs = 16.0 * units / world / (sweep_kernel_ms * 1e-3) / 1e9 if sweep_kernel_ms > 0 else None
        llmse_gbs = 16.0 * units / world / (kt[4] * 1e-3) / 1e9 if kt[4] > 0 else None

        step_gbs = 32.0 * units / world / (ms / args.steps * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic (device Philox generator, same distribution as generate_data)",
            "config": config_dict(n, T, r, world, requested_n),
            "roofline": {"kernel": ("k_sweep (persistent fused Gauss-Seidel sweep: streaming CTAs contract Y with the partner means while the chain CTAs walk the nodes)"
                                    if fused else "k_contract (partner contraction of the sweep: static upper part + right-looking pushes, summed over its launches in one step)"),
                         "bound": "hbm", "achieved": contract_gbs, "peak": peak, "unit": "GB/s",
                         "frac": (contract_gbs / peak) if contract_gbs else None,
                         "traffic": measured_traffic(n, T, r) if (fused and world == 1) else None, "peak_source": peak_src,
                         "algorithmic_bytes_per_unit": 16, "units_per_step": units,
                         "step": {"achieved": step_gbs, "frac": step_gbs / peak, "algorithmic_bytes_per_unit": 32},
                         "kernels_ms_per_step": {"sweep_total": kt[0], "elbo_total": kt[1], "k_contract": kt[2], ("k_sweep" if fused else "k_chain"): kt[3], "k_llmse": kt[4]},
                         "k_llmse": {"achieved": llmse_gbs, "frac": (llmse_gbs / peak) if llmse_gbs else None,
                                     "algorithmic_bytes_per_unit": 16,
                                     "streamed_bytes_per_unit": 8 if y_sym else 16,
                                     "achieved_streamed": (llmse_gbs * (0.5 if y_sym else 1.0)) if llmse_gbs else None,
                                     "frac_streamed": (llmse_gbs * (0.5 if y_sym else 1.0) / peak) if llmse_gbs else None,
                                     "note": ("Y verified mirror-consistent at bind: the pass streams the i<j half (8 B per unit); "
                                              "frac is on the 16 B contract, frac_streamed on the bytes actually read") if y_sym else
                                             "full pass (16 B per unit)"}},
            "clocks": clocks, "gpu_launches": int(launches), "elbo_trace_tail": elbos[-2:], "chain_probes": probes,
        }
        if align:
            line["align"] = align
        if e2e:
            line["e2e"] = e2e
        if extra:
            line["extra"] = extra
        if parity:
            line["parity"] = parity
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_e2e(lib, _lib, shape, n_full, host, steps, dev, why=None):
    """tame_fit_host with pinned host buffers (host = dict(Y, Xm, Xc) of pinned CPU tensors)."""
    n_e, T, r = shape
    c = hyper_constants(n_e, T, r)
    cfg, keep = make_cfg(_lib, c, n_e, T, r, dev.index, 1, 0)
    el = np.zeros(steps); msq = np.zeros(steps); nd = C.c_int32(0)
    Yh, Xmh, Xch = host["Y"], host["Xm"], host["Xc"]
    t0 = time.perf_counter()
    _lib.check(lib.tame_fit_host(C.byref(cfg), Yh.data_ptr(), Xmh.data_ptr(), Xch.data_ptr(), steps, 0.0,
                                 _lib.dptr(el), _lib.dptr(msq), C.byref(nd)))
    dt = time.perf_counter() - t0
    units = float(n_e) * n_e * T
    h2d = (Yh.numel() + Xmh.numel() + Xch.numel()) * 8
    d2h = (Xmh.numel() + Xch.numel()) * 8 + steps * 6 * 8
    out = {"value": units * nd.value / dt, "unit": UNIT, "h2d_bytes_per_step": h2d / nd.value, "d2h_bytes_per_step": d2h / nd.value,
           "seconds": dt, "steps": int(nd.value), "n": n_e,
           "api": "tame_fit_host (C ABI, pinned host buffers; timed region = device alloc + H2D of Y and state + fit + D2H of state)"}
    out["same_config"] = (n_e == n_full)
    if n_e != n_full:
        out["note"] = f"host-buffer run uses n={n_e} (host Y = {n_e * n_e * T * 16 / 1e9:.1f} GB) instead of n={n_full}: {why}"
    return out


def multi_gpu_parity(lib, _lib, h, c, Y, Xm, Xc, rows, rank, dev, n_spots=3):
    """After the timed region at N > 1: snapshot the means, run ONE more sweep on all ranks, and let rank 0 re-derive a
    few of ITS nodes with the oracle's update_node (structured_mf.py:220-287) from 'new means below i, old means from
    i on' + row i of Y.  Returns the worst relative errors (rank 0) -- the 1e-9 bar of north_star applies."""
    import torch
    from oracle import tame_oracle as orc
    oc = orc.derived_constants(dict(n=c["n"], T=c["T"], r=c["r"], d=c["d"], R=c["R"], Sigma=c["S0"][:2, :2], Psi=c["S0"][2:, 2:],
                                   Phi=c["Phi"], Q=c["Q"]))
    n = c["n"]
    # spot nodes of rank 0: first node, a sub-block / refresh / panel boundary of its second panel, its last node
    mine = [i for (a, b) in rows for i in range(a, b)]
    spots = sorted({mine[0], mine[min(len(mine) - 1, 64)], mine[min(len(mine) - 1, 64 + 33)], mine[-1]})[:max(1, n_spots + 1)]
    old_m = Xm.cpu().numpy() if rank == 0 else None
    old_c = {i: Xc[i].cpu().numpy() for i in spots} if rank == 0 else None
    _lib.check(lib.tame_sweep(h))
    torch.cuda.synchronize(dev)
    if rank != 0:
        return None

    class OneRow:
        def __init__(self, i, blk): self.i, self.rows = i, blk
        def __getitem__(self, k): return self.rows[k[1]]
        def __setitem__(self, k, v): self.rows[k[1]] = v
    new_m = Xm.cpu().numpy()
    local_of = {}
    at = 0
    for a, b in rows:
        for i in range(a, b):
            local_of[i] = at + (i - a)
        at += b - a
    wm = wc = 0.0
    mix = new_m.copy()
    for i in spots:
        mix[:i] = new_m[:i]
        mix[i:] = old_m[i:]
        row = Y[local_of[i]].cpu().numpy()[None]
        cov = OneRow(i, old_c[i].copy())
        orc.update_node(row, mix, cov, i, oc, LR, orc.GOOD, row=0)
        wm = max(wm, float(np.max(np.abs(mix[i] - new_m[i])) / np.max(np.abs(mix[i]))))
        wc = max(wc, float(np.max(np.abs(cov.rows - Xc[i].cpu().numpy())) / np.max(np.abs(cov.rows))))
    return {"mean": wm, "cov": wc, "spot_nodes": spots, "tolerance": 1e-9, "ok": bool(wm < 1e-9 and wc < 1e-9),
            "how": "one extra sweep after the timed region; oracle update_node on rank 0's spot nodes (new means below i, old from i on)"}


def extra_config3(lib, _lib, dev, sweeps=200):
    """BASELINE config 3: good SMF, n=1024 T=64 r=4, 200 sweeps (fit iterations), reciprocity rho in {0, 0.5, 0.8}."""
    import torch
    n, T, r = CONFIGS["3"]
    d = 2 + 2 * r
    stream = torch.cuda.current_stream(dev).cuda_stream
    peak, _ = measured_peak()
    out = {"workload": f"good SMF, n={n} T={T} r={r}, lr={LR}, {sweeps} fit iterations (sweep + ELBO + MSE), inputs resident", "runs": []}
    for rho in (0.0, 0.5, 0.8):
        c = hyper_constants(n, T, r, rho=rho)
        X = gen_latents(c).to(dev)
        Y = torch.empty(n, n, T, 2, dtype=torch.float64, device=dev)
        _lib.check(lib.tame_generate_Y(n, T, r, _lib.dptr(np.ascontiguousarray(c["R"].reshape(4))), X.data_ptr(), C.c_uint64(42), 0, n,
                                       Y.data_ptr(), stream))
        Xm, Xc = init_state(n, T, d, dev)
        cfg, keep = make_cfg(_lib, c, n, T, r, dev.index, 1, 0)
        h = C.c_void_p()
        _lib.check(lib.tame_create(C.byref(cfg), C.byref(h)))
        _lib.check(lib.tame_bind_Y(h, Y.data_ptr()))
        _lib.check(lib.tame_bind_state(h, Xm.data_ptr(), Xc.data_ptr()))
        el = np.zeros(sweeps); ms = np.zeros(sweeps); nd = C.c_int32(0)
        _lib.check(lib.tame_fit(h, 3, 0.0, _lib.dptr(el), _lib.dptr(ms), C.byref(nd)))        # warm-up
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(lib.tame_fit(h, sweeps, 0.0, _lib.dptr(el), _lib.dptr(ms), C.byref(nd)))
        e1.record()
        torch.cuda.synchronize(dev)
        per = e0.elapsed_time(e1) / nd.value
        gbs = 32.0 * n * n * T / (per * 1e-3) / 1e9
        out["runs"].append({"rho": rho, "ms_per_step": per, "value": float(n) * n * T / (per * 1e-3), "unit": UNIT,
                            "step_frac_of_hbm_peak": gbs / peak, "elbo_first": float(el[0]), "elbo_last": float(el[nd.value - 1]),
                            "mse_last": float(ms[nd.value - 1])})
        lib.tame_destroy(h)
        del Y, X, Xm, Xc
    return out


def extra_config5(lib, _lib, dev, max_iter=150, tolerance=1e-4):
    """BASELINE config 5: 512 independent fits (n x T x ar x rho grid, r=2, naive + good) through tame_fit_batch."""
    import torch
    stream = torch.cuda.current_stream(dev).cuda_stream
    r = 2
    d = 2 + 2 * r
    ns, Ts, ars, rhos = [10, 20, 32, 50, 64, 100, 160, 256], [5, 10, 20, 40], [0.5, 0.9], [0.0, 0.3, 0.6, 0.8]
    problems = [(n, T, ar, rho) for n in ns for T in Ts for ar in ars for rho in rhos]
    nf = 2 * len(problems)
    cfgs = (_lib.TameConfig * nf)()
    Yp, Mp, Cp = (C.c_void_p * nf)(), (C.c_void_p * nf)(), (C.c_void_p * nf)()
    keep, f = [], 0
    for k, (n, T, ar, rho) in enumerate(problems):
        c = hyper_constants(n, T, r, ar=ar, rho=rho)
        X = gen_latents(c, seed=100 + k).to(dev)
        Y = torch.empty(n, n, T, 2, dtype=torch.float64, device=dev)
        _lib.check(lib.tame_generate_Y(n, T, r, _lib.dptr(np.ascontiguousarray(c["R"].reshape(4))), X.data_ptr(), C.c_uint64(100 + k), 0, n,
                                       Y.data_ptr(), stream))
        for mode in (_lib.MODE_NAIVE, _lib.MODE_GOOD):
            Xm, Xc = init_state(n, T, d, dev, seed=7 + k)
            cfg, kk = make_cfg(_lib, c, n, T, r, dev.index, 1, 0)
            cfg.mode = mode
            cfgs[f] = cfg
            keep.append((kk, Y, Xm, Xc))
            Yp[f], Mp[f], Cp[f] = Y.data_ptr(), Xm.data_ptr(), Xc.data_ptr()
            f += 1
    torch.cuda.synchronize(dev)
    el = np.zeros((nf, max_iter)); ms = np.zeros((nf, max_iter)); nd = (C.c_int32 * nf)()
    # warm-up (module load of the r=2 kernels, allocator): a few iterations of the first fits, then restore their state
    warm = min(nf, 16)
    saved = [(keep[f][2].clone(), keep[f][3].clone()) for f in range(warm)]
    _lib.check(lib.tame_fit_batch(warm, cfgs, Yp, Mp, Cp, 2, 0.0, _lib.dptr(el), _lib.dptr(ms), nd, 0))
    for f in range(warm):
        keep[f][2].copy_(saved[f][0]); keep[f][3].copy_(saved[f][1])
    torch.cuda.synchronize(dev)
    launches0 = lib.tame_launch_count()
    t0 = time.time()
    _lib.check(lib.tame_fit_batch(nf, cfgs, Yp, Mp, Cp, max_iter, tolerance, _lib.dptr(el), _lib.dptr(ms), nd, 0))
    torch.cuda.synchronize(dev)
    sec = time.time() - t0
    iters = np.array(list(nd), dtype=np.int64)
    units = sum(float(n) * n * T * float(it2.sum()) for (n, T, ar, rho), it2 in zip(problems, iters.reshape(-1, 2)))
    return {"workload": f"{nf} independent fits (n in {ns}, T in {Ts}, ar in {ars}, rho in {rhos}, r=2, naive + good), max_iter {max_iter}, "
                        f"tolerance {tolerance}, lr {LR}; inputs resident, traces to the host",
            "seconds": sec, "fits_per_s": nf / sec, "iterations_total": int(iters.sum()), "value": units / sec, "unit": UNIT,
            "early_stopped": int((iters < max_iter).sum()), "gpu_launches": int(lib.tame_launch_count() - launches0),
            "finite": bool(np.all(np.isfinite(el[np.arange(nf), iters - 1])))}



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="4", help="4 (default), 3, 2, 1 or n,T,r")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--no-extra", action="store_true", help="skip the config-3 / config-5 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    shape = parse_shape(args.config)
    if args.impl == "reference":
        run_reference(args, shape)
    else:
        run_ours(args, shape)


if __name__ == "__main__":
    main()
