"""Multi-GPU parity (needs >= 2 visible GPUs; skipped otherwise): the node-sharded fit on 2 ranks -- fused sweep with
NVLink peer hand-over, and the NCCL panel scheduler -- against the oracle."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

WORKER = r'''
import ctypes as C, os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.path.join(ROOT, "python-temporal-ame-svi_b200")); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from tame_b200 import _lib
from tame_b200.sharding import shard_rows
from oracle import tame_oracle as orc
from gpu_util import make_config, random_problem
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank); dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
lib = _lib.load()
n, T, r, lr, iters = 256, 9, 3, 0.3, 2
c, Y, Xm, Xc = random_problem(n, T, r, seed=77)
if os.environ.get("TAME_TEST_ASYM") == "1":
    Y = Y.copy(); Y[3, 200, 2, 0] += 0.125          # one dyad no longer mirror-consistent -> full ELBO pass on every rank
for meth in ("good", "naive"):
    mode = orc.MODE_OF[meth]
    cfg, keep = make_config(c, lr, mode, device=rank, world=world, rank=rank, panel=64)
    Yd = torch.as_tensor(shard_rows(Y, 64, world, rank)).to(dev).contiguous()
    Xmd, Xcd = torch.as_tensor(Xm).to(dev).contiguous(), torch.as_tensor(Xc).to(dev).contiguous()
    h = C.c_void_p(); _lib.check(lib.tame_create(C.byref(cfg), C.byref(h)))
    idb = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        raw = (C.c_ubyte * 128)(); _lib.check(lib.tame_comm_unique_id(raw)); idb = torch.tensor(list(raw), dtype=torch.uint8, device=dev)
    dist.broadcast(idb, 0)
    _lib.check(lib.tame_comm_init(h, (C.c_ubyte * 128)(*idb.cpu().tolist())))
    if os.environ.get("TAME_SWEEP") != "panel":
        mine = (C.c_ubyte * 64)(); _lib.check(lib.tame_ipc_export(h, mine))
        tab = [torch.zeros(64, dtype=torch.uint8, device=dev) for _ in range(world)]
        dist.all_gather(tab, torch.tensor(list(mine), dtype=torch.uint8, device=dev))
        _lib.check(lib.tame_ipc_import(h, (C.c_ubyte * (64 * world))(*torch.cat(tab).cpu().tolist())))
        dist.barrier()
    _lib.check(lib.tame_bind_Y(h, Yd.data_ptr())); _lib.check(lib.tame_bind_state(h, Xmd.data_ptr(), Xcd.data_ptr()))
    out = (C.c_double * 6)(); el = []
    for _ in range(iters):
        _lib.check(lib.tame_iterate(h, out)); el.append(out[0])
    _lib.check(lib.tame_gather_state(h)); torch.cuda.synchronize()
    Om, Oc = Xm.copy(), Xc.copy(); oel = []
    for _ in range(iters):
        orc.sweep_fast(Y, Om, Oc, c, lr, mode); oel.append(orc.elbo(Y, Om, Oc, c, mode))
    em = np.max(np.abs(Xmd.cpu().numpy() - Om)) / np.max(np.abs(Om)); ec = np.max(np.abs(Xcd.cpu().numpy() - Oc)) / np.max(np.abs(Oc))
    ee = max(abs(a - b) / abs(b) for a, b in zip(el, oel))
    assert em < 1e-9 and ec < 1e-9 and ee < 1e-9, (meth, em, ec, ee)
    lib.tame_destroy(h)
    if rank == 0: print("OK", meth, em, ec, ee, flush=True)
dist.destroy_process_group()
'''


@pytest.mark.parametrize("scheduler", ["fused", "panel", "fused-asymmetricY"])
def test_two_rank_fit_matches_oracle(tmp_path, scheduler):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "w.py"
    script.write_text(f"ROOT = {ROOT!r}\n" + WORKER)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    env = dict(os.environ)
    env.pop("TAME_SWEEP", None)
    env.pop("TAME_TEST_ASYM", None)
    if scheduler == "panel":
        env["TAME_SWEEP"] = "panel"
    if scheduler == "fused-asymmetricY":
        env["TAME_TEST_ASYM"] = "1"
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                          "127.0.0.1", "--master-port", str(port), str(script)], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-3000:]
    assert res.stdout.count("OK") == 2, res.stdout


def test_drop_in_devices_keyword_matches_single_gpu():
    """`TemporalAMEStructuredMFVI(model, devices=[0, 1])` (additive keyword, SURVEY.md section 5): one process, one handle per
    GPU, fused sweep with NVLink peer hand-over -- the same history and state as the single-GPU object at rel 1e-9."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import sys
    sys.path.insert(0, os.path.join(ROOT, "python-temporal-ame-svi_b200"))
    from src.models import TemporalAMEModel
    from src.inference import TemporalAMENaiveMFVI, TemporalAMEStructuredMFVI
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        model = TemporalAMEModel(n_nodes=128, n_time=6, latent_dim=2, ar_coefficient=0.8, rho_dyadic=0.5, seed=42)
        model.generate_data()
        for make in (lambda **kw: TemporalAMEStructuredMFVI(model, factorization="good", learning_rate=0.3, seed=42, **kw),
                     lambda **kw: TemporalAMENaiveMFVI(model, learning_rate=0.3, seed=42, **kw)):
            one, two = make(device="cuda:0"), make(devices=[0, 1])
            h1 = one.fit(max_iter=3, tolerance=0.0, verbose=False)
            h2 = two.fit(max_iter=3, tolerance=0.0, verbose=False)
            e1, e2 = np.array(h1["elbo"]), np.array(h2["elbo"])
            assert np.all(np.abs(e1 - e2) <= 1e-9 * np.abs(e1)), (e1, e2)
            assert torch.allclose(one.X_mean, two.X_mean, rtol=1e-9, atol=1e-12)
            assert torch.allclose(one.X_cov, two.X_cov, rtol=1e-9, atol=1e-12)
        with pytest.raises(ValueError):
            m2 = TemporalAMEModel(n_nodes=100, n_time=3, latent_dim=2, seed=42)
            m2.generate_data()
            TemporalAMEStructuredMFVI(m2, devices=[0, 1]).fit(max_iter=1, verbose=False)
    finally:
        torch.set_default_dtype(old)
