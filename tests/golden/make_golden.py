#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ by running the UNMODIFIED
reference (/root/reference, read-only) in float64.

This is test infrastructure: it only runs in the build container (the GPU box
has no /root/reference); the .npz files it writes are committed.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [case ...]

Recipe (SURVEY.md section 8c): torch.set_default_dtype(torch.float64) BEFORE the
model is constructed, then generate_data(), construct the VI object, fit().
Each fixture holds: the hyper-parameters, Y, the initial X_mean/X_cov (taken
right after construction, i.e. the RNG-order-exact init of
structured_mf.py:74-113 / naive_mf.py:71-87), the per-iteration ELBO and MSE
traces of base.py:127-208, the four ELBO parts of the final state and the final
X_mean/X_cov.
"""
import os
import sys
import time

import numpy as np

REF = os.environ.get("TAME_REFERENCE", "/root/reference")
sys.dont_write_bytecode = True
sys.path.insert(0, REF)

import torch  # noqa: E402

torch.set_default_dtype(torch.float64)
torch.set_num_threads(1)

from src.models import TemporalAMEModel  # noqa: E402
from src.inference import TemporalAMENaiveMFVI, TemporalAMEStructuredMFVI  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

# name -> (model kwargs, lr, max_iter, tolerance)
CASES = {
    # tests/conftest.py:35-43 shape
    "conftest_lr1": (dict(n_nodes=10, n_time=5, latent_dim=2, ar_coefficient=0.8, seed=42), 1.0, 6, 0.0),
    "conftest_lr001": (dict(n_nodes=10, n_time=5, latent_dim=2, ar_coefficient=0.8, seed=42), 0.01, 6, 0.0),
    # odd latent dim, strong reciprocity, T=1 edge (no AR neighbours at all) and T=2
    "r3_rho08": (dict(n_nodes=12, n_time=4, latent_dim=3, ar_coefficient=0.6, rho_dyadic=0.8,
                      rho_additive=0.2, rho_multiplicative=0.1), 0.3, 5, 0.0),
    "r1_T1": (dict(n_nodes=7, n_time=1, latent_dim=1, ar_coefficient=0.5, rho_dyadic=0.0), 0.5, 4, 0.0),
    "r4_T2": (dict(n_nodes=9, n_time=2, latent_dim=4, ar_coefficient=0.9, rho_dyadic=-0.4), 1.0, 4, 0.0),
    # early stopping (base.py:183-203): tiny lr converges in relative terms
    "earlystop": (dict(n_nodes=10, n_time=5, latent_dim=2, ar_coefficient=0.8, seed=42), 0.001, 100, 1.09e-3),
    # BASELINE config 1 (demo.py:49-101)
    "config1": (dict(n_nodes=15, n_time=10, latent_dim=2, ar_coefficient=0.8, rho_dyadic=0.5, seed=42), 0.01, 100, 0.0),
    # BASELINE config 2 shape (three_way_conparison), truncated to a few iterations: the
    # reference needs ~5-10 s per iteration here
    "config2": (dict(n_nodes=50, n_time=20, latent_dim=2), 0.01, 4, 0.0),
    # the same, 50 iterations of all three methods (~15 minutes of reference time): per-method ELBO-trace parity on
    # BASELINE config 2 proper (experiments/three_way_conparison.py:122-179 runs 500 at this step size)
    "config2_long": (dict(n_nodes=50, n_time=20, latent_dim=2), 0.01, 50, 0.0),
}

METHODS = {
    "naive": lambda m, lr: TemporalAMENaiveMFVI(m, learning_rate=lr, seed=42),
    "good": lambda m, lr: TemporalAMEStructuredMFVI(m, factorization="good", learning_rate=lr, seed=42),
    "bad": lambda m, lr: TemporalAMEStructuredMFVI(m, factorization="bad", learning_rate=lr, seed=42),
}

# Runs of one problem store its inputs once, with Y as its first channel (Y is mirror-consistent), so that every
# fixture stays under 1 MB; tests/conftest.py:load_golden joins them back.
SHARED_INPUTS = {"config2": "config2_inputs", "config2_long": "config2_inputs"}
RUN_KEYS = ["lr", "max_iter", "tolerance"] + [f"{m}_{k}" for m in METHODS
                                              for k in ("elbo", "mse", "parts", "final_mean", "final_cov")]


def run_case(name):
    kw, lr, max_iter, tol = CASES[name]
    model = TemporalAMEModel(**kw)
    Y, X = model.generate_data(return_latents=True)
    out = dict(
        Y=Y.numpy().copy(), X_true=X.numpy().copy(),
        R=model.R.numpy(), R_inv=model.R_inv.numpy(), Sigma=model.Sigma.numpy(), Psi=model.Psi.numpy(),
        Phi=model.Phi.numpy(), Q=model.Q.numpy(),
        n=model.n, T=model.T, r=model.r, lr=lr, max_iter=max_iter, tolerance=tol,
        model_kwargs=np.array(repr(kw)), torch_version=np.array(torch.__version__),
    )
    for meth, ctor in METHODS.items():
        t0 = time.time()
        vi = ctor(model, lr)
        out[f"{meth}_init_mean"] = vi.X_mean.numpy().copy()
        out[f"{meth}_init_cov"] = vi.X_cov.numpy().copy()
        hist = vi.fit(max_iter=max_iter, tolerance=tol, verbose=False)
        out[f"{meth}_elbo"] = np.array([float(e) for e in hist["elbo"]])
        out[f"{meth}_mse"] = np.array([float(e) for e in hist["reconstruction_error"]])
        out[f"{meth}_parts"] = np.array([
            float(vi._compute_expected_log_likelihood()), float(vi._compute_log_prior_initial()),
            float(vi._compute_log_prior_transitions()), float(vi._compute_entropy())])
        out[f"{meth}_final_mean"] = vi.X_mean.numpy().copy()
        out[f"{meth}_final_cov"] = vi.X_cov.numpy().copy()
        print(f"  {name}/{meth}: {len(hist['elbo'])} iters in {time.time() - t0:.1f}s "
              f"elbo[0]={out[f'{meth}_elbo'][0]:.10f} elbo[-1]={out[f'{meth}_elbo'][-1]:.10f}", flush=True)
    inputs = SHARED_INPUTS.get(name)
    if inputs is not None:
        shared = {k: v for k, v in out.items() if k not in RUN_KEYS}
        Y = shared.pop("Y")
        assert np.array_equal(Y[:, :, :, 1], np.swapaxes(Y[:, :, :, 0], 0, 1))
        np.savez_compressed(os.path.join(HERE, f"{inputs}.npz"), Y0=np.ascontiguousarray(Y[:, :, :, 0]), **shared)
        out = {"inputs": np.array(inputs), **{k: out[k] for k in RUN_KEYS}}
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **out)


if __name__ == "__main__":
    names = sys.argv[1:] or list(CASES)
    for nm in names:
        print(f"[golden] {nm}", flush=True)
        run_case(nm)
