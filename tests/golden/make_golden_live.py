#!/usr/bin/env python
"""Generates tests/golden/oracle_vs_ref.npz and tests/golden/lite_branin.npz by EXECUTING the reference (through
oracle/ref_shim.py); needs the reference tree (SPEARMINT_REFERENCE):
    python tests/golden/make_golden_live.py

oracle_vs_ref.npz   -- the reference's kernels, log-probabilities, compute_ei, Sobol generator and optimize_hypers on the
                       seeded problems of tests/test_oracle_vs_reference.py, with the exact inputs it was given.
lite_branin.npz     -- the reference's UNMODIFIED spearmint-lite controller proposing Branin experiments through the
                       drop-in chooser (loaded by name through the INTEGRATION.md stub, numerics from the oracle stand-in
                       backend): every chooser.next() call the controller made, with its arguments and what it returned.
                       tests/test_dropin_spearmint_lite.py replays those calls.
"""
import os
import shutil
import sys
import tempfile
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import ref_shim  # noqa: E402

KINDS = ["SE", "ARDSE", "Matern32", "Matern52"]


def _problem(seed, D=3, N=25, M=40):
    rs = np.random.RandomState(seed)
    comp, cand = rs.rand(N, D), rs.rand(M, D)
    y = np.sin(3 * comp).sum(1) + 0.05 * rs.randn(N)
    return comp, cand, (y - y.mean()) / y.std(), rs


def golden_oracle_vs_ref():
    R = ref_shim.load()
    gp, OPT, sb = R["gp"], R["OPT"], R["sobol_lib"]
    out = {}
    for kind in KINDS:
        comp, cand, vals, rs = _problem(1)
        ls = rs.uniform(0.4, 1.8, comp.shape[1])
        f = getattr(gp, kind)
        g = gp.GP(kind)
        g.real_init(comp.shape[1], vals)
        g.ls, g.amp2, g.noise, g.mean = ls, 1.3, 2e-3, 0.1
        out.update({"k_%s_comp" % kind: comp, "k_%s_cand" % kind: cand, "k_%s_vals" % kind: vals,
                    "k_%s_ls" % kind: ls, "k_%s_self" % kind: f(ls, comp), "k_%s_cross" % kind: f(ls, comp, cand),
                    "k_%s_logprob" % kind: g.logprob(comp, vals)})

    comp, cand, vals, rs = _problem(2)
    ch = OPT.init(tempfile.mkdtemp(), "mcmc_iters=2,burnin=1,use_multiprocessing=0")
    ch.D = comp.shape[1]
    np.random.seed(4)
    ch.randomstate = np.random.get_state()
    ch.mean, ch.noise, ch.amp2, ch.ls = 0.05, 1e-3, 0.9, rs.uniform(0.4, 1.8, ch.D)
    out.update(ei_comp=comp, ei_cand=cand, ei_vals=vals, ei_mean=ch.mean, ei_noise=ch.noise, ei_amp2=ch.amp2,
               ei_ls=ch.ls, ei_nopend=ch.compute_ei(comp, np.zeros((0, ch.D)), cand, vals))
    pend = rs.rand(2, ch.D)
    np.random.set_state(ch.randomstate)
    normals = np.random.randn(2, ch.pending_samples)          # what the reference draws after npr.set_state (OPT:588-589)
    out.update(ei_pend=pend, ei_normals=normals, ei_withpend=ch.compute_ei(comp, pend, cand, vals))

    out["sobol_6x50_skip2"] = sb.i4_sobol_generate(6, 50, 2)
    comp, cand, vals, rs = _problem(3, D=2, N=20)
    g = gp.GP("Matern52")
    g.real_init(2, vals)
    g.optimize_hypers(comp, vals)
    out.update(mll_comp=comp, mll_vals=vals, mll_mean=g.mean, mll_noise=g.noise, mll_amp2=g.amp2, mll_ls=g.ls)
    np.savez_compressed(os.path.join(HERE, "oracle_vs_ref.npz"), **out)


STUB = "from spearmint_b200.chooser.GPEIOptChooserB200 import *  # noqa: F401,F403\n"
CHOOSER_ARGS = "mcmc_iters=3,burnin=5,grid_subset=4,use_multiprocessing=0"
ITERS = 8


def branin(x):
    """spearmint/examples/braninpy/branin.py:6-16 (x in the unit square)."""
    x1, x2 = x[0] * 15 - 5, x[1] * 15
    return float(np.square(x2 - (5.1 / (4 * np.square(np.pi))) * np.square(x1) + (5 / np.pi) * x1 - 6)
                 + 10 * (1 - (1. / (8 * np.pi))) * np.cos(x1) + 10)


def golden_lite_branin():
    lite = ref_shim.load_lite()
    tmp = tempfile.mkdtemp()
    plug = os.path.join(tmp, "plugins")
    os.mkdir(plug)
    with open(os.path.join(plug, "GPEIOptChooserB200.py"), "w") as fh:
        fh.write(STUB)
    sys.modules["chooser"].__path__ = [plug]
    sys.modules.pop("chooser.GPEIOptChooserB200", None)
    import spearmint_b200.backend as be
    from spearmint_b200.chooser.GPEIOptChooserB200 import GPEIOptChooserB200 as cls
    from tests.oracle_backend import OracleBackend
    be.DeviceBackend = lambda **kw: OracleBackend()

    calls = []
    inner = cls.next

    def recording_next(self, grid, values, durations, candidates, pending, complete):
        ret = inner(self, grid, values, durations, candidates, pending, complete)
        calls.append(dict(grid=np.array(grid), values=np.array(values), durations=np.array(durations),
                          candidates=np.array(candidates), pending=np.array(pending), complete=np.array(complete),
                          ret_tuple=isinstance(ret, tuple), ret_index=ret[0] if isinstance(ret, tuple) else ret,
                          ret_point=np.array(ret[1] if isinstance(ret, tuple) else grid[ret], dtype=float)))
        return ret
    cls.next = recording_next

    expt = os.path.join(tmp, "braninpy")
    os.mkdir(expt)
    shutil.copy(os.path.join(ref_shim.REF_ROOT, "spearmint-lite", "braninpy", "config.json"), expt)
    opts = types.SimpleNamespace(num_jobs=1, max_finished_jobs=1000, chooser_module="GPEIOptChooserB200",
                                 chooser_args=CHOOSER_ARGS, grid_size=300, grid_seed=1, config_file="config.json",
                                 results_file="results.dat")
    res = os.path.join(expt, "results.dat")
    np.random.seed(0)
    for it in range(ITERS):
        lite.main_controller(opts, [expt])                   # appends one "P P x1 x2" line (LITE:199-215)
        lines = open(res).read().splitlines()
        x = [float(t) for t in lines[-1].split()[2:]]
        lines[-1] = "%f 1 %s" % (branin(x), " ".join(lines[-1].split()[2:]))   # braninrunner.py fills the result in
        with open(res, "w") as fh:
            fh.write("\n".join(lines) + "\n")
    cls.next = inner
    assert len(calls) == ITERS
    out = dict(chooser_args=CHOOSER_ARGS, iters=ITERS, seed=0,
               results_dat=open(res).read())                 # the controller's own record of the run
    for i, c in enumerate(calls):
        out.update({"%s_%d" % (k, i): v for k, v in c.items()})
    np.savez_compressed(os.path.join(HERE, "lite_branin.npz"), **out)


if __name__ == "__main__":
    golden_oracle_vs_ref()
    golden_lite_branin()
    for n in ("oracle_vs_ref.npz", "lite_branin.npz"):
        print("wrote", n, os.path.getsize(os.path.join(HERE, n)), "bytes")
