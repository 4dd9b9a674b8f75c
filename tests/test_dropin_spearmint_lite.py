"""CPU: BASELINE config 1 -- the reference's UNMODIFIED spearmint-lite controller proposing Branin experiments through our
chooser, loaded by name via the 3-line stub of INTEGRATION.md.  tests/golden/lite_branin.npz records every
chooser.next() call that controller made in such a run (tests/golden/make_golden_live.py) and what the chooser returned;
this test imports the chooser the way the controller does ('chooser.' + name), makes a fresh one per proposal as the
controller does, and replays those calls.  Only the numerics behind the chooser are the oracle stand-in here (no GPU
needed) -- the same chooser class is exercised with the real DeviceBackend in tests/test_gpu_chooser.py."""
import importlib
import os
import sys

import numpy as np

from tests.helpers import load
from tests.oracle_backend import OracleBackend

STUB = "from spearmint_b200.chooser.GPEIOptChooserB200 import *  # noqa: F401,F403\n"


def branin(x):
    """spearmint/examples/braninpy/branin.py:6-16 (x in the unit square)."""
    x1, x2 = x[0] * 15 - 5, x[1] * 15
    return float(np.square(x2 - (5.1 / (4 * np.square(np.pi))) * np.square(x1) + (5 / np.pi) * x1 - 6)
                 + 10 * (1 - (1. / (8 * np.pi))) * np.cos(x1) + 10)


def test_spearmint_lite_drives_the_dropin_chooser(tmp_path, monkeypatch):
    g = load("lite_branin")
    # the stub a maintainer drops into spearmint/spearmint/chooser/
    plug = tmp_path / "plugins" / "chooser"
    plug.mkdir(parents=True)
    (plug / "__init__.py").write_text("")
    (plug / "GPEIOptChooserB200.py").write_text(STUB)
    monkeypatch.syspath_prepend(str(tmp_path / "plugins"))
    for name in [m for m in sys.modules if m == "chooser" or m.startswith("chooser.")]:
        monkeypatch.delitem(sys.modules, name)
    module = importlib.import_module("chooser.GPEIOptChooserB200")
    # numerics: oracle stand-in; the product default is DeviceBackend and raises without CUDA
    import spearmint_b200.backend as be
    monkeypatch.setattr(be, "DeviceBackend", lambda **kw: OracleBackend())

    expt = tmp_path / "braninpy"
    expt.mkdir()
    lines = str(g["results_dat"]).splitlines()          # the controller's results.dat after the run (values filled in)
    assert len(lines) == int(g["iters"]) == 8
    np.random.seed(int(g["seed"]))
    best = np.inf
    for i in range(int(g["iters"])):
        c = {k: g["%s_%d" % (k, i)] for k in ("grid", "values", "durations", "candidates", "pending", "complete",
                                              "ret_tuple", "ret_index", "ret_point")}
        # the controller passes a float, not an array, when exactly one result is complete
        durations = float(c["durations"]) if c["durations"].ndim == 0 else c["durations"]
        ch = module.init(str(expt), str(g["chooser_args"]))
        ret = ch.next(c["grid"], c["values"], durations, c["candidates"], c["pending"], c["complete"])
        if bool(c["ret_tuple"]):
            assert isinstance(ret, tuple) and ret[0] == int(c["ret_index"])
            x = np.asarray(ret[1], dtype=float)
            np.testing.assert_allclose(x, c["ret_point"], rtol=0, atol=1e-6)
        else:
            assert int(ret) == int(c["ret_index"])
            x = c["grid"][int(ret)]
        assert x.shape == (2,) and np.all((0.0 <= x) & (x <= 1.0))
        np.testing.assert_allclose(x, [float(t) for t in lines[i].split()[2:]], rtol=0, atol=1e-6)   # what it wrote
        best = min(best, branin(x))
    # GP-EI picked the last 6 (the first two proposals are "candidates[0]" with < 2 completed, OPT:221-222)
    assert os.path.exists(str(expt / "spearmint_b200.chooser.GPEIOptChooserB200.pkl"))
    assert best < 25.0      # Branin over the unit square spans 0.4 .. 300; 8 evaluations already land in the basin
