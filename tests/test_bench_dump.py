"""bench.py --dump-outputs: which worlds it writes (host logic) and that the files hold what the timed path computed (GPU)."""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def _bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_sample_is_fixed_and_within_the_budget():
    b = _bench()
    m = 7 * 128 + 7 * 128 * 10 + 28  # the default workload: 10 obstacles
    idx = b.dump_sample(1024, m)
    assert 0 < len(idx) < 1024 and np.array_equal(idx, np.unique(idx)) and idx.max() < 1024
    assert len(idx) * 8 * m * 8 <= b.DUMP_BYTES - 1024
    assert np.array_equal(idx, b.dump_sample(1024, m))
    assert np.array_equal(b.dump_sample(8, m), np.arange(8))


@pytest.mark.gpu
def test_dump_holds_the_last_iterate_of_the_timed_step(built, tmp_path):
    """128 worlds x 10 obstacles exceed the 64 MB budget, so the dump is the sampled subset of worlds."""
    nprob, nobs, iters = 128, 10, 2
    args = ["--nprob", str(nprob), "--nobs", str(nobs), "--iters", str(iters), "--steps", "2", "--warmup", "1",
            "--sweep-worlds", "0", "--no-configs", "--no-cpu-baseline", "--no-e2e", "--no-m1"]
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    g, jac = np.load(tmp_path / "g.npy"), np.load(tmp_path / "jac.npy")
    from armour_b200 import ReachSetEngine, worlds
    q0, qd0, qdd0, _, obs = worlds.random_problems(nprob, nobs, seed=20261017)
    k = worlds.halton_k(iters * nprob).reshape(iters, nprob, 7)[-1]
    eng = ReachSetEngine(max_problems=nprob, max_obstacles=nobs)
    eng.build(q0, qd0, qdd0, obs)
    g_ref, jac_ref = eng.eval(k)
    eng.close()
    idx = _bench().dump_sample(nprob, g_ref.shape[1])
    assert len(idx) < nprob and g.shape[0] == jac.shape[0] == len(idx)
    assert g.dtype == jac.dtype == np.float64
    assert np.array_equal(g, g_ref[idx]) and np.array_equal(jac, jac_ref[idx])
