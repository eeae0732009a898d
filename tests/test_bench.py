"""bench.py --dump-outputs: the last timed step's results as .npy files, the same from run to run, so that two
builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True,
                          text=True, cwd=ROOT, timeout=900)


def test_arguments_that_time_nothing_or_dump_nothing_are_refused():
    r = _bench("--steps", "0")
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    r = _bench("--impl", "reference", "--dump-outputs", "unused")
    assert r.returncode == 2 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_steps_sets_the_timed_steps_and_the_dump_is_the_last_one(tmp_path):
    """Step k evaluates the k-th theta after the warm-up ones, so the last timed step of --warmup 1 --steps 3 and the
    only one of --warmup 3 --steps 1 are the same evaluation: the same dumped bits, and the second run's first value."""
    n = 3000
    runs = []
    for warmup, steps in ((1, 3), (3, 1)):
        out = tmp_path / ("w%d_s%d" % (warmup, steps))
        r = _bench("--sites", str(n), "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline", "--no-large",
                   "--dump-outputs", str(out))
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        runs.append((line, {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}))
    (line_a, a), (line_b, b) = runs
    assert sorted(a) == ["logdet", "logdet_w", "neg2loglik", "quad", "rank"]
    for name in a:
        assert a[name].dtype == np.float64 and np.array_equal(a[name], b[name]), name
    assert a["neg2loglik"][0] == line_b["config"]["objective_value_step0"]
    assert a["neg2loglik"][0] != line_a["config"]["objective_value_step0"]
    # the value is the one formed from the dumped terms
    assert a["neg2loglik"][0] == n * np.log(2 * np.pi) + 2 * a["logdet"][0] + a["quad"][0]
