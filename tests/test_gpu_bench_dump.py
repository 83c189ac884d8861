"""bench.py --dump-outputs: the scores of the last timed step of the headline workload, in the base batch's row order
whichever rotating buffer that step read, equal the CPU oracle's on the same seeded rows."""

import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_steps_scores(tmp_path):
    from mlrun_b200.synthetic import flow3_workload
    from oracle import batch as obatch

    B = 4096
    dumps = []
    for per_step in (2, 3):  # the last launch reads a different rotating buffer
        out = tmp_path / f"lps{per_step}"
        done = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", str(B), "--steps", "2", "--warmup", "1",
                               "--launches-per-step", str(per_step), "--no-cpu-baseline", "--no-e2e", "--no-configs",
                               "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert done.returncode == 0, done.stderr[-2000:]
        assert sorted(os.listdir(out)) == ["outputs.npy"]
        dumps.append(np.load(out / "outputs.npy"))
    assert dumps[0].dtype == np.float32 and dumps[0].shape[0] == B
    assert np.array_equal(dumps[0], dumps[1])
    want = obatch.flow3(flow3_workload(n_rows=65536, n_num=56, n_cat=8, seed=2, n_models=4))["out"][:B]
    np.testing.assert_allclose(dumps[0][:, 0], want, rtol=1e-5, atol=1e-5)
