"""GPU: bench.py --dump-outputs writes what the timed path returned in its last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _support as S

sys.path.insert(0, S.ROOT)
import bench  # noqa: E402

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_timed_step(engine, tmp_path):
    steps, warmup, gates, batch = 3, 1, 40, 8
    res = subprocess.run([sys.executable, os.path.join(S.ROOT, "bench.py"), "--steps", str(steps),
                          "--warmup", str(warmup), "--no-extras", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, check=True, timeout=600)
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert (line["steps"], line["warmup"], line["config"]["gates"]) == (steps, warmup, gates)
    # the states of the last timed step, searched again through the same batch call
    states = bench.build_batch(gates, batch, 1000 + warmup + steps - 1)
    for i, st in enumerate(states):
        engine.stage(i, st["tables"], st["target"], st["mask"], st["inbits"])
    got = engine.search_batch([dict(slot=i, order5=st["order5"], outer=st["outer"],
                                    middle=st["middle"]) for i, st in enumerate(states)])
    want = {"r5": [bench._result_row(r.r5) for r in got], "r7": [bench._result_row(r.r7) for r in got]}
    assert sorted(os.listdir(tmp_path)) == ["node.npy", "r5.npy", "r7.npy"]
    for name, cols in (("r5", bench.RESULT_COLUMNS), ("r7", bench.RESULT_COLUMNS),
                       ("node", bench.NODE_COLUMNS)):
        arr = np.load(tmp_path / (name + ".npy"))
        assert arr.dtype == np.float64 and arr.shape == (batch, len(cols))
        if name in want:
            assert np.array_equal(arr, np.array(want[name], dtype=np.float64)), name
