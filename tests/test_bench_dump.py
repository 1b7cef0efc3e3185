"""bench.py --dump-outputs: exact values, the same seeded sample on every run, at most 64 MB in all (CPU tensors); on the
GPU, the dump of a real run is the output of its last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_exact_seeded_and_capped(tmp_path, monkeypatch):
    full = 2 * bench.DUMP_CAP["bytes"][0] * 4 + 2 * bench.DUMP_CAP["off"][0] * 8
    assert full <= 64_000_000
    monkeypatch.setitem(bench.DUMP_CAP, "bytes", (1000, np.float32))
    g = torch.Generator().manual_seed(1)
    arrays = {"path_bytes": torch.randint(0, 256, (5000,), dtype=torch.uint8, generator=g),
              "path_off": torch.arange(0, 3001 * 2 ** 40, 2 ** 40, dtype=torch.int64)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "cpu", arrays)
    pb, po = np.load(tmp_path / "a" / "path_bytes.npy"), np.load(tmp_path / "a" / "path_off.npy")
    assert pb.dtype == np.float32 and po.dtype == np.float64
    assert np.array_equal(po, arrays["path_off"].numpy().astype(np.float64))        # under the cap: all of it
    assert po[-1] == 3000 * 2 ** 40
    idx = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(5000, 1000, replace=False))
    assert np.array_equal(pb, arrays["path_bytes"].numpy()[idx])                    # over the cap: the seeded sample
    assert np.array_equal(np.load(tmp_path / "b" / "path_bytes.npy"), pb)


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(built, tmp_path):
    from oracle import oracle
    from registrar_b200 import synth
    n, steps = 20_000, 6                 # small enough that every array is dumped whole
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--records", str(n), "--steps", str(steps),
                          "--warmup", "3", "--only-headline", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["verified"]["ok"]
    # measure_single rotates 4 resident batches of n records for n <= 2 M: the last step ran batch (steps - 1) % 4
    want = oracle.register_batch(synth.generate("config3", n=n, start=(steps - 1) % 4 * n))
    assert want.bad_bits == 0
    for name, dtype, a in (("path_bytes", np.float32, want.path_bytes), ("path_off", np.float64, want.path_off),
                           ("json_bytes", np.float32, want.json_bytes), ("json_off", np.float64, want.json_off)):
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == dtype and np.array_equal(got, a.astype(dtype)), name
