"""The oracle (CPU) and the kernels (GPU) against what the reference itself computed (oracle/_ref/regref: unmodified
lib/register.js on the reference tree's JS engine) for synthetic batches beyond the other fixtures.  The reference's
host nodes are stored as per-record digests in tests/golden/reference_runs.jsonl (tests/golden/make_golden.py)."""
import pytest

from golden_util import digest, inputs_digest, load
from oracle import oracle
from registrar_b200 import synth

RUNS = {(r["config"], r["start"], r["n"]): r for r in load("reference_runs.jsonl")}


def reference_run(config, start, n):
    """(batch, stored reference run) of records [start, start + n) of `config`."""
    batch = synth.generate(config, n=n, start=start)
    run = RUNS[(config, start, n)]
    recs = [batch.record(i) for i in range(batch.n)]
    assert inputs_digest(recs) == run["inputs"], "the synthetic generator no longer makes the inputs of the stored run"
    assert len(run["path"]) == len(run["json"]) == batch.n
    return batch, run


def assert_equals_reference(got, batch, run):
    for i, (p, j) in enumerate(zip(run["path"], run["json"])):
        assert digest(got.path(i)) == p and digest(got.json(i)) == j, (i, batch.record(i), got.path(i), got.json(i))


@pytest.mark.parametrize("config,start", [("config1", 5000), ("config3", 123456), ("config5", 77)])
def test_oracle_vs_live_reference(built, config, start):
    batch, run = reference_run(config, start, 400)
    assert_equals_reference(oracle.register_batch(batch), batch, run)


@pytest.mark.gpu
@pytest.mark.parametrize("config,start", [("config1", 9000), ("config3", 654321), ("config5", 4242)])
def test_kernels_vs_live_reference(built, config, start):
    from registrar_b200 import _native
    batch, run = reference_run(config, start, 600)
    ctx = _native.Context(0)
    got = ctx.register_batch(batch)
    assert_equals_reference(got, batch, run)
    ctx.close()
