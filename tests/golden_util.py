"""Load the committed golden fixtures (tests/golden/*.jsonl; produced by tests/golden/make_golden.py from the
reference's own lib/register.js)."""
import hashlib
import json
import os

HERE = os.path.dirname(os.path.abspath(__file__))
HARNESS_INTERFACE_ADDRESS = "10.77.77.7"


def digest(b: bytes) -> str:
    """64-bit digest of one output (reference_runs.jsonl stores these instead of the bytes)."""
    return hashlib.blake2b(b, digest_size=8).hexdigest()


def inputs_digest(records) -> str:
    """Digest of the harness input text of `records`: pins the inputs a stored reference run was made from."""
    from oracle import refrun
    return digest("\n".join(refrun.opts_line(r) for r in records).encode("ascii"))


def load(name):
    rows = []
    with open(os.path.join(HERE, "golden", name)) as f:
        for line in f:
            if line.strip():
                rows.append(json.loads(line))
    return rows


def as_record(d):
    """fixture "in" object -> record dict for RecordBatch.from_records (latin-1 == the raw bytes)."""
    # lib/register.js:143 `opts.adminIp ? opts.adminIp : address()`: an empty adminIp is falsy, so the reference
    # falls back to the first non-internal interface — 10.77.77.7 in the harness (oracle/harness_prelude.js).
    addr = d.get("address", "") or HARNESS_INTERFACE_ADDRESS
    r = {"domain": d["domain"].encode("latin-1"), "hostname": d["hostname"].encode("latin-1"),
         "type": d["type"].encode("utf-8"), "address": addr.encode("latin-1"),
         "ttl": d.get("ttl"), "ports": d.get("ports")}
    return r
