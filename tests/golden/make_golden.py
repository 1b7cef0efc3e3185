"""Generate the committed golden fixtures by EXECUTING the reference.

Needs oracle/_ref/regref, built from a checkout of the reference: the unmodified lib/register.js of that
checkout is evaluated on the SpiderMonkey engine of its tree with a recording fake ZooKeeper client, and
what it passes to zk.create()/zk.put() is stored next to the inputs.

    make -C oracle ref REF=<reference checkout>
    python tests/golden/make_golden.py

Outputs (tests/golden/):
  config1.jsonl   BASELINE.json configs[0]: the 1k synthetic 3-label records; per line
                  {"in": record, "path": ..., "json": ...}
  edge.jsonl      hand-picked edge cases (empty labels, case folding, long labels, escapes, ttl/ports
                  shapes, the reference's README / test-suite inputs); same schema
  calls.jsonl     full call traces of register() for alias / service registrations:
                  {"in": record, "calls": [[op, ...], ...]}
  reference_runs.jsonl
                  the host nodes of synthetic batches (REFERENCE_RUNS) as 64-bit digests, one line per batch:
                  {"config", "start", "n", "inputs": digest of the harness input text,
                   "path": [digest per record], "json": [digest per record]}
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from golden_util import digest, inputs_digest  # noqa: E402
from oracle import refrun  # noqa: E402
from registrar_b200 import synth  # noqa: E402

# (config, start, n) of the synthetic batches tests/test_reference_live.py compares with the reference
REFERENCE_RUNS = [("config1", 5000, 400), ("config3", 123456, 400), ("config5", 77, 400),
                  ("config1", 9000, 600), ("config3", 654321, 600), ("config5", 4242, 600)]


def rec_json(r):
    dec = lambda x: x.decode("latin-1") if isinstance(x, (bytes, bytearray)) else x
    return {k: (dec(v) if not isinstance(v, list) else [dec(x) for x in v]) for k, v in r.items() if v is not None}


def edge_records():
    uu = "a2674d3b-a9c4-46bc-a835-b6ce21d522c2"
    recs = []
    domains = ["", ".", "..", "a", "A", "a.", ".a", "a..b", "...a...b...", "com", "x" * 63,
               ".".join(["l" * 63] * 6), "1.moray.us-east.joyent.com", "authcache.emy-10.joyent.us",
               "test.laptop.joyent.us", "test.coal.joyent.us", "alias-1.test.coal.joyent.us",
               "ABCDEFGHIJKLMNOPQRSTUVWXYZ.[\\]^_`.@az{|}~", "a.b.c.d.e.f.g.h.i.j.k.l.m.n.o.p", "MiXeD.CaSe.ExAmPlE",
               "with space.and\ttab", "UPPER-0123456789.lower_under"]
    hosts = [uu, "h", "host.example.com", "headnode", "..."]
    addrs = ["127.0.0.1", "1.2.3.4", "255.255.255.255", "172.27.10.62", "fe80::1ff:fe23:4567:890a%eth0",
             "abcdefghijklmnop", "abcdefghijklmnopq", 'quo"te', "back\\slash", "ctl\x01\x1f\n\r\t\b\x0c", "\x7f", ""]
    ttls = [None, 0, 5, 30, 60, 120, 3600, 86400, 2147483647, -1, -2147483647, 99999, 100000, 1000000000]
    ports = [None, [], [80], [6379], [1, 22, 333, 4444, 55555], [65535, 0],
             [4294967295, 1000000000, 999999999, 10000, 9999, 100000000, 99999999]]
    types = ["host", "load_balancer", "redis_host", "db_host", "moray_host", "ops_host", "rr_host",
             "custom \"type\"", "t"]
    i = 0
    for d in domains:
        for h in hosts:
            i += 1
            recs.append({"domain": d, "hostname": h, "type": types[i % len(types)], "address": addrs[i % len(addrs)],
                         "ttl": ttls[i % len(ttls)], "ports": ports[i % len(ports)]})
    # the reference's own test-suite and README inputs
    recs.append({"domain": "test.laptop.joyent.us", "hostname": "myhost", "type": "host", "address": "127.0.0.1"})
    recs.append({"domain": "test.laptop.joyent.us", "hostname": "myhost", "type": "host", "address": "127.0.0.1", "ttl": 120})
    recs.append({"domain": "authcache.emy-10.joyent.us", "hostname": uu, "type": "redis_host",
                 "address": "172.27.10.62", "ttl": 30, "ports": [6379]})
    recs.append({"domain": "example.emy-10.joyent.us", "hostname": uu, "type": "load_balancer",
                 "address": "172.27.10.72", "ports": [80]})
    return recs


def call_records():
    svc = lambda **kw: {"type": "service", "service": dict(kw)}
    return [
        {"domain": "test.coal.joyent.us", "hostname": "headnode", "type": "host", "address": "10.99.99.7",
         "aliases": ["alias-1.test.coal.joyent.us"]},
        {"domain": "test.laptop.joyent.us", "hostname": "myhost", "type": "host", "address": "127.0.0.1", "ttl": 120,
         "service": svc(srvce="_http", proto="_tcp", ttl=60, port=80)},
        {"domain": "authcache.emy-10.joyent.us", "hostname": "a2674d3b-a9c4-46bc-a835-b6ce21d522c2",
         "type": "redis_host", "address": "172.27.10.62", "ttl": 30,
         "service": svc(srvce="_redis", proto="_tcp", port=6379)},
        {"domain": "Web.Example.COM", "hostname": "z1", "type": "load_balancer", "address": "10.0.0.9",
         "ports": [80, 443], "aliases": ["a..b", "www.example.com", ""],
         "service": svc(srvce="_http", proto="_tcp", port=8080, ttl=15)},
        {"domain": "nosvc.example.com", "hostname": "z2", "type": "host", "address": "10.0.0.10", "aliases": []},
    ]


def main():
    if not refrun.available():
        raise SystemExit("oracle/_ref/regref is missing: run `make -C oracle ref REF=<reference checkout>`")
    # config1: records as the product sees them (bytes fields decoded as latin-1 == ASCII here)
    b = synth.generate("config1")
    recs = [b.record(i) for i in range(b.n)]
    outs = refrun.host_records(recs)
    with open(os.path.join(HERE, "config1.jsonl"), "w") as f:
        for r, (p, j) in zip(recs, outs):
            f.write(json.dumps({"in": rec_json(r), "path": p.decode("latin-1"), "json": j.decode("utf-8")},
                               separators=(",", ":")) + "\n")
    recs = edge_records()
    outs = refrun.host_records(recs)
    with open(os.path.join(HERE, "edge.jsonl"), "w") as f:
        for r, (p, j) in zip(recs, outs):
            f.write(json.dumps({"in": rec_json(r), "path": p.decode("latin-1"), "json": j.decode("utf-8")},
                               separators=(",", ":")) + "\n")
    recs = call_records()
    traces = refrun.run(recs)
    with open(os.path.join(HERE, "calls.jsonl"), "w") as f:
        for r, calls in zip(recs, traces):
            f.write(json.dumps({"in": rec_json(r), "calls": calls}, separators=(",", ":")) + "\n")
    with open(os.path.join(HERE, "reference_runs.jsonl"), "w") as f:
        for config, start, n in REFERENCE_RUNS:
            b = synth.generate(config, n=n, start=start)
            recs = [b.record(i) for i in range(b.n)]
            outs = refrun.host_records(recs)
            f.write(json.dumps({"config": config, "start": start, "n": n, "inputs": inputs_digest(recs),
                                "path": [digest(p) for p, _ in outs], "json": [digest(j) for _, j in outs]},
                               separators=(",", ":")) + "\n")
    print("golden fixtures written:", [x for x in sorted(os.listdir(HERE)) if x.endswith(".jsonl")])


if __name__ == "__main__":
    main()
