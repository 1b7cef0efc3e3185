#!/usr/bin/env python
"""bench.py — registration hot path throughput on N B200s (driver contract, see DESIGN.md §5).

    python bench.py --gpus 1 --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...             # CPU arm: the oracle's C port on the host cores
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path over one batch of synthetic records (regk_path_kernel: paths + offsets + the
payload lengths as a side job, then regk_json_kernel: payload bytes + offsets).

Workload (`config.workload`, identical in both arms and at every N): BASELINE.json configs[2] — 10 M records of
config 3 (2-6 labels, 75 % with 1-4 SRV ports), the largest single-GPU entry of `configs`.
  N = 1   the whole batch on one GPU.  The same run also measures configs[1] (config 2, 1 M records) and one
          rank's share of configs[4] (config 5, 12.5 M records) and reports them under `configs`.
  N > 1   BASELINE.json configs[3]: the SAME 10 M records sharded over the N GPUs by contiguous record range, the
          job-wide byte streams and offsets reassembled on EVERY rank inside the timed region.  The reassembly
          is fused into the compose kernels (regk_register_batch + REGK_JOB_STEP: every tile is stored into all
          ranks' whole-job buffers over NVLink straight from shared memory; the shard totals travel through a
          peer-memory mailbox; no NCCL call on the data path), so `value` = records of the job / time of
          exchange + path kernel + exchange + payload kernel + closing barrier, max over ranks.  Total work is
          fixed: "scaling": "strong".  `no_collective` keeps the old figure (shards computed, nothing exchanged).

  value  records/s with inputs and outputs resident in HBM: K steps between two CUDA events on the launching
         stream, barrier + synchronize on both sides, max over ranks.  Two distinct resident batches (inputs
         ~1.2 GB each, far larger than the 126 MB L2) are rotated.
  e2e    the same metric through the public call a user makes (Context.submit / collect = the C-ABI
         regk_register_batch with HOST buffers): pinned host inputs -> H2D -> kernels -> D2H of paths, payloads
         and both offset arrays (as 32-bit arrays: option "offsets32"), every step, wall clock between barriers
         (each rank its shard when N > 1).
  roofline   per kernel: algorithmic bytes per launch / mean launch duration (CUDA events recorded by the
         library around each launch inside the timed region), against MEASURED_PEAKS.json hbm_gbs.
  check  outside the timed regions the outputs of the timed configuration are fingerprinted on the GPU
         (position-weighted 64-bit sums of the byte streams and the offset arrays) and compared with the same
         fingerprints of the CPU oracle's output for the same records: `verified` in the JSON line.
  cpu_baseline   the oracle's C port of the reference algorithm timed on this box's host cores (rank 0, N=1).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "service-records/sec"
UNIT = "records/s"
HEADLINE = ("config3", 10_000_000)
EXTRAS = (("config2", 1_000_000), ("config5", 12_500_000))
DESCR = {
    "config2": "3-label domains + instance UUID (BASELINE.json configs[1])",
    "config3": "mixed 2-6 label depth with SRV ports[] in the JSON payload (BASELINE.json configs[2]; sharded over "
               "the GPUs with the output streams all-gathered when n_gpus > 1 = configs[3])",
    "config5": "Zipf-distributed label lengths 1-63 bytes (BASELINE.json configs[4]: 100M records over 8 GPUs; "
               "12500000 = one rank's share)",
}
NVLINK_PEAK_GBS = 770.0     # B200_PROFILING.md: measured peer copy per direction per GPU (900 nominal)


def workload_name(cfg: str, n: int) -> str:
    """The one string both arms put in config.workload."""
    return "%s: %d records, %s" % (cfg, n, DESCR.get(cfg, "synthetic"))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures,
    keyed by (kernel source hash, config, records): profiles/traffic.json, written by tools/ncu_traffic.py from a
    capture of the CURRENT kernels.  No entry for the current sources -> traffic is null."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}
    return table.get(kernel_hash(), {})


def kernel_hash() -> str:
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "registrar_b200", "csrc")
    for f in ("regk_core.cuh", "regk_kernels.cuh"):
        h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


# ------------------------------------------------------------------------------------------ clocks

class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled through NVML while the timed regions run."""

    def __init__(self, index: int, period: float = 0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples = []
        self.active = threading.Event()
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            if self.active.is_set():
                try:
                    mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                        nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.samples.append((mhz, int(reasons)))
                except Exception:  # noqa: BLE001
                    pass
            time.sleep(self.period)

    def summary(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")]}
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                 0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        mhz = sorted(s[0] for s in self.samples)
        bits = 0
        for _, r in self.samples:
            bits |= r
        reasons = [n for b, n in names.items() if bits & b and n != "gpu_idle"]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(mhz)}


def bind_to_gpu_numa(index: int):
    """Run this rank's threads (and, by first touch, its pinned staging buffers) on the CPUs next to its GPU:
    GPUs 4-7 of the 8-GPU box sit on NUMA node 1, and an unbound rank copied across the socket link (VERDICT r1:
    e2e efficiency 0.46 at N=8).  Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": len(cpus), "first": min(cpus), "how": "sched_setaffinity to nvmlDeviceGetCpuAffinity"}
    except Exception as e:  # noqa: BLE001
        return {"cpus": None, "how": "unbound (%r)" % (e,)}
    return {"cpus": None, "how": "unbound"}


# ------------------------------------------------------------------------------- accounting helpers

def kernel_bytes(batch, path_total, json_total):
    """Algorithmic bytes per launch (SURVEY.md §8d split by kernel): every input byte once, every output
    byte once, offsets as stored (u32 in, u64 out)."""
    n = batch.n
    dom = int(batch.domain_off[-1])
    host = n * batch.host_stride if batch.host_off is None else int(batch.host_off[-1])
    addr = int(batch.addr_off[-1])
    k = int(batch.ports_off[-1]) if batch.ports_off is not None else 0
    path_b = (dom + 4 * n + host) + (path_total + 8 * n)
    json_b = (addr + n + n + 4 * n + 4 * n + 4 * k) + (json_total + 8 * n)
    return path_b, json_b


def pinned_copy(ctx, batch):
    """The batch with every array in pinned host memory (what the e2e arm copies from)."""
    import dataclasses
    repl = {}
    for f in ("domain_bytes", "domain_off", "host_bytes", "host_off", "type_id", "addr_bytes", "addr_off", "ttl",
              "ports_off", "ports", "ports_present"):
        a = getattr(batch, f)
        if a is None:
            continue
        p = ctx.pinned_array(a.shape, a.dtype)
        p[...] = a
        repl[f] = p
    return dataclasses.replace(batch, **repl), [v for v in repl.values()]


def free_pinned(ctx, arrays):
    for a in arrays:
        ctx.host_free(a.ctypes.data)


# --------------------------------------------------------------------------------- output fingerprints

MASK64 = (1 << 64) - 1


class Fingerprint:
    """sum over 8-byte little-endian words w_i of a byte stream of w_i * (2i + 1), mod 2^64 (zero padded)."""

    def __init__(self):
        self.acc, self.words, self.left = 0, 0, np.zeros(0, np.uint8)

    def update(self, a: np.ndarray):
        buf = np.concatenate([self.left, a.view(np.uint8).reshape(-1)]) if self.left.size else a.view(np.uint8).reshape(-1)
        nw = buf.size // 8
        if nw:
            w = buf[:8 * nw].view(np.uint64)
            idx = np.arange(self.words, self.words + nw, dtype=np.uint64)
            self.acc = (self.acc + int((w * (idx * np.uint64(2) + np.uint64(1))).sum(dtype=np.uint64))) & MASK64
            self.words += nw
        self.left = buf[8 * nw:].copy()

    def value(self) -> int:
        if self.left.size:
            self.update(np.zeros(8 - self.left.size, np.uint8))
        return self.acc


def fingerprint_gpu(t) -> int:
    """The same fingerprint of a uint8 / int64 CUDA tensor, computed on the GPU in chunks."""
    import torch
    v = t.view(torch.uint8).reshape(-1) if t.dtype != torch.uint8 else t.reshape(-1)
    n = v.numel()
    nw = n // 8
    acc = 0
    step = 1 << 25
    for lo in range(0, nw, step):
        hi = min(nw, lo + step)
        w = v[8 * lo:8 * hi].view(torch.int64)
        idx = torch.arange(lo, hi, device=v.device, dtype=torch.int64)
        acc = (acc + int((w * (2 * idx + 1)).sum().item())) & MASK64
    if n > 8 * nw:
        tail = torch.zeros(8, dtype=torch.uint8, device=v.device)
        tail[:n - 8 * nw] = v[8 * nw:]
        acc = (acc + int(tail.view(torch.int64)[0].item()) * (2 * nw + 1)) & MASK64
    return acc


def oracle_fingerprints(cfg, start, n, chunk=1_000_000):
    """Fingerprints of the CPU oracle's output for records [start, start + n) of `cfg`, chunk by chunk."""
    from oracle import oracle
    from registrar_b200 import synth
    fp = [Fingerprint() for _ in range(4)]          # path bytes, payload bytes, path offsets, payload offsets
    pbase = jbase = 0
    for lo in range(0, n, chunk):
        cn = min(chunk, n - lo)
        hb = synth.generate(cfg, n=cn, start=start + lo)
        r = oracle.register_batch(hb)
        assert r.bad_bits == 0
        fp[0].update(r.path_bytes)
        fp[1].update(r.json_bytes)
        fp[2].update(r.path_off[:cn] + np.uint64(pbase))
        fp[3].update(r.json_off[:cn] + np.uint64(jbase))
        pbase += int(r.path_off[-1])
        jbase += int(r.json_off[-1])
    fp[2].update(np.array([pbase], np.uint64))
    fp[3].update(np.array([jbase], np.uint64))
    return [f.value() for f in fp], pbase, jbase


def verify_against_oracle(cfg, start, n, path_bytes, path_off, json_bytes, json_off):
    """GPU tensors of a finished result (job-wide or single batch) vs the oracle; returns the `verified` object."""
    t0 = time.perf_counter()
    want, ptot, jtot = oracle_fingerprints(cfg, start, n)
    got = [fingerprint_gpu(path_bytes[:ptot]), fingerprint_gpu(json_bytes[:jtot]), fingerprint_gpu(path_off[:n + 1]),
           fingerprint_gpu(json_off[:n + 1])]
    names = ("path_bytes", "payload_bytes", "path_offsets", "payload_offsets")
    bad = [nm for nm, g, w in zip(names, got, want) if g != w]
    return {"ok": not bad, "mismatch": bad, "records": n, "path_bytes": ptot, "payload_bytes": jtot,
            "how": "position-weighted 64-bit sums of both byte streams and both offset arrays, GPU result vs "
                   "oracle/regoracle.c on the same records, outside the timed region",
            "seconds": round(time.perf_counter() - t0, 2)}


# ------------------------------------------------------------------------------------------- dumps

DUMP_SEED = 20251017
DUMP_CAP = {"bytes": (4 << 20, np.float32), "off": (1 << 20, np.float64)}    # elements, dtype: 48 MiB in all


def dump_outputs(out_dir, dev, arrays):
    """Write the outputs of the last timed step as out_dir/<name>.npy, so that two builds run with the same arguments
    can be compared output for output.  `arrays`: name -> device tensor (uint8 byte stream or int64 offsets); byte
    values go out as float32 and offsets as float64, both exactly.  An array longer than its cap is written as a
    fixed, seeded sample of its elements in index order (the same indices for the same length)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        cap, dtype = DUMP_CAP["bytes" if t.dtype == torch.uint8 else "off"]
        if t.numel() > cap:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(t.numel(), cap, replace=False))
            t = t[torch.from_numpy(idx).to(dev)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(dtype))


# ---------------------------------------------------------------------------------------- GPU arm

class Rig:
    """What every measurement of this process shares: device, stream, context, clock sampler, process group."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from registrar_b200 import _native
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit("--gpus %d but WORLD_SIZE=%d: launch with torch.distributed.run --nproc-per-node %d"
                             % (args.gpus, self.world, args.gpus))
        self.numa = bind_to_gpu_numa(self.local)
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.ctx = _native.Context(self.local)
        self.stream = torch.cuda.Stream(device=self.dev)    # one explicit stream: the library's kernels and the timing events
        torch.cuda.set_stream(self.stream)
        self.ctx.set_stream(self.stream.cuda_stream)
        self.sampler = ClockSampler(self.local)
        self.sampler.start()
        self.peak, self.peak_src = load_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


def roof(rig, name, nbytes, ms, launches, time_every, traffic):
    ach = nbytes / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
    return {"kernel": name, "bound": "hbm", "achieved": round(ach, 1), "peak": rig.peak, "unit": "GB/s",
            "frac": round(ach / rig.peak, 4), "traffic": traffic, "algorithmic_bytes": nbytes,
            "mean_launch_ms": round(ms, 5), "launches_timed": launches,
            "timing": "CUDA events around the launch on every %s step of the timed region" % (
                "" if time_every == 1 else "%d-th" % time_every),
            "peak_source": rig.peak_src}


def device_outputs(res, dev):
    """The byte streams and offset arrays of a finished REGK_OUT_DEVICE result as device tensors, by name."""
    import torch
    from registrar_b200 import multigpu
    n = int(res.n)
    return {"path_bytes": multigpu.device_tensor(res.path_bytes, int(res.path_total), torch.uint8, dev),
            "path_off": multigpu.device_tensor(res.path_off, n + 1, torch.int64, dev),
            "json_bytes": multigpu.device_tensor(res.json_bytes, int(res.json_total), torch.uint8, dev),
            "json_off": multigpu.device_tensor(res.json_off, n + 1, torch.int64, dev)}


def device_resident(rig, host_batches):
    from registrar_b200 import multigpu
    pairs = [multigpu.device_batch(hb, rig.dev) for hb in host_batches]
    rig.torch.cuda.synchronize()
    return [p[0] for p in pairs], [p[1] for p in pairs]


def timed_resident_loop(rig, submit, steps, warmup, depth=24):
    """warm-up, then `steps` submissions between two events on the launching stream; returns (ms_total, stats)."""
    torch, ctx = rig.torch, rig.ctx
    inflight = []
    stats = {"path_ms": 0.0, "json_ms": 0.0, "steps": 0, "launches": 0, "last": None, "generic_tiles": 0}

    def drain(limit, count):
        while len(inflight) > limit:
            r = ctx.finish(inflight.pop(0))
            if count:
                if r.kernel_ms > 0:                                # a step that carried the timing events
                    stats["path_ms"] += r.path_kernel_ms
                    stats["json_ms"] += r.json_kernel_ms
                    stats["steps"] += 1
                stats["launches"] += r.launches
                stats["generic_tiles"] = max(stats["generic_tiles"], int(r.generic_tiles))
            stats["last"] = r

    for i in range(warmup):
        inflight.append(submit(i))
        drain(depth, False)
    drain(0, False)
    rig.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rig.sampler.active.set()
    ev0.record(rig.stream)
    for i in range(steps):
        inflight.append(submit(i))
        drain(depth, True)
    ev1.record(rig.stream)
    drain(0, True)
    torch.cuda.synchronize()
    rig.sampler.active.clear()
    rig.barrier()
    return ev0.elapsed_time(ev1), stats


def e2e_loop(rig, pinned, steps, depth=2):
    """Host buffers in, host buffers out, `depth` batches in flight; wall clock between barriers."""
    ctx, torch = rig.ctx, rig.torch
    ctx.set_option("async", 1)
    ctx.set_option("offsets32", 1)           # host results with 32-bit offsets: both streams are far below 4 GiB
    res = None
    for i in range(2):
        res = ctx.collect(ctx.submit(pinned[i % len(pinned)]))
    h2d = pinned[0].h2d_bytes()
    d2h = int(res.path_bytes.nbytes + res.json_bytes.nbytes + res.path_off.nbytes + res.json_off.nbytes)
    rig.barrier()
    torch.cuda.synchronize()
    rig.sampler.active.set()
    t0 = time.perf_counter()
    checksum, tickets = 0, []
    for i in range(steps):
        tickets.append(ctx.submit(pinned[i % len(pinned)]))
        if len(tickets) == depth:
            res = ctx.collect(tickets.pop(0))
            checksum ^= int(res.path_off[-1]) ^ int(res.json_off[-1])    # the host reads the result
    while tickets:
        res = ctx.collect(tickets.pop(0))
        checksum ^= int(res.path_off[-1]) ^ int(res.json_off[-1])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    ctx.set_option("async", 0)
    ctx.set_option("offsets32", 0)
    rig.sampler.active.clear()
    rig.barrier()
    return dt, h2d, d2h


def measure_single(rig, cfg, n, start, steps, warmup, e2e_steps, time_every, verify=True, dump=None):
    """One configuration on this rank's GPU alone: value arm, e2e arm, per-kernel roofline, output check.
    dump: directory for the outputs of the last timed step (dump_outputs)."""
    from registrar_b200 import synth
    torch, ctx = rig.torch, rig.ctx
    NB = 4 if n <= 2_000_000 else 2
    host_batches = [synth.generate(cfg, n=n, start=start + b * n) for b in range(NB)]
    ctx.set_types(host_batches[0].types)
    cbatches, keep = device_resident(rig, host_batches)

    ctx.set_option("async", 1)
    ctx.set_option("time_every", time_every)
    ms_total, stats = timed_resident_loop(rig, lambda i: ctx.register_raw(cbatches[i % NB]), steps, warmup)
    ctx.set_option("async", 0)
    ctx.set_option("time_every", 1)
    last = stats["last"]
    path_total, json_total = int(last.path_total), int(last.json_total)
    if dump:
        dump_outputs(dump, rig.dev, device_outputs(last, rig.dev))      # before the next call overwrites them

    verified = None
    if verify:
        # one more, synchronous run of batch 0: its device result against the oracle
        o = device_outputs(ctx.register_raw(cbatches[0]), rig.dev)
        verified = verify_against_oracle(cfg, start, n, o["path_bytes"], o["path_off"], o["json_bytes"], o["json_off"])

    # ---- end-to-end arm: host buffers through the public call ----
    del cbatches, keep
    torch.cuda.empty_cache()
    pins = [pinned_copy(ctx, hb) for hb in host_batches[:2]]
    e2e_s, h2d, d2h = e2e_loop(rig, [p[0] for p in pins], e2e_steps)
    for p in pins:
        free_pinned(ctx, p[1])

    ms_total, e2e_ms = rig.max_over_ranks([ms_total, e2e_s * 1e3])
    pbytes, jbytes = kernel_bytes(host_batches[0], path_total, json_total)
    p_ms = stats["path_ms"] / max(stats["steps"], 1)
    j_ms = stats["json_ms"] / max(stats["steps"], 1)
    traffic = ncu_traffic().get("%s:%d" % (cfg, n), {})
    roofs = {"path": roof(rig, "regk_path_kernel<false,false>", pbytes, p_ms, stats["steps"], time_every, traffic.get("path")),
             "json": roof(rig, "regk_json_kernel", jbytes, j_ms, stats["steps"], time_every, traffic.get("json"))}
    both = (pbytes + jbytes) / ((p_ms + j_ms) * 1e-3) / 1e9 if p_ms + j_ms > 0 else 0.0
    step_gbs = (pbytes + jbytes) / (ms_total / steps * 1e-3) / 1e9
    return {
        "workload": workload_name(cfg, n), "records": n, "steps": steps,
        "value": n * steps / (ms_total * 1e-3), "unit": UNIT, "ms_per_step": ms_total / steps,
        "roofline": roofs["path" if p_ms >= j_ms else "json"], "roofline_kernels": roofs,
        "roofline_both_kernels": {"achieved": round(both, 1), "frac": round(both / rig.peak, 4), "unit": "GB/s",
                                  "algorithmic_bytes_per_step": pbytes + jbytes},
        "roofline_step": {"achieved": round(step_gbs, 1), "frac": round(step_gbs / rig.peak, 4), "unit": "GB/s",
                          "what": "algorithmic bytes of both kernels / whole step time (launch gaps included)"},
        "e2e": {"value": n * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                "api": "registrar_b200.Context.submit/collect -> regk_register_batch (host buffers, option offsets32)"},
        "gpu_launches": stats["launches"], "verified": verified,
        "generic_tiles": {"per_step": stats["generic_tiles"], "of": 2 * ((n + 127) // 128),
                          "what": "tiles (128 records, both kernels) that outgrew the shared-memory budget and were composed in global memory"},
        "l2": "rotating %d distinct resident batches (%.0f MB of traffic per step, > 126 MB L2)" % (NB, (pbytes + jbytes) / 1e6),
        "_host_batch": host_batches[0],
    }


def json_capacity(hb, max_type_len=13):
    """Upper bound of a shard's payload bytes (the library's own bound, regk_api.cu)."""
    return hb.n * (38 + 2 * max_type_len + 4 + 18 + 11) + 2 * int(hb.addr_off[-1]) + 11 * int(hb.ports_off[-1]) + 16


def measure_job(rig, cfg, n_total, steps, warmup, e2e_steps, verify=True, dump=None):
    """N > 1: the job sharded over the ranks, reassembled on every rank inside the timed region (fused push).
    dump: directory for rank 0's copy of the whole job's outputs of the last timed step (dump_outputs)."""
    from registrar_b200 import multigpu, synth
    torch, ctx, dist = rig.torch, rig.ctx, rig.dist
    lo, hi = multigpu.shard_range(n_total, rig.rank, rig.world)
    n = hi - lo
    NB = 2
    host_batches = [synth.generate(cfg, n=n, start=b * n_total + lo) for b in range(NB)]
    ctx.set_types(host_batches[0].types)
    cbatches, keep = device_resident(rig, host_batches)
    path_cap = max(int(hb.domain_off[-1]) + hb.n * (hb.host_stride + 2) for hb in host_batches) + 64
    json_cap = max(json_capacity(hb) for hb in host_batches) + 64

    # (a) shards only, nothing exchanged: the old weak/"no collective" figure, and the per-kernel HBM rooflines
    ctx.set_option("async", 1)
    ctx.set_option("time_every", 1)
    ms_plain, st_plain = timed_resident_loop(rig, lambda i: ctx.register_raw(cbatches[i % NB]), steps, warmup)
    ctx.set_option("async", 0)

    # (b) the job: every step reassembles the whole streams on every rank
    job = multigpu.PeerJob(ctx, n, path_cap, json_cap, rig.dev)
    ctx.set_option("async", 1)
    ms_job, st_job = timed_resident_loop(rig, lambda i: job.step(cbatches[i % NB]), steps, warmup, depth=8)
    ctx.set_option("async", 0)
    last = st_job["last"]
    recv = job.nbytes_received(last)
    if dump and rig.rank == 0:
        g = job.result(last)
        dump_outputs(dump, rig.dev, {"path_bytes": g.path_bytes, "path_off": g.path_off, "json_bytes": g.json_bytes,
                                     "json_off": g.json_off})
    verified = None
    if verify:
        # every rank checks ITS OWN copy of the gathered streams on its own record range against the CPU oracle (the
        # ranges together cover the job), then the ranks compare fingerprints of their whole copies with each other
        r = job.wait(job.step(cbatches[0]))
        g = job.result(r)
        t0 = time.perf_counter()
        po, jo = g.path_off, g.json_off
        p_lo, p_hi, j_lo, j_hi = int(po[lo]), int(po[hi]), int(jo[lo]), int(jo[hi])
        want, ptot, jtot = oracle_fingerprints(cfg, lo, n)
        got = [fingerprint_gpu(g.path_bytes[p_lo:p_hi].clone()), fingerprint_gpu(g.json_bytes[j_lo:j_hi].clone()),
               fingerprint_gpu(po[lo:hi + 1] - p_lo), fingerprint_gpu(jo[lo:hi + 1] - j_lo)]
        mine_ok = got == want and ptot == p_hi - p_lo and jtot == j_hi - j_lo
        whole = torch.tensor([fingerprint_gpu(g.path_bytes) >> 1, fingerprint_gpu(g.json_bytes) >> 1,
                              fingerprint_gpu(po) >> 1, fingerprint_gpu(jo) >> 1, int(mine_ok)], dtype=torch.int64, device=rig.dev)
        allf = [torch.empty_like(whole) for _ in range(rig.world)]
        dist.all_gather(allf, whole)
        same = all(bool(torch.equal(f[:4], allf[0][:4])) for f in allf)
        ranks_ok = [bool(int(f[4])) for f in allf]
        if rig.rank == 0:
            verified = {"ok": all(ranks_ok) and same, "ranks_ok": ranks_ok, "same_on_every_rank": same, "records": n_total,
                        "path_bytes": int(r.job_path_total), "payload_bytes": int(r.job_json_total),
                        "how": "every rank: position-weighted 64-bit sums of its own copy of the gathered byte streams "
                               "and offset arrays over its record range vs oracle/regoracle.c on the same records (the "
                               "ranges cover the job); then the fingerprints of the whole copies compared across ranks; "
                               "outside the timed region",
                        "seconds": round(time.perf_counter() - t0, 2)}
    job.close()

    # (c) e2e: each rank its shard through host buffers
    del cbatches, keep
    torch.cuda.empty_cache()
    if e2e_steps > 0:
        pins = [pinned_copy(ctx, hb) for hb in host_batches[:2]]
        e2e_s, h2d, d2h = e2e_loop(rig, [p[0] for p in pins], e2e_steps)
        for p in pins:
            free_pinned(ctx, p[1])
    else:
        e2e_s, h2d, d2h = float("nan"), 0, 0

    ms_plain, ms_job, e2e_ms = rig.max_over_ranks([ms_plain, ms_job, e2e_s * 1e3])
    pbytes, jbytes = kernel_bytes(host_batches[0], int(last.path_total), int(last.json_total))
    traffic = ncu_traffic().get("%s:%d" % (cfg, n), {})

    def roofs(st):
        p_ms, j_ms = st["path_ms"] / max(st["steps"], 1), st["json_ms"] / max(st["steps"], 1)
        r = {"path": roof(rig, "regk_path_kernel<false,false>", pbytes, p_ms, st["steps"], 1, traffic.get("path")),
             "json": roof(rig, "regk_json_kernel", jbytes, j_ms, st["steps"], 1, traffic.get("json"))}
        return r, ("path" if p_ms >= j_ms else "json")

    r_plain, dom_plain = roofs(st_plain)
    r_job, dom_job = roofs(st_job)
    step_ms = ms_job / steps
    link = recv / (step_ms * 1e-3) / 1e9
    return {
        "workload": workload_name(cfg, n_total), "records": n_total, "records_per_rank": n, "steps": steps,
        "value": n_total * steps / (ms_job * 1e-3), "unit": UNIT, "ms_per_step": step_ms,
        # contract key `roofline`: with the all-gather fused into both compose kernels the bound that applies is the
        # NVLink ingress of a rank (B200_PROFILING.md: a fused compute+collective kernel is measured against the slower
        # of its compute roofline and bytes-over-NVLink / link bandwidth) - the kernels' launch times ARE the time to
        # push the tile images through the link; their fractions of the HBM roofline are kept in roofline_kernels
        "roofline": {"kernel": "regk_path_kernel + regk_json_kernel, fused compose + push (whole step incl. the exchanges)",
                     "bound": "nvlink", "achieved": round(link, 1), "peak": NVLINK_PEAK_GBS, "unit": "GB/s",
                     "frac": round(link / NVLINK_PEAK_GBS, 4), "traffic": None,
                     "algorithmic_bytes": recv, "mean_launch_ms": round(step_ms, 5), "launches_timed": steps,
                     "what": "bytes the peers store into one rank's whole-job buffers per step / whole step time; peak = "
                             "measured peer copy per direction (B200_PROFILING.md; 900 GB/s nominal)",
                     "peak_source": "B200_PROFILING.md measured peer copy, 770 GB/s per direction"},
        "roofline_kernels": r_job,
        "roofline_nvlink": {"bound": "nvlink", "achieved": round(link, 1), "peak": NVLINK_PEAK_GBS, "unit": "GB/s",
                            "frac": round(link / NVLINK_PEAK_GBS, 4), "recv_bytes_per_rank_per_step": recv,
                            "what": "bytes the peers store into one rank's whole-job buffers per step / whole step time "
                                    "(exchanges, both fused compose+push kernels, closing barrier); peak = measured peer "
                                    "copy per direction (B200_PROFILING.md; 900 GB/s nominal)"},
        "no_collective": {"value": n_total * steps / (ms_plain * 1e-3), "unit": UNIT, "ms_per_step": ms_plain / steps,
                          "roofline_kernels": r_plain, "roofline": r_plain[dom_plain],
                          "what": "the same shards computed with nothing exchanged (round-1 figure)"},
        "e2e": ({"value": n_total * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                 "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": e2e_ms / e2e_steps,
                 "api": "registrar_b200.Context.submit/collect -> regk_register_batch (host buffers), each rank its shard"}
                if e2e_steps > 0 else {"value": None, "unit": UNIT, "skipped": "--e2e-steps 0"}),
        "gpu_launches": st_job["launches"], "verified": verified,
        "l2": "rotating 2 distinct resident shards per rank (%.0f MB of traffic per rank and step, > 126 MB L2)" % ((pbytes + jbytes) / 1e6),
        "_host_batch": host_batches[0],
    }


def run_b200(args):
    rig = Rig(args)
    cfg, n = args.config, args.records
    e2e_steps = 0 if args.e2e_steps <= 0 and rig.world > 1 else max(3, min(args.steps, args.e2e_steps))
    if rig.world == 1:
        m = measure_single(rig, cfg, n, 0, args.steps, args.warmup, e2e_steps, time_every=1 if n > 2_000_000 else 8,
                           verify=not args.no_verify, dump=args.dump_outputs)
        extras = {}
        if not args.only_headline:
            for xcfg, xn in EXTRAS:
                if (xcfg, xn) == (cfg, n):
                    continue
                small = xn <= 2_000_000
                xs = max(args.steps, 20) * (8 if small else 1)              # >= 20 launches behind every per-kernel figure
                x = measure_single(rig, xcfg, xn, 0, xs, args.warmup, e2e_steps, time_every=8 if small else 1,
                                   verify=not args.no_verify)
                x.pop("_host_batch")
                extras["%s_%d" % (xcfg, xn)] = x
        scaling = "strong"
    else:
        m = measure_job(rig, cfg, n, args.steps, args.warmup, e2e_steps, verify=not args.no_verify,
                        dump=args.dump_outputs)
        extras = {}
        scaling = "strong"
    rig.sampler.stop_flag = True
    if rig.rank == 0:
        hb = m.pop("_host_batch")
        line = {
            "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": rig.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": m["workload"], "records": n},
            "detail": {"records_per_rank": m.get("records_per_rank", n), "l2": m["l2"], "numa": rig.numa,
                       "sharding": "one GPU" if rig.world == 1 else
                       "contiguous record ranges; all-gather of both byte streams and both offset arrays fused into the "
                       "compose kernels (tiles pushed to every rank over NVLink), inside `value`"},
        }
        for k in ("roofline", "roofline_kernels", "roofline_both_kernels", "roofline_step", "roofline_nvlink",
                  "no_collective", "e2e", "gpu_launches", "verified", "generic_tiles"):
            if k in m:
                line[k] = m[k]
        if extras:
            line["configs"] = extras
        line["clocks"] = rig.sampler.summary()
        line["impl"] = "b200"
        line["kernel_hash"] = kernel_hash()
        if rig.world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, range(os.cpu_count() or 1))           # the CPU arm may use every core of the box
            line["cpu_baseline"] = cpu_baseline(hb, args.cpu_seconds)
        print(json.dumps(line), flush=True)
    rig.ctx.close()
    if rig.world > 1:
        rig.dist.destroy_process_group()


# ---------------------------------------------------------------------------------------- CPU arm

def cpu_baseline(batch, budget_s: float):
    """The oracle's C port of the reference algorithm on the host cores: all threads, repeated over the
    same batch for about `budget_s` seconds; mean rate reported."""
    from oracle import oracle
    threads, rates = oracle.calibrate_threads(batch)
    oracle.register_batch(batch.slice(0, min(batch.n, 10000)), threads=threads)     # warm the thread pool
    best, spent, reps, t_end = None, 0.0, 0, time.perf_counter() + budget_s
    while reps < 3 or time.perf_counter() < t_end:
        r = oracle.register_batch(batch, threads=threads, timing_only=True)
        best = r.seconds if best is None else min(best, r.seconds)
        spent += r.seconds
        reps += 1
        if reps >= 200:
            break
    one = oracle.register_batch(batch.slice(0, min(batch.n, 200_000)), threads=1)
    return {"value": batch.n * reps / spent, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d back-to-back repetitions of the full %d-record batch, mean rate (best repetition: %.0f "
                      "records/s); C restatement of lib/register.js (oracle/regoracle.c, OpenMP, thread count "
                      "calibrated on this host) - a port, not Node/V8 (no node on the box)" % (reps, batch.n, batch.n / best),
            "single_thread_value": min(batch.n, 200_000) / one.seconds,
            "thread_calibration": {str(k): round(v) for k, v in sorted(rates.items())}}


def reference_js_sample(batch, count=2000, repeat=3):
    """The reference's own lib/register.js on the reference tree's JS engine (1 core), if the binary is here."""
    from oracle import refrun
    if not refrun.available():
        return None
    recs = [batch.record(i) for i in range(min(count, batch.n))]
    t = refrun.time_records(recs, repeat)
    if t["ms"] <= 0:
        return None
    return {"value": t["records"] / (t["ms"] * 1e-3), "unit": UNIT, "cores": 1,
            "what": "unmodified lib/register.js on SpiderMonkey 1.7 (deps/javascriptlint), fake zk, %d records" % t["records"]}


def node_probe():
    """BASELINE.md's preferred CPU baseline is the reference on Node/V8; say whether this box could run it."""
    import shutil
    path = shutil.which("node") or shutil.which("nodejs")
    return {"node": path, "note": "node found but the reference's npm dependencies (assert-plus, once, vasync) are not "
            "vendored: oracle/harness_prelude.js would have to stand in for them" if path else
            "no node binary on this box: the executed reference is oracle/_ref/regref (SpiderMonkey 1.7), the timed "
            "CPU arm is the C port"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from registrar_b200 import synth
    n, cfg = args.records, args.config
    batch = synth.generate(cfg, n=n, start=0)
    from oracle import oracle
    threads, rates = oracle.calibrate_threads(batch)        # same choice of thread count as the b200 arm's cpu_baseline
    for _ in range(max(min(args.warmup, 3), 1)):
        oracle.register_batch(batch, threads=threads, timing_only=True)
    done, total_s = args.steps, 0.0
    for _ in range(done):
        total_s += oracle.register_batch(batch, threads=threads, timing_only=True).seconds
    value = n * done / total_s
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": done, "warmup": args.warmup,
        "ms_per_step": total_s / done * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "impl": "reference",
        "config": {"workload": workload_name(cfg, n), "records": n},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d steps of the full %d-record batch; C restatement of lib/register.js "
                                   "(oracle/regoracle.c, OpenMP, thread count calibrated on this host) - a port, "
                                   "not Node/V8" % (done, n),
                         "thread_calibration": {str(k): round(v) for k, v in sorted(rates.items())}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "node": node_probe(),
    }
    js = reference_js_sample(batch)
    if js:
        line["reference_js"] = js
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=HEADLINE[0])
    ap.add_argument("--records", type=int, default=HEADLINE[1], help="records of the whole job per step")
    ap.add_argument("--e2e-steps", type=int, default=10, help="N > 1: 0 skips the host-buffer arm (very large jobs)")
    ap.add_argument("--cpu-seconds", type=float, default=4.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true", help="skip the oracle fingerprint check (profiling runs)")
    ap.add_argument("--only-headline", action="store_true", help="N=1: skip the extra configurations")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (large ones as a seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
