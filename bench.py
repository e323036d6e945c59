#!/usr/bin/env python3
"""bench.py - MCP tools/call transcodes/sec on B200 (BASELINE.json metric).

One step = one pass of the hot path over one synthetic batch: the request side (arguments JSON ->
protobuf wire) followed by the reply side (protobuf wire -> protojson text) for every item.
Default workload: BASELINE.json configs[2] (nested+repeated messages from the reference's
complex.proto descriptors, ~4 KB JSON, 151 552 items per GPU) - the config the target is quoted on.
The default N=1 run also takes short side runs of the other configs (flat, blob, mixed) and reports
them under `configs`, each with its own roofline entry.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload nested|flat|blob|mixed] [--items M]
  python bench.py --impl reference ...      (the CPU path: oracle port on all host cores, same items)
  python bench.py ... --dump-outputs DIR    (a seeded sample of what the last timed step returned, as .npy files)

Under torchrun (N > 1) every rank owns one GPU and its own shard of the batch (items shard by
index, no collective on the data path); rank 0 prints one JSON line.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOAD_NAMES = {
    "nested": "configs[2] nested+repeated ~4KB JSON (complex.proto ProcessNodeRequest/CreateDocumentRequest; replies Node/GetUserProfileResponse)",
    "flat": "configs[1] 64K flat-scalar bench.Flat ~256B JSON",
    "blob": "configs[3] bench.Blob 64KiB bytes replies (reply side only)",
    "mixed": "configs[4] mixed replay: 32 methods (4 of the reference's protos + 28 generated), method Zipf(1.1), size Zipf(1.2) 64B-64KiB",
}
DEFAULT_ITEMS = {"nested": 148 * 1024, "flat": 148 * 1024, "blob": 4096, "mixed": 128 * 1024}
METRIC = "tools_call_transcodes_per_sec"
UNIT = "transcodes/s"
# profile slot -> kernel function (for the ncu traffic table) and what it reads / writes
KERNEL_FN = {"encode_coop_tok": "k_encode_tok3", "encode_place": "k_encode_place", "encode_type": "k_encode_type",
             "encode_coop_parse": "k_encode_coop_parse", "encode_coop_emit": "k_encode_coop_emit", "encode_parse": "k_encode_parse",
             "encode_emit": "k_encode_emit", "decode_coop_size": "k_decode_coop_size", "decode_coop_write": "k_decode_coop_write",
             "decode_size": "k_decode_size", "decode_write": "k_decode_write"}


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def load_fds():
    with open(os.path.join(ROOT, "tests", "golden", "schemas.binpb"), "rb") as fh:
        return fh.read()


def make_workload(kind, n, msg_index, first):
    import benchgen
    if kind == "nested":
        return benchgen.nested(n, msg_index, first=first)
    if kind == "flat":
        return benchgen.flat(n, msg_index, first=first)
    if kind == "blob":
        return benchgen.blob(n, msg_index, first=first)
    if kind == "mixed":
        return benchgen.mixed(n, msg_index, first=first)
    raise SystemExit("unknown workload " + kind)


def config_dict(kind, n, world, J_in, W_out, W_in, J_out):
    """the same dictionary in the engine arm and in the reference arm (the driver compares them)"""
    return {"workload": WORKLOAD_NAMES[kind], "items_per_gpu": n, "boundary": "InvokeMethod (arguments JSON -> wire, wire -> protojson)",
            "avg_bytes": {"J_in": round(J_in / n, 2), "W_out": round(W_out / n, 2), "W_in": round(W_in / n, 2), "J_out": round(J_out / n, 2)},
            "l2": "inputs exceed L2 (%.0f MB read per step)" % ((J_in + W_in) / 1e6), "parallelism": "shard-by-index x%d, no collective" % world}


def source_sha():
    """hash of the kernel sources: the ncu traffic table is only valid for the build it was captured on"""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "ggrmcp_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh", ".h", ".cc")):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def ncu_traffic(kernel, workload, items):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture of this very build and
    configuration (profiles/ncu_traffic.json, written by scripts/ncu_traffic.py); None when there is none or it is stale"""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None, "no capture"
    sha = source_sha()
    stale = False
    for e in json.load(open(path)):
        if e["kernel"] == kernel and e["workload"] == workload and e["items"] == items:
            if e["source_sha"] == sha:
                return int(e["dram_read"] + e["dram_write"]), "profiles/%s" % e["report"]
            stale = True
    return None, "capture is of another build (stale)" if stale else "no capture of this kernel / configuration"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                parts = [p.strip() for p in out.split(",")]
                self.samples.append(float(parts[0]))
                self.max_mhz = float(parts[1])
                for nm, v in zip(names, parts[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nm)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=10)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---- CPU oracle (port of the reference path): the reference arm, the baseline, the parity checker ----
_ORC = {}


def oracle_schema():
    import orc
    if "S" not in _ORC:
        _ORC["S"] = orc.Schema(load_fds())
    return _ORC["S"]


def oracle_workload(kind, n, first=0):
    key = (kind, n, first)
    if key not in _ORC:
        _ORC[key] = make_workload(kind, n, oracle_schema().msg, first)
    return _ORC[key]


def oracle_pass(wl, threads):
    """one step of the CPU path over wl; returns (seconds, request-side output, reply-side output)"""
    S = oracle_schema()
    t0 = time.perf_counter()
    req = None
    if wl.req_json is not None:
        req = S.encode_batch(wl.req_msg, wl.req_json, wl.req_off, threads=threads)
    rep = S.decode_batch(wl.rep_msg, wl.rep_wire, wl.rep_off, threads=threads, cap=int(len(wl.rep_wire) * 2.5 + 64 * wl.n + 4096))
    return time.perf_counter() - t0, req, rep


def host_cpus():
    """CPUs this process may actually use: the affinity mask, cut by the container's CPU quota (cgroup v2 cpu.max, v1
    cfs quota) - os.cpu_count() of a 128-thread box says 128 inside a container that is throttled to 16"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(quota + 0.999)))
    return n


_cpu_threads = {}


def cpu_threads(kind):
    """thread count of the CPU arm: the fastest of {1, 2, 4} x host_cpus() on a short sample (under a CPU quota more
    threads than quota-CPUs still help until the throttling sets in; beyond that they cost: 128 threads on a 16-CPU
    quota ran at 0.6 of what 32 reach, scripts/cpu_scaling_probe.py)"""
    if kind in _cpu_threads:
        return _cpu_threads[kind]
    cpus, cap = host_cpus(), os.cpu_count() or 1
    cand = sorted({min(cap, cpus * m) for m in (1, 2, 4)})
    wl = oracle_workload(kind, 8192 if kind != "blob" else 256)
    oracle_pass(wl, cand[0])
    best, best_t = cand[0], None
    for th in cand:
        t = min(oracle_pass(wl, th)[0] for _ in range(2))
        if best_t is None or t < best_t * 0.97:
            best, best_t = th, t
    _cpu_threads[kind] = best
    return best


def cpu_baseline(kind, n, min_seconds=8.0):
    """transcodes/s of the port: one thread (bounded sample) and every host thread (the bench's own items)"""
    cores, threads = host_cpus(), cpu_threads(kind)
    wl_all = oracle_workload(kind, n)
    k1 = max(256, min(n, 4096 if kind != "blob" else 128))
    wl_1 = oracle_workload(kind, k1)
    oracle_pass(oracle_workload(kind, min(n, 256)), threads)  # warm the thread pool / page in
    t1, r1 = 0.0, 0
    while t1 < min_seconds / 4 and r1 < 32:
        t1 += oracle_pass(wl_1, 1)[0]
        r1 += 1
    ta, ra = 0.0, 0
    while (ta < min_seconds or ra < 2) and ra < 64:
        ta += oracle_pass(wl_all, threads)[0]
        ra += 1
    v1, va = k1 * r1 / t1, n * ra / ta
    return {"value": va, "unit": UNIT, "cores": cores, "kind": "port", "threads": threads, "value_allcores": va, "value_1thread": v1,
            "scaling_eff": va / (v1 * cores), "logical_cpus": os.cpu_count(),
            "sample": "%d items of the %s workload x %d on %d threads (%.1f s; %d CPUs usable: affinity and cgroup quota); one thread: "
                      "%d items x %d (%.1f s); oracle C++ port - no Go toolchain in the image, so not the Go path itself"
                      % (n, kind, ra, threads, ta, cores, k1, r1, t1)}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores.  The Go reference
    cannot be built in this image (no Go toolchain), so this arm times the oracle port, all host threads, on the
    very items the engine arm takes (same generator, same seed, same count)."""
    if rank != 0:
        return
    cores, threads = host_cpus(), cpu_threads(args.workload)
    n = args.items
    wl = oracle_workload(args.workload, n)
    for _ in range(max(1, min(args.warmup, 2))):
        oracle_pass(oracle_workload(args.workload, min(n, 2048)), threads)
    t0 = time.perf_counter()
    t_sum, last = 0.0, None
    for _ in range(args.steps):
        t, req, rep = oracle_pass(wl, threads)
        t_sum += t
        last = (req, rep)
    req, rep = last
    if args.dump_outputs:
        sides = {} if req is None else {"request": (req[1], req[2], req[0].__getitem__)}
        sides["reply"] = (rep[1], rep[2], rep[0].__getitem__)
        dump_outputs(args.dump_outputs, sides)
    J_in = int(len(wl.req_json)) if wl.req_json is not None else 0
    W_out = int(req[1][n]) if req is not None else 0
    value = n * args.steps / t_sum
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * t_sum / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": config_dict(args.workload, n, max(world, args.gpus), J_in, W_out, int(len(wl.rep_wire)), int(rep[1][n])),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "threads": threads, "logical_cpus": os.cpu_count(),
                         "sample": "%d items of the %s workload per step (the engine arm's items), oracle C++ port, %d threads on %d usable CPUs"
                                   % (n, args.workload, threads, cores)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


DUMP_SEED = 0xD0B5
DUMP_ITEMS = 4096
DUMP_BYTES = 7 << 20  # output bytes per direction: two directions of float32 bytes stay under 64 MB


def dump_outputs(directory, sides):
    """--dump-outputs: for each direction {name: (output offsets[n + 1], status[n], gather)}, the items of a fixed seeded
    permutation of the batch (at most DUMP_ITEMS, while their output bytes fit DUMP_BYTES), written as
    <name>_items (index in the batch), <name>_status, <name>_lengths and <name>_bytes (their outputs, concatenated).
    gather(idx) returns the output bytes at the byte positions idx.  Two builds fed the same arguments dump the same
    items unless their output lengths differ."""
    os.makedirs(directory, exist_ok=True)
    for name, (out_off, status, gather) in sides.items():
        off = np.asarray(out_off).astype(np.int64)
        lens = np.diff(off)
        order = np.random.default_rng(DUMP_SEED).permutation(len(lens))[:DUMP_ITEMS]
        items = np.sort(order[np.cumsum(lens[order]) <= DUMP_BYTES])
        ln = lens[items]
        idx = np.repeat(off[items] - np.cumsum(ln) + ln, ln) + np.arange(int(ln.sum()), dtype=np.int64)
        data = np.asarray(gather(idx), np.uint8)
        arrays = {"items": items.astype(np.float64), "status": np.asarray(status)[items].astype(np.float32),
                  "lengths": ln.astype(np.float64), "bytes": data.astype(np.float32)}
        for k, a in arrays.items():
            np.save(os.path.join(directory, "%s_%s.npy" % (name, k)), a)


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).view(np.uint8).reshape(-1).data)
    return h.hexdigest()


class Resident:
    """one workload resident in HBM: buffers, the step, timing, per-kernel table"""

    def __init__(self, torch, eng, schema, kind, n, rank, dev):
        self.torch, self.eng, self.schema, self.kind, self.n, self.dev = torch, eng, schema, kind, n, dev
        self.wl = wl = make_workload(kind, n, schema.message, rank * n)
        self.have_req = wl.req_json is not None

        def to_dev(a, pad=0):
            t = torch.empty(a.nbytes + pad, dtype=torch.uint8, device=dev)
            t[: a.nbytes] = torch.from_numpy(a.view(np.uint8).reshape(-1))
            if pad:
                t[a.nbytes:] = 0
            return t

        self.to_dev = to_dev
        self.J_in = int(len(wl.req_json)) if self.have_req else 0
        self.W_in = int(len(wl.rep_wire))
        self.d_rep, self.d_rep_off, self.d_rep_msg = to_dev(wl.rep_wire, 64), to_dev(wl.rep_off), to_dev(wl.rep_msg)
        self.rep_cap = int(self.W_in * 2.5 + 64 * n + 4096)
        self.d_rep_out = torch.empty(self.rep_cap, dtype=torch.uint8, device=dev)
        self.d_rep_out_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
        self.d_rep_st = torch.empty(n, dtype=torch.int32, device=dev)
        if self.have_req:
            self.d_req, self.d_req_off, self.d_req_msg = to_dev(wl.req_json, 64), to_dev(wl.req_off), to_dev(wl.req_msg)
            self.req_cap = int(self.J_in + 64)
            self.d_req_out = torch.empty(self.req_cap, dtype=torch.uint8, device=dev)
            self.d_req_out_off = torch.empty(n + 1, dtype=torch.int64, device=dev)
            self.d_req_st = torch.empty(n, dtype=torch.int32, device=dev)
        # a dedicated (non-NULL) stream: the engine enqueues its kernels on it and the CUDA events that bracket the
        # timed region are recorded on the same stream.  Request side and reply side of a step are independent
        # (different calls in flight), so they are enqueued on two streams and share the GPU.
        self.stream = torch.cuda.Stream(device=dev)
        self.stream2 = torch.cuda.Stream(device=dev)
        self.sp, self.sp2 = self.stream.cuda_stream, self.stream2.cuda_stream
        assert self.sp != 0 and self.sp2 != 0

    def step(self, one_stream=False):
        e, s, n = self.eng, self.schema, self.n
        if self.have_req:
            e.encode_batch_dev(s, n, self.d_req_msg.data_ptr(), self.d_req.data_ptr(), self.d_req_off.data_ptr(), self.J_in,
                               self.d_req_out.data_ptr(), self.req_cap, self.d_req_out_off.data_ptr(), self.d_req_st.data_ptr(), 0, self.sp)
        e.decode_batch_dev(s, n, self.d_rep_msg.data_ptr(), self.d_rep.data_ptr(), self.d_rep_off.data_ptr(), self.W_in,
                           self.d_rep_out.data_ptr(), self.rep_cap, self.d_rep_out_off.data_ptr(), self.d_rep_st.data_ptr(), 0,
                           self.sp if one_stream else self.sp2)

    def warm(self, steps):
        torch = self.torch
        for _ in range(max(steps, 3)):
            self.step()
        torch.cuda.synchronize()
        if self.have_req:
            assert int((self.d_req_st != 0).sum()) == 0, "request-side items failed"
        assert int((self.d_rep_st != 0).sum()) == 0, "reply-side items failed"
        self.W_out = int(self.d_req_out_off[self.n].item()) if self.have_req else 0
        self.J_out = int(self.d_rep_out_off[self.n].item())

    def timed(self, steps, barrier, one_stream=False):
        """K steps bracketed by CUDA events on the launching stream; returns milliseconds"""
        torch = self.torch
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        self.stream2.wait_event(e0)      # the reply-side stream starts inside the timed region
        for _ in range(steps):
            self.step(one_stream)
        e_join = torch.cuda.Event()
        e_join.record(self.stream2)
        self.stream.wait_event(e_join)   # ... and must be finished before the closing event
        e1.record(self.stream)
        barrier()
        return e0.elapsed_time(e1)

    def outputs(self):
        """what the last step returned, per direction, in the form dump_outputs takes"""
        torch, dev = self.torch, self.dev

        def side(out, off, st):
            return (off.cpu().numpy(), st.cpu().numpy(), lambda idx: out[torch.from_numpy(idx).to(dev)].cpu().numpy())

        sides = {"request": side(self.d_req_out, self.d_req_out_off, self.d_req_st)} if self.have_req else {}
        sides["reply"] = side(self.d_rep_out, self.d_rep_out_off, self.d_rep_st)
        return sides

    def kernel_table(self):
        """per-kernel device time: the same kernels, same inputs, serialized on one stream so that each launch has the
        GPU to itself (CUDA events around every launch), with the bytes of the items each kernel actually takes"""
        eng, torch, wl = self.eng, self.torch, self.wl
        eng.profile_enable(True)
        eng.profile_read()
        for _ in range(3):
            self.step(one_stream=True)
        torch.cuda.synchronize()
        prof = eng.profile_read()
        eng.profile_enable(False)
        # the router's rule (k_route): lock-step kernels take items of at least 1 KB of JSON / 640 B of wire (and, on the
        # request side, below the parser's input limit); the per-thread kernels take the rest plus what the lock-step
        # tiers leave (counted with the lock-step kernels here: the device-side list lengths are not read back)
        min_json = env_int("GGR_LOCKSTEP_MIN_BYTES", 1024)
        min_wire = env_int("GGR_LOCKSTEP_MIN_BYTES", 640)
        wlen = np.diff(wl.rep_off.astype(np.int64))
        w_big = int(wlen[wlen >= min_wire].sum())
        w_small = self.W_in - w_big
        jo = np.diff(self.d_rep_out_off.cpu().numpy().astype(np.int64))
        jo_big = int(jo[wlen >= min_wire].sum())
        jo_small = self.J_out - jo_big
        if self.have_req:
            jlen = np.diff(wl.req_off.astype(np.int64))
            big = (jlen >= min_json) & (jlen <= 65000 - 16)
            j_big = int(jlen[big].sum())
            j_small = self.J_in - j_big
            wo = np.diff(self.d_req_out_off.cpu().numpy().astype(np.int64))
            wo_big = int(wo[big].sum())
            wo_small = self.W_out - wo_big
        else:
            j_big = j_small = wo_big = wo_small = 0
        alg = {"encode_parse": j_small, "encode_emit": wo_small, "decode_size": w_small, "decode_write": w_small + jo_small,
               "encode_scan": 0, "decode_scan": 0, "decode_coop_size": w_big, "decode_coop_write": w_big + jo_big,
               "encode_coop_parse": j_big, "encode_block_sums": 4 * self.n, "encode_coop_emit": j_big + wo_big, "encode_coop_tok": j_big,
               "encode_place": j_big, "encode_type": j_big}
        kern = {}
        for k, (tot_ms, cnt) in prof.items():
            if cnt and k in alg:
                avg = tot_ms / cnt
                b = alg[k]
                kern[k] = {"avg_ms": avg, "launches": cnt, "algorithmic_bytes": b,
                           "gbs": (b / (avg / 1000.0) / 1e9) if (avg > 0 and b > 0) else None}
        return kern

    def parity(self, threads):
        """the whole batch against the CPU oracle, outside every timed region: digests of bytes, offsets and statuses"""
        S = oracle_schema()
        names = {}
        for full in ("com.example.complex.ProcessNodeRequest", "com.example.complex.CreateDocumentRequest", "com.example.complex.Node",
                     "com.example.complex.GetUserProfileResponse", "bench.Flat", "bench.Blob"):
            try:
                names[self.schema.message(full)] = S.msg(full)
            except KeyError:
                pass
        wl = self.wl
        if self.kind == "mixed":
            import benchgen
            _, pairs = benchgen._mixed_plan(load_fds())
            oreq = np.array([S.msg(a) for a, _ in pairs], np.int32)[wl.method]
            orep = np.array([S.msg(b) for _, b in pairs], np.int32)[wl.method]
        else:
            oreq = np.array([names[int(m)] for m in wl.req_msg], np.int32) if self.have_req else None
            orep = np.array([names[int(m)] for m in wl.rep_msg], np.int32)
        out = {"items": self.n, "directions": 0}
        ok = True
        if self.have_req:
            ow, owoff, ost = S.encode_batch(oreq, wl.req_json, wl.req_off, threads=threads)
            mine = digest(self.d_req_out[: self.W_out].cpu().numpy(), self.d_req_out_off.cpu().numpy().astype(np.uint64), self.d_req_st.cpu().numpy())
            ref = digest(ow, owoff, ost)
            ok &= mine == ref
            out["request_sha256"] = mine
            out["directions"] += 1
        oj, ojoff, ost = S.decode_batch(orep, wl.rep_wire, wl.rep_off, threads=threads, cap=self.rep_cap)
        mine = digest(self.d_rep_out[: self.J_out].cpu().numpy(), self.d_rep_out_off.cpu().numpy().astype(np.uint64), self.d_rep_st.cpu().numpy())
        ref = digest(oj, ojoff, ost)
        ok &= mine == ref
        out["reply_sha256"] = mine
        out["directions"] += 1
        out["equal"] = bool(ok)
        return out


def pcie_probe(torch, eng, dev, mb=256):
    """H2D and D2H of a NUMA-local pinned buffer, both directions at once: GB/s each way"""
    n = mb << 20
    h_in, h_out = torch.from_numpy(eng.host_array(n)), torch.from_numpy(eng.host_array(n))
    d_a = torch.empty(n, dtype=torch.uint8, device=dev)
    d_b = torch.empty(n, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    for _ in range(2):
        with torch.cuda.stream(s1):
            d_a.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_b, non_blocking=True)
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 4
    for _ in range(reps):
        with torch.cuda.stream(s1):
            d_a.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_b, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return reps * n / dt / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="nested", choices=["nested", "flat", "blob", "mixed"])
    ap.add_argument("--items", type=int, default=0, help="items per GPU per step (default: config size)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer measurement (default: min(steps, 5))")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-configs", action="store_true", help="skip the short runs of the other configs")
    ap.add_argument("--no-parity", action="store_true", help="skip the whole-batch comparison with the CPU oracle")
    ap.add_argument("--e2e-serial", action="store_true", help="end-to-end: request call, then reply call (default: both in flight)")
    ap.add_argument("--one-stream", action="store_true", help="serialize request and reply side on one stream")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of what the last step "
                                                          "returned to DIR/<name>.npy (float32 / float64, under 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.items == 0:
        args.items = DEFAULT_ITEMS[args.workload]
    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import ggrmcp_b200
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    eng = ggrmcp_b200.Engine(local)
    # this rank's host side lives on its GPU's NUMA node: the thread that issues the copies and the pinned buffers
    eng.bind_thread()
    schema = eng.register(load_fds())
    n = args.items
    dev = torch.device("cuda", local)
    R = Resident(torch, eng, schema, args.workload, n, rank, dev)
    wl, have_req = R.wl, R.have_req
    J_in, W_in = R.J_in, R.W_in

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_ranks(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if dist is None:
            return [float(x)]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    # ---- warm-up (also sizes the engine's scratch), then the timed region: K steps, CUDA events, max over ranks ----
    R.warm(args.warmup)
    W_out, J_out = R.W_out, R.J_out
    launches0 = eng.launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    ms = R.timed(args.steps, barrier, args.one_stream)
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, R.outputs())
    ms_max = max_ranks(ms)
    value = world * n * args.steps / (ms_max / 1000.0)
    kern = R.kernel_table()

    # ---- whole-batch parity against the CPU oracle (outside the timed region) ----
    parity = None
    if not args.no_parity and rank == 0 and world == 1:
        parity = R.parity(cpu_threads(args.workload))
        assert parity["equal"], "engine output differs from the CPU oracle on the bench batch"

    # ---- the same step at the HTTP-body boundary (SURVEY rows A1-A10): request bodies in, result bodies out ----
    bodies_value = None
    if have_req and args.workload == "nested":
        L0 = ggrmcp_b200.engine._load()
        tool_of = {}
        for mi in reversed(schema.methods()):
            tool_of[mi["input_msg"]] = mi["tool_name"].encode()
        jblob = wl.req_json.tobytes()
        parts = []
        for i in range(n):
            parts.append(b'{"jsonrpc":"2.0","id":%d,"method":"tools/call","params":{"name":"%s","arguments":' % (i, tool_of[int(wl.req_msg[i])]))
            parts.append(jblob[int(wl.req_off[i]):int(wl.req_off[i + 1])])
            parts.append(b"}}")
        lens = np.fromiter((len(parts[3 * i]) + len(parts[3 * i + 1]) + 2 for i in range(n)), np.uint64, n)
        b_off = np.zeros(n + 1, np.uint64)
        b_off[1:] = np.cumsum(lens)
        b_all = np.frombuffer(b"".join(parts), np.uint8).copy()
        del parts
        id_txt = [b"%d" % i for i in range(n)]
        i_off = np.zeros(n + 1, np.uint64)
        i_off[1:] = np.cumsum([len(t) for t in id_txt])
        id_all = np.frombuffer(b"".join(id_txt), np.uint8).copy()
        d_b, d_b_off = R.to_dev(b_all, 64), R.to_dev(b_off)
        d_ids, d_ids_off = R.to_dev(id_all, 64), R.to_dev(i_off)
        d_method = torch.empty(n, dtype=torch.int32, device=dev)
        d_span = torch.empty(2 * n, dtype=torch.int32, device=dev)
        body_cap = int(R.rep_cap * 1.5 + 128 * n)
        d_body_out = torch.empty(body_cap, dtype=torch.uint8, device=dev)
        d_body_off = torch.empty(n + 1, dtype=torch.int64, device=dev)

        def step_bodies_resident():
            rc = L0.ggr_request_batch_dev(eng.h, schema.h, n, d_b.data_ptr(), d_b_off.data_ptr(), len(b_all), R.d_req_out.data_ptr(), R.req_cap,
                                          R.d_req_out_off.data_ptr(), d_method.data_ptr(), d_span.data_ptr(), R.d_req_st.data_ptr(), R.sp)
            assert rc == 0, rc
            rc = L0.ggr_decode_wrap_batch_dev(eng.h, schema.h, n, R.d_rep_msg.data_ptr(), R.d_rep.data_ptr(), R.d_rep_off.data_ptr(), W_in,
                                              d_ids.data_ptr(), d_ids_off.data_ptr(), d_body_out.data_ptr(), body_cap,
                                              d_body_off.data_ptr(), R.d_rep_st.data_ptr(), 0, R.sp2)
            assert rc == 0, rc

        for _ in range(3):
            step_bodies_resident()
        torch.cuda.synchronize()
        assert int((R.d_req_st != 0).sum()) == 0, "request bodies not taken by the device"
        assert int(R.d_req_out_off[n].item()) == W_out and int((R.d_rep_st != 0).sum()) == 0
        body_bytes = int(d_body_off[n].item())
        if parity is not None:
            # request bodies and result bodies of the whole batch against orc_request / orc_response
            S = oracle_schema()
            cores = cpu_threads(args.workload)
            owire, owoff, omethod, oids, oioff, ost = S.request_batch(b_all, b_off, threads=cores)
            assert int((ost != 0).sum()) == 0
            same_req = digest(owire, owoff) == digest(R.d_req_out[:W_out].cpu().numpy(), R.d_req_out_off.cpu().numpy().astype(np.uint64))
            eng_tools = [m["tool_name"] for m in schema.methods()]
            orc_tools = [m["tool"] for m in S.methods()]
            dm = d_method.cpu().numpy()
            same_method = all(eng_tools[int(a)] == orc_tools[int(b)] for a, b in zip(dm[::97], omethod[::97]))
            omsg = {int(schema.message(nm)): S.msg(nm) for nm in ("com.example.complex.Node", "com.example.complex.GetUserProfileResponse")}
            rmsg = np.array([omsg[int(v)] for v in wl.rep_msg], np.int32)
            ob, oboff, ost2 = S.response_batch(rmsg, wl.rep_wire, wl.rep_off, id_all, i_off, threads=cores, cap=body_cap)
            same_body = digest(ob, oboff) == digest(d_body_out[:body_bytes].cpu().numpy(), d_body_off.cpu().numpy().astype(np.uint64))
            parity["http_bodies_equal"] = bool(same_req and same_method and same_body)
            parity["directions"] += 2
            assert parity["http_bodies_equal"], "HTTP-body boundary differs from the CPU oracle"
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record(R.stream)
        R.stream2.wait_event(b0)
        for _ in range(args.steps):
            step_bodies_resident()
        bj = torch.cuda.Event()
        bj.record(R.stream2)
        R.stream.wait_event(bj)
        b1.record(R.stream)
        barrier()
        t_b = max_ranks(b0.elapsed_time(b1))
        bodies_value = {"value": world * n * args.steps / (t_b / 1000.0), "unit": UNIT,
                        "boundary": "HTTP bodies: JSON-RPC request body -> method + wire, wire -> complete result body (rows A1-A10)",
                        "request_body_bytes": int(len(b_all)), "result_body_bytes": body_bytes}
        del d_b, d_body_out

    # ---- end-to-end: host buffers through the public C-ABI call, copies included.  The buffers are the engine's
    # NUMA-local page-locked memory (ggr_host_alloc), the issuing threads are bound to the GPU's node ----
    e2e_steps = args.e2e_steps or min(args.steps, 5)
    L = ggrmcp_b200.engine._load()
    h_rep, h_rep_off, h_rep_msg = eng.host_copy(wl.rep_wire), eng.host_copy(wl.rep_off), eng.host_copy(wl.rep_msg)
    h_rep_out = eng.host_array(R.rep_cap)
    h_rep_out_off = eng.host_array((n + 1) * 8)
    h_rep_st = eng.host_array(n * 4)
    if have_req:
        h_req, h_req_off, h_req_msg = eng.host_copy(wl.req_json), eng.host_copy(wl.req_off), eng.host_copy(wl.req_msg)
        h_req_out = eng.host_array(R.req_cap)
        h_req_out_off = eng.host_array((n + 1) * 8)
        h_req_st = eng.host_array(n * 4)

    def ptr(a):
        return a.ctypes.data

    def host_request():
        rc = L.ggr_encode_batch(eng.h, schema.h, n, ptr(h_req_msg), ptr(h_req), ptr(h_req_off), ptr(h_req_out),
                                R.req_cap, ptr(h_req_out_off), ptr(h_req_st), 0)
        assert rc == 0, rc

    def host_reply():
        rc = L.ggr_decode_batch(eng.h, schema.h, n, ptr(h_rep_msg), ptr(h_rep), ptr(h_rep_off), ptr(h_rep_out),
                                R.rep_cap, ptr(h_rep_out_off), ptr(h_rep_st), 0)
        assert rc == 0, rc

    def on_node(fn):
        def run():
            eng.bind_thread()
            fn()
        return run

    def step_host():
        # a server has request batches and reply batches in flight at the same time: the two calls
        # are issued from two host threads (the C ABI takes one batch per direction concurrently)
        if have_req and not args.e2e_serial:
            t = threading.Thread(target=on_node(host_request))
            t.start()
            host_reply()
            t.join()
            return
        if have_req:
            host_request()
        host_reply()

    step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_host()
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    e2e_per_rank = [n * e2e_steps / t for t in all_ranks(t_e2e)]
    e2e_value = world * n * e2e_steps / max_ranks(t_e2e)
    # the host path's result is the resident path's result (whole batch)
    assert digest(h_rep_out[:J_out]) == digest(R.d_rep_out[:J_out].cpu().numpy()), "host path differs from the resident path"
    if have_req:
        assert digest(h_req_out[:W_out]) == digest(R.d_req_out[:W_out].cpu().numpy())
    probe = all_ranks(pcie_probe(torch, eng, dev))

    # the same, with the reply side producing complete MCP result bodies (SURVEY row A10) instead of the
    # bare protojson texts: reported next to e2e, not instead of it
    e2e_bodies = None
    if have_req and not args.e2e_serial and args.workload == "nested":
        ids = np.frombuffer(b"".join(b"%d" % (i % 100000) for i in range(n)), np.uint8).copy()
        ids_off = np.zeros(n + 1, np.uint64)
        ids_off[1:] = np.cumsum([len(b"%d" % (i % 100000)) for i in range(n)])
        h_ids, h_ids_off = eng.host_copy(ids), eng.host_copy(ids_off)
        body_cap = int(R.rep_cap * 1.5 + 128 * n)
        h_body = eng.host_array(body_cap)

        def host_reply_bodies():
            rc = L.ggr_decode_wrap_batch(eng.h, schema.h, n, ptr(h_rep_msg), ptr(h_rep), ptr(h_rep_off),
                                         ptr(h_ids), ptr(h_ids_off), ptr(h_body), body_cap, ptr(h_rep_out_off), ptr(h_rep_st), 0)
            assert rc == 0, rc

        def step_bodies():
            t = threading.Thread(target=on_node(host_request))
            t.start()
            host_reply_bodies()
            t.join()

        step_bodies()
        assert int((h_rep_st.view(np.int32) != 0).sum()) == 0
        assert bytes(h_body[:61]) == b'{"jsonrpc":"2.0","result":{"content":[{"type":"text","text":"'
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step_bodies()
        torch.cuda.synchronize()
        e2e_bodies = world * n * e2e_steps / max_ranks(time.perf_counter() - t0)
    h2d = J_in + W_in + (n + 1) * 8 * (2 if have_req else 1) + n * 4 * (2 if have_req else 1)
    d2h = W_out + J_out + ((n + 1) * 8 + n * 4) * (2 if have_req else 1)

    # ---- short side runs of the other configs (N = 1, default workload only) ----
    side = None
    if world == 1 and args.workload == "nested" and not args.no_side_configs:
        side = {}
        del R.d_rep_out, h_rep_out
        for kind in ("flat", "blob", "mixed"):
            try:
                r2 = Resident(torch, eng, schema, kind, DEFAULT_ITEMS[kind] if kind != "mixed" else 64 * 1024, 0, dev)
                r2.warm(3)
                steps2 = 5 if kind == "mixed" else 20
                ms2 = r2.timed(steps2, barrier)
                k2 = r2.kernel_table()
                par = None if args.no_parity else r2.parity(cpu_threads('nested'))
                step2 = ms2 / steps2
                dom2 = max(k2, key=lambda k: k2[k]["avg_ms"]) if k2 else None
                side[kind] = {"workload": WORKLOAD_NAMES[kind], "items": r2.n, "value": r2.n * steps2 / (ms2 / 1000.0), "unit": UNIT, "ms_per_step": step2, "steps": steps2,
                              "kernels_ms": {k: round(v["avg_ms"], 4) for k, v in k2.items()} if k2 else None,
                              "avg_bytes": {"J_in": r2.J_in / r2.n, "W_out": r2.W_out / r2.n, "W_in": r2.W_in / r2.n, "J_out": r2.J_out / r2.n},
                              "roofline": roofline_of(k2, dom2, kind, r2.n, step2, r2.J_in, r2.W_in, r2.W_out, r2.J_out, False),
                              "parity_checked_items": (par["items"] * par["directions"]) if par else 0,
                              "parity_equal": par["equal"] if par else None}
                del r2
                torch.cuda.empty_cache()
            except Exception as ex:  # a side run must not cost the headline line
                side[kind] = {"error": repr(ex)[:300]}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    step_ms = ms_max / args.steps
    dom = max(kern, key=lambda k: kern[k]["avg_ms"]) if kern else None
    roofline = roofline_of(kern, dom, args.workload, n, step_ms, J_in, W_in, W_out, J_out, True)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.workload, n)
        if bodies_value is not None:
            # the CPU port at the HTTP-body boundary (orc_request + orc_response: envelope decode, validation,
            # canonicalisation, transcoding, result wrapping) on a bounded sample
            S = oracle_schema()
            cores = cpu_threads(args.workload)
            k = min(n, 32768)
            sb_off = b_off[: k + 1].copy()
            sb = b_all[: int(sb_off[k])]
            omsg = {int(schema.message(nm)): S.msg(nm) for nm in ("com.example.complex.Node", "com.example.complex.GetUserProfileResponse")}
            rmsg = np.array([omsg[int(v)] for v in wl.rep_msg[:k]], np.int32)
            roff = wl.rep_off[: k + 1].copy()
            t0 = time.perf_counter()
            reps = 0
            while reps < 1 or time.perf_counter() - t0 < 4.0:
                _, _, _, oids, oioff, ost = S.request_batch(sb, sb_off, threads=cores)
                S.response_batch(rmsg, wl.rep_wire[: int(roff[k])], roff, oids, oioff, threads=cores)
                reps += 1
            bodies_value["cpu_value"] = k * reps / (time.perf_counter() - t0)
            bodies_value["cpu_sample"] = "%d bodies x %d, oracle C++ port on %d threads" % (k, reps, cores)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": config_dict(args.workload, n, world, J_in, W_out, W_in, J_out),
        "http_bodies": bodies_value,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                "timing": "wall clock around the C-ABI host-buffer calls (NUMA-local page-locked buffers from ggr_host_alloc; request batch and "
                          "reply batch %s), max over ranks" % ("one after the other" if args.e2e_serial else "in flight together from two host threads"),
                "with_result_bodies": e2e_bodies, "per_rank": e2e_per_rank,
                "host_wait": ("sleep" if (os.environ.get("GGR_BLOCKING_SYNC", "1" if host_cpus() < 4 * torch.cuda.device_count() else "0") != "0") else "spin")
                             + " (usable CPUs %d, visible GPUs %d)" % (host_cpus(), torch.cuda.device_count()), "pcie_probe_gbs_each_way_per_rank": probe,
                "numa_node": eng.numa_node()},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "parity_checked_items": (parity["items"] * parity["directions"]) if parity else 0,
        "parity": parity,
        "configs": side,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def roofline_of(kern, dom, workload, n, step_ms, J_in, W_in, W_out, J_out, with_table):
    """roofline of the dominant kernel (device time from CUDA events around each launch, algorithmic bytes of the
    items it takes) against the measured HBM copy bandwidth"""
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    if not dom:
        return None
    a = kern[dom]["gbs"] or 0.0
    traffic, traffic_src = ncu_traffic(KERNEL_FN.get(dom, dom), workload, n)
    r = {"bound": "hbm", "kernel": dom, "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
         "step_read_gbs": (J_in + W_in) / (step_ms / 1000.0) / 1e9,
         "step_read_frac": (J_in + W_in) / (step_ms / 1000.0) / 1e9 / peak,
         "step_total_gbs": (J_in + W_in + W_out + J_out) / (step_ms / 1000.0) / 1e9}
    if with_table:
        r["kernels"] = kern
    return r


if __name__ == "__main__":
    main()
