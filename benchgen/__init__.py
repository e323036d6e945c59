"""Synthetic workloads for bench.py and the full-size parity tests (SURVEY.md section 8d).

Benchmark infrastructure - neither the product nor the oracle.  gen.cc is compiled with g++ into
benchgen/libggr_benchgen.so (built by __graft_entry__.build(); the .so travels to the GPU box).
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libggr_benchgen.so")
SEEDS = {2: 0xB2000002, 3: 0xB2000003, 4: 0xB2000004, 5: 0xB2000005}
_lib = None


def build(force=False):
    srcs = [os.path.join(HERE, "gen.cc"), os.path.join(HERE, "mixed.cc")]
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(x) for x in srcs):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", "-o", LIB] + srcs)
    return LIB


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):  # build() keeps it current; loading never writes into a built tree
            build()
        L = C.CDLL(LIB)
        vp = C.c_void_p
        L.ggr_gen_flat.argtypes = [C.c_uint64, C.c_int64, vp, C.c_uint64, vp, vp, C.c_uint64, vp]
        L.ggr_gen_nested.argtypes = [C.c_uint64, C.c_int64, vp, C.c_uint64, vp, vp, vp, C.c_uint64, vp]
        L.ggr_gen_blob.argtypes = [C.c_uint64, C.c_int64, C.c_uint32, vp, C.c_uint64, vp]
        L.ggr_gen_mixed.argtypes = [C.c_char_p, C.c_uint64, C.c_uint64, C.c_int64, vp, C.c_uint64, vp, vp, C.c_uint64, vp, vp]
        _lib = L
    return _lib


class Workload:
    """req_json/req_off/req_msg: request side (canonical arguments); rep_wire/rep_off/rep_msg: reply side."""

    def __init__(self, name):
        self.name = name
        self.req_json = self.req_off = self.req_msg = None
        self.rep_wire = self.rep_off = self.rep_msg = None

    @property
    def n(self):
        return len(self.rep_msg) if self.rep_msg is not None else len(self.req_msg)


def flat(n, msg_index, seed=SEEDS[2], first=0):
    """Config 2.  msg_index: callable full_name -> message index of the engine/oracle in use.
    `first` offsets the item indices (rank sharding: rank r generates items [r*n, (r+1)*n))."""
    L = _load()
    jc, wc = n * 700 + 4096, n * 320 + 4096
    j = np.empty(jc, np.uint8); jo = np.empty(n + 1, np.uint64)
    w = np.empty(wc, np.uint8); wo = np.empty(n + 1, np.uint64)
    rc = L.ggr_gen_flat(seed + 0x100000001B3 * first, n, j.ctypes.data, jc, jo.ctypes.data, w.ctypes.data, wc, wo.ctypes.data)
    assert rc == 0
    wl = Workload("flat")
    wl.req_json, wl.req_off = j[: int(jo[n])].copy(), jo
    wl.rep_wire, wl.rep_off = w[: int(wo[n])].copy(), wo
    wl.req_msg = np.full(n, msg_index("bench.Flat"), np.int32)
    wl.rep_msg = wl.req_msg.copy()
    return wl


def nested(n, msg_index, seed=SEEDS[3], first=0):
    """Config 3."""
    L = _load()
    jc, wc = n * 9000 + 4096, n * 7000 + 4096
    j = np.empty(jc, np.uint8); jo = np.empty(n + 1, np.uint64)
    w = np.empty(wc, np.uint8); wo = np.empty(n + 1, np.uint64)
    kind = np.empty(n, np.int32)
    rc = L.ggr_gen_nested(seed + 0x100000001B3 * first, n, j.ctypes.data, jc, jo.ctypes.data, kind.ctypes.data, w.ctypes.data, wc,
                          wo.ctypes.data)
    assert rc == 0
    wl = Workload("nested")
    wl.req_json, wl.req_off = j[: int(jo[n])].copy(), jo
    wl.rep_wire, wl.rep_off = w[: int(wo[n])].copy(), wo
    P = "com.example.complex."
    req = np.array([msg_index(P + "ProcessNodeRequest"), msg_index(P + "CreateDocumentRequest")], np.int32)
    rep = np.array([msg_index(P + "Node"), msg_index(P + "GetUserProfileResponse")], np.int32)
    wl.req_msg, wl.rep_msg = req[kind], rep[kind]
    wl.kind = kind
    return wl


def blob(n, msg_index, payload=65536, seed=SEEDS[4], first=0):
    """Config 4 (reply side only)."""
    L = _load()
    wc = n * (payload + 64) + 4096
    w = np.empty(wc, np.uint8); wo = np.empty(n + 1, np.uint64)
    rc = L.ggr_gen_blob(seed + 0x100000001B3 * first, n, payload, w.ctypes.data, wc, wo.ctypes.data)
    assert rc == 0
    wl = Workload("blob")
    wl.rep_wire, wl.rep_off = w[: int(wo[n])].copy(), wo
    wl.rep_msg = np.full(n, msg_index("bench.Blob"), np.int32)
    return wl


# ---- configs[4]: mixed replay -------------------------------------------------------------------
MIXED_METHODS = ["hello.HelloService.SayHello", "com.example.complex.UserProfileService.GetUserProfile",
                 "com.example.complex.DocumentService.CreateDocument", "com.example.complex.NodeService.ProcessNode"] + \
                ["mixed.MixedService.Call%02d" % k for k in range(28)]
_plans = {}


def _mixed_plan(fds_bytes):
    """(plan bytes for gen_mixed, [(input full name, output full name)] per method) from a FileDescriptorSet"""
    import struct
    from google.protobuf import descriptor_pb2, descriptor_pool
    key = hash(fds_bytes)
    if key in _plans:
        return _plans[key]
    fds = descriptor_pb2.FileDescriptorSet()
    fds.ParseFromString(fds_bytes)
    pool = descriptor_pool.DescriptorPool()
    for f in fds.file:
        pool.Add(f)
    msgs, enums, index, eindex = [], [], {}, {}

    def s(b):
        b = b.encode()
        return struct.pack("<I", len(b)) + b

    def enum_id(ed):
        if ed.full_name not in eindex:
            eindex[ed.full_name] = len(enums)
            enums.append(ed)
        return eindex[ed.full_name]

    def msg_id(md):
        if md.full_name in index:
            return index[md.full_name]
        index[md.full_name] = len(msgs)
        msgs.append(md)
        for f in md.fields:
            if f.message_type is not None and f.message_type.full_name != "google.protobuf.Timestamp":
                msg_id(f.message_type)
        return index[md.full_name]

    methods = []
    for full in MIXED_METHODS:
        svc, meth = full.rsplit(".", 1)
        m = pool.FindServiceByName(svc).methods_by_name[meth]
        methods.append((m.input_type, m.output_type))
        msg_id(m.input_type)
        msg_id(m.output_type)
    out = [struct.pack("<I", 0)]
    i = 0
    while i < len(msgs):  # msgs grows while nested types are discovered
        md = msgs[i]
        i += 1
        rec = [struct.pack("<I", len(md.fields))]
        for f in md.fields:
            flags, child = 0, -1
            is_map = f.message_type is not None and f.message_type.GetOptions().map_entry
            repeated = f.label == f.LABEL_REPEATED
            if is_map:
                flags |= 4
            elif repeated:
                flags |= 1
                packable = f.type not in (f.TYPE_STRING, f.TYPE_BYTES, f.TYPE_MESSAGE)
                if packable and (not f.has_options or not f.GetOptions().HasField("packed") or f.GetOptions().packed):
                    flags |= 2
            real_oneof = f.containing_oneof is not None and not f.containing_oneof.name.startswith("_")
            if real_oneof:
                flags |= 8
            if f.has_presence and not real_oneof:
                flags |= 16
            if f.message_type is not None:
                if f.message_type.full_name == "google.protobuf.Timestamp":
                    flags |= 32
                else:
                    child = msg_id(f.message_type)
            if f.enum_type is not None:
                child = enum_id(f.enum_type)
            oneof = f.containing_oneof.index if real_oneof else -1
            rec.append(struct.pack("<IIIii", f.number, f.type, flags, oneof, child) + s(f.name) + s(f.json_name))
        out.append(b"".join(rec))
    out[0] = struct.pack("<I", len(msgs))
    out.append(struct.pack("<I", len(enums)))
    for ed in enums:
        out.append(struct.pack("<I", len(ed.values)) + b"".join(struct.pack("<i", v.number) + s(v.name) for v in ed.values))
    out.append(struct.pack("<I", len(methods)) + b"".join(struct.pack("<II", index[a.full_name], index[b.full_name]) for a, b in methods))
    _plans[key] = (b"".join(out), [(a.full_name, b.full_name) for a, b in methods])
    return _plans[key]


def mixed(n, msg_index, fds_bytes=None, seed=SEEDS[5], first=0):
    """Config 5: calls over 32 methods (4 of the reference's own protos + 28 generated, tests/golden/make_descriptors.py
    mixed_file), method Zipf(1.1), size Zipf(1.2) over 64 B .. 64 KiB.  wl.method[i] indexes MIXED_METHODS."""
    L = _load()
    if fds_bytes is None:
        with open(os.path.join(os.path.dirname(HERE), "tests", "golden", "schemas.binpb"), "rb") as fh:
            fds_bytes = fh.read()
    plan, names = _mixed_plan(fds_bytes)
    jc = wc = n * 1100 + (1 << 20)
    while True:
        j = np.empty(jc, np.uint8); jo = np.empty(n + 1, np.uint64)
        w = np.empty(wc, np.uint8); wo = np.empty(n + 1, np.uint64)
        meth = np.empty(n, np.int32)
        rc = L.ggr_gen_mixed(plan, len(plan), seed + 0x100000001B3 * first, n, j.ctypes.data, jc, jo.ctypes.data, w.ctypes.data, wc,
                             wo.ctypes.data, meth.ctypes.data)
        if rc == 0:
            break
        assert rc == -1, rc
        jc, wc = int(jo[n]) + 64, int(wo[n]) + 64
    wl = Workload("mixed")
    wl.req_json, wl.req_off = j[: int(jo[n])].copy(), jo
    wl.rep_wire, wl.rep_off = w[: int(wo[n])].copy(), wo
    req = np.array([msg_index(a) for a, _ in names], np.int32)
    rep = np.array([msg_index(b) for _, b in names], np.int32)
    wl.method = meth
    wl.req_msg, wl.rep_msg = req[meth], rep[meth]
    wl.method_names = list(MIXED_METHODS)
    return wl
