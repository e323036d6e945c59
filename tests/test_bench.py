"""bench.py --dump-outputs: the sample of the last timed step's outputs, on the CPU arm against the oracle run here,
and (GPU) the engine arm's dump against the CPU arm's on the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import benchgen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--items", "3000", "--steps", "2", "--warmup", "1"]


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + list(args), cwd=ROOT, check=True,
                         capture_output=True, text=True).stdout
    line = json.loads(out.strip().splitlines()[-1])
    assert line["steps"] == 2
    return line


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_reference_arm_dump(tmp_path, oracle):
    _bench("--impl", "reference", "--dump-outputs", str(tmp_path))
    got = _load(tmp_path)
    assert sorted(got) == sorted("%s_%s" % (s, k) for s in ("request", "reply") for k in ("items", "status", "lengths", "bytes"))
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in os.listdir(tmp_path)) <= 64e6
    wl = benchgen.nested(3000, oracle.msg)
    for side, (out, off, st) in (("request", oracle.encode_batch(wl.req_msg, wl.req_json, wl.req_off, threads=4)),
                                 ("reply", oracle.decode_batch(wl.rep_msg, wl.rep_wire, wl.rep_off, threads=4))):
        items = got[side + "_items"].astype(np.int64)
        # the batch is larger than the sample: a strict, sorted subset of it
        assert 0 < len(items) < 3000 and (np.diff(items) > 0).all()
        assert (got[side + "_status"] == st[items]).all() and (st[items] == 0).all()
        off = off.astype(np.int64)
        assert (got[side + "_lengths"] == off[items + 1] - off[items]).all()
        want = np.concatenate([out[off[i]:off[i + 1]] for i in items])
        assert (got[side + "_bytes"] == want).all()


@pytest.mark.gpu
def test_engine_dump_equals_reference_arm(tmp_path):
    _bench("--no-cpu-baseline", "--no-side-configs", "--no-parity", "--dump-outputs", str(tmp_path / "engine"))
    _bench("--impl", "reference", "--dump-outputs", str(tmp_path / "reference"))
    eng, ref = _load(tmp_path / "engine"), _load(tmp_path / "reference")
    assert sorted(eng) == sorted(ref)
    for k in ref:
        assert eng[k].dtype == ref[k].dtype and np.array_equal(eng[k], ref[k]), k
