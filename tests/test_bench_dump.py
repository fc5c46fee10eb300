"""bench.py --dump-outputs: the files hold exactly what the timed path returned for the sampled documents (state JSON,
re-exported bytes, version vector, frontiers, import status) and the batch counters, in float32 / float64, within the
size budget.  The same checks run on the emulated build here and on the real library through bench.py itself."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from oracle import OracleDoc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EMU = os.path.join(HERE, "emu", "libloro_b200_emu.so")


def words(v):
    return [(v >> 32) & 0xFFFFFFFF, v & 0xFFFFFFFF]


def check_dump(d, blobs, atom_ops):
    files = os.listdir(d)
    assert sum(os.path.getsize(os.path.join(d, f)) for f in files) <= 64 << 20
    o = {f[:-4]: np.load(os.path.join(d, f)) for f in files}
    assert all(a.dtype in (np.float32, np.float64) for a in o.values())
    c = dict(zip(("docs", "docs_ok", "atom_ops"), (int(hi) << 32 | int(lo) for hi, lo in o["counters"][[0, 1, 6]])))
    assert c == {"docs": len(blobs), "docs_ok": len(blobs), "atom_ops": atom_ops}
    docs = o["docs"].astype(np.int64)
    k = min(len(blobs), bench.DUMP_DOCS)
    assert len(docs) == k and (np.diff(docs) > 0).all() and (o["status"] == 0).all()
    for r, i in enumerate(docs):
        ref = OracleDoc(1)
        st = ref.import_(blobs[i])
        for name, whole in (("json", ref.json_text()), ("export", ref.export_updates())):
            a, b = o[name + "_offsets"][r:r + 2].astype(np.int64)
            assert b - a == min(len(whole), bench.DUMP_STREAM_BYTES // k)
            assert o[name][a:b].astype(np.uint8).tobytes() == whole[:b - a], (name, i)
            assert o[name + "_len"][r] == len(whole)
            assert o[name + "_sha256"][r].astype(np.uint8).tobytes() == hashlib.sha256(whole).digest()
        rows = lambda a: [[int(x) for x in row[1:]] for row in a if row[0] == r]   # noqa: E731
        assert rows(o["vv"]) == [words(p) + [n] for p, n in sorted(ref.oplog_vv().items())]
        assert rows(o["frontiers"]) == [words(p) + [n] for p, n in sorted(ref.frontiers())]
        want = [[0] + words(p) + list(s) for p, s in sorted(st["success"].items())]
        want += [[1] + words(p) + list(s) for p, s in sorted((st["pending"] or {}).items())]
        assert rows(o["status_spans"]) == want
    return o


def test_dump_of_an_emulated_batch(tmp_path):
    import loro_b200
    from loro_b200 import api
    from loro_b200.workload import C3Batch
    subprocess.check_call([os.path.join(HERE, "emu", "build_emu.sh")])
    gen = C3Batch(70, n_ops=300, threads=4)
    buf = np.ascontiguousarray(gen.bytes)
    b = loro_b200.import_batch_device(buf.ctypes.data, gen.offsets, gen.lens, flags=api.LB_FLAG_EXPORT, lib_path=EMU, keep=buf)
    bench.dump_outputs(b, str(tmp_path), with_export=True)
    o = check_dump(str(tmp_path), gen.blobs(), gen.atom_ops)
    assert [int(hi) << 32 | int(lo) for hi, lo in o["counters"]] == list(b.counters().values())


@pytest.mark.gpu
def test_bench_dumps_its_last_step(tmp_path):
    from loro_b200.workload import C3Batch
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--docs", "96", "--ops-per-doc", "400", "--steps", "2",
                          "--warmup", "1", "--no-e2e", "--cpu-sample-docs", "2", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 2 and line["config"]["distinct_docs_per_gpu"] == 96
    gen = C3Batch(96, n_ops=400, threads=4)
    check_dump(str(tmp_path), gen.blobs(), gen.atom_ops)
