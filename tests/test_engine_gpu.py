"""Parity tests proper: the CUDA library on a real B200, through the C ABI, against the oracle.

Every test is marked gpu (skipped in the GPU-less build container, where tests/test_engine_emu.py runs the
same checks over the emulated build)."""
import gzip
import json
import os

import pytest

import oracle
from oracle import OracleDoc
from tests import workloads
from tests.engine_checks import check_batch_against_oracle

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def test_library_is_the_cuda_build():
    import loro_b200
    assert os.path.exists(loro_b200.library_path())
    blob, js, _, _ = workloads.make_doc_history(5, n_sites=2, n_ops=60)
    b = check_batch_against_oracle([blob], expect_json=[js])
    assert b.timings()["kernel_launches"] > 10


def test_small_mixed_and_fugue_known_answers():
    a = OracleDoc(1)
    t = a.get_text("text"); a.text_insert(t, 0, "Hello"); a.text_insert(t, 5, " World")
    l = a.get_list("list"); a.list_insert(l, 0, 1, 2, 3); a.delete(l, 1, 1)
    m = a.get_map("map"); a.map_set(m, "k", 5); a.map_set(m, "z", "str"); a.map_delete(m, "k")
    x, y = OracleDoc(0), OracleDoc(1)
    for ch in "olleH":
        x.text_insert(x.get_text("text"), 0, ch)
    for ch in "!dlroW ":
        y.text_insert(y.get_text("text"), 0, ch)
    workloads.merge(x, y)
    a2, b2, c2 = OracleDoc(0), OracleDoc(1), OracleDoc(2)
    c2.text_insert(c2.get_text("text"), 0, "2")
    workloads.merge(a2, c2)
    a2.text_insert(a2.get_text("text"), 0, "1")
    b2.text_insert(b2.get_text("text"), 0, "b")
    workloads.merge(a2, b2)
    batch = check_batch_against_oracle([a.export_updates(), x.export_updates(), a2.export_updates()])
    assert batch.get_deep_value(0) == {"text": "Hello World", "list": [1, 3], "map": {"z": "str"}}
    assert batch.get_deep_value(1) == {"text": "Hello World!"}
    assert batch.get_deep_value(2) == {"text": "b12"}


def test_pending_bad_blobs_and_empty_batch():
    import loro_b200
    a = OracleDoc(1)
    a.text_insert(a.get_text("t"), 0, "abc")
    a.commit()
    vv1 = a.oplog_vv()
    a.text_insert(a.get_text("t"), 3, "def")
    full, tail = a.export_updates(), a.export_updates(vv1)
    bad_sum = full[:30] + bytes([full[30] ^ 1]) + full[31:]
    batch = check_batch_against_oracle([full, tail, bad_sum, b"lor0" + full[4:], full[:10], b""])
    assert batch.status(1).pending == {1: (3, 6)} and batch.status(1).success == {}
    assert [batch.status(i).code for i in range(2, 6)] == [2, 1, 1, 1]
    assert loro_b200.import_batch([]).n_docs == 0


@pytest.mark.parametrize("seed", range(4))
def test_random_multi_site_histories(seed):
    blobs, jsons = [], []
    for k in range(48):
        blob, js, vv, _ = workloads.make_doc_history(seed * 1000 + k, n_sites=2 + (seed + k) % 4, n_ops=150 + 10 * (k % 20))
        blobs.append(blob)
        jsons.append(js)
    check_batch_against_oracle(blobs, expect_json=jsons)


def test_c1_two_peer_list_sync():
    """BASELINE config C1: 2 peers x 1000 List inserts each, import/export plumbing bit-exact."""
    blob, js = workloads.c1_two_peer_list(seed=1, n_each=1000)
    check_batch_against_oracle([blob] * 3, expect_json=[js] * 3)


def test_long_concurrent_branches():
    blobs, jsons = [], []
    for seed in range(6):
        blob, js, _, _ = workloads.make_doc_history(7000 + seed, n_sites=3, n_ops=2500, sync_prob=0.004)
        blobs.append(blob)
        jsons.append(js)
    check_batch_against_oracle(blobs, expect_json=jsons)


def test_more_than_32_peers_c4_shape():
    """Many concurrent sites on few documents (C4 shape at test size): peers >= 32 use the global-memory paths."""
    from tests.export_checks import check_export_against_oracle
    blobs, js = [], []
    for i in range(6):
        blob, j, _, _ = workloads.make_doc_history(4200 + i, n_sites=40 + 8 * (i % 3), n_ops=1500, sync_prob=0.04)
        blobs.append(blob)
        js.append(j)
    check_batch_against_oracle(blobs, expect_json=js)
    check_export_against_oracle(blobs)


def test_import_batch_groups_blobs_by_doc_id():
    """Several update blobs per document (doc_id grouping = LoroDoc::import_batch), shuffled, with duplicates."""
    import random
    import loro_b200
    from tests.test_engine_emu import _per_peer_blobs
    blobs, ids, want = [], [], []
    for d in range(24):
        whole, js, tot, parts = _per_peer_blobs(3100 + d, n_sites=2 + d % 4, n_ops=150 + 40 * (d % 7))
        random.Random(d).shuffle(parts)
        if d % 2:
            parts.append(parts[0])
        blobs += parts
        ids += [1000 + d] * len(parts)
        want.append((js, tot))
    order = list(range(len(blobs)))
    random.Random(99).shuffle(order)
    b = loro_b200.import_batch([blobs[i] for i in order], doc_ids=[ids[i] for i in order])
    assert b.n_docs == 24
    first_seen = []
    for i in order:
        if ids[i] not in first_seen:
            first_seen.append(ids[i])
    for k, did in enumerate(first_seen):
        js, tot = want[did - 1000]
        # the status is the reference's fold of per-blob statuses (loro.rs:1228-1258): changes parked by one blob and
        # released by a later one still show up in `pending`
        ost = OracleDoc(77).import_batch([blobs[i] for i in order if ids[i] == did])
        st = b.status(k)
        assert st.code == 0 and st.success == ost["success"] and st.pending == ost["pending"], (did, st, ost)
        assert b.json_bytes(k) == js
        assert b.oplog_vv(k) == tot


def test_automerge_trace_end_content(golden_dir):
    """BASELINE config C2 shape at small replication: the automerge-paper editing trace (259,778 patches,
    crates/loro-internal/benches/text_r.rs) must materialise to its recorded endContent."""
    import loro_b200
    blob = gzip.open(os.path.join(golden_dir, "automerge_trace_blob.bin.gz"), "rb").read()
    end = json.load(gzip.open(os.path.join(golden_dir, "automerge_trace.json.gz")))["endContent"]
    batch = loro_b200.import_batch([blob] * 4)
    for i in range(4):
        assert batch.status(i).code == 0
        assert batch.get_deep_value(i) == {"text": end}
    assert batch.counters()["atom_ops"] == 4 * 259778


def test_device_resident_entry_point_matches_host_path():
    import torch
    import loro_b200
    blobs = [workloads.make_doc_history(9000 + k, n_sites=3, n_ops=200)[0] for k in range(16)]
    host = loro_b200.import_batch(blobs)
    buf, offs, lens = loro_b200.pack_blobs(blobs)
    t = torch.from_numpy(buf).cuda()
    dev = loro_b200.import_batch_device(t.data_ptr(), offs, lens, keep=t)
    for i in range(len(blobs)):
        assert dev.status(i) == host.status(i)
        assert dev.json_bytes(i) == host.json_bytes(i)
    assert dev.counters()["state_hash"] == host.counters()["state_hash"]


# ---------------------------------------------------------------- phase 7: re-export (lb_doc_export_updates)
def test_export_matches_oracle_bytes_and_round_trips():
    from tests.export_checks import check_export_against_oracle
    blobs = [workloads.make_doc_history(7000 + i, n_sites=2 + i % 4, n_ops=200 + 30 * i, sync_prob=0.03 + 0.02 * (i % 3))[0]
             for i in range(24)]
    a = OracleDoc(7)   # typing runs and merged delete spans across commits
    t = a.get_text("t")
    for i, ch in enumerate("the quick brown fox"):
        a.text_insert(t, i, ch)
        if i % 3 == 2:
            a.commit()
    l = a.get_list("l")
    for i in range(40):
        a.list_insert(l, i, i)
    a.commit()
    for i in range(10):
        a.delete(l, 5, 1)
    for i in range(10):
        a.delete(l, 20 - i, 1)
    blobs.append(a.export_updates())
    check_export_against_oracle(blobs)


def test_export_generator_documents_and_scale_round_trip():
    """Byte parity with the oracle on a sample of C3 documents; on the whole batch the size-independent property:
    importing what was exported reproduces the state hash, and exporting again reproduces the bytes."""
    import loro_b200
    from loro_b200 import api
    from loro_b200.workload import C3Batch
    from tests.export_checks import check_export_against_oracle
    gen = C3Batch(512, n_ops=10000, threads=8)   # full-size documents: the 1,000-op prefix change gets split
    blobs = gen.blobs()
    check_export_against_oracle(blobs[:12], reimport=False)
    first = loro_b200.import_batch(blobs, flags=api.LB_FLAG_EXPORT)
    outs = [first.export_updates(i) for i in range(len(blobs))]
    again = loro_b200.import_batch(outs, flags=api.LB_FLAG_EXPORT)
    assert again.counters()["state_hash"] == first.counters()["state_hash"]
    assert again.counters()["atom_ops"] == first.counters()["atom_ops"] == gen.atom_ops
    for i in range(0, len(blobs), 37):
        assert again.export_updates(i) == outs[i]


def test_export_automerge_trace(golden_dir):
    from tests.export_checks import check_export_against_oracle
    blob = gzip.open(os.path.join(golden_dir, "automerge_trace_blob.bin.gz"), "rb").read()
    check_export_against_oracle([blob])


def test_export_with_pending_changes_and_after_import_batch():
    import random
    import loro_b200
    from loro_b200 import api
    from tests.test_engine_emu import _per_peer_blobs

    def change_num(blob):
        return sum(b["n_changes"] for b in oracle.decode_dump(blob)["blocks"])

    singles, single_refs, groups, ids, group_refs = [], [], [], [], []
    for k, seed in enumerate(range(3300, 3316)):
        whole, js, tot, parts = _per_peer_blobs(seed, n_sites=2 + seed % 3, n_ops=200)
        for p in parts:
            ref = OracleDoc(5)
            ref.import_(p)
            singles.append(p)
            single_refs.append(ref.export_updates())
        random.Random(seed).shuffle(parts)
        if seed % 2:
            parts.append(parts[0])
        ref = OracleDoc(5)
        for p in sorted(parts, key=lambda p: -change_num(p)):
            ref.import_(p)
        groups += parts
        ids += [k] * len(parts)
        group_refs.append((ref.json_text(), ref.export_updates()))
    b = loro_b200.import_batch(singles, flags=api.LB_FLAG_EXPORT)
    for i in range(len(singles)):
        assert b.export_updates(i) == single_refs[i], i
    g = loro_b200.import_batch(groups, doc_ids=ids, flags=api.LB_FLAG_EXPORT)
    for k, (js, ex) in enumerate(group_refs):
        assert g.json_bytes(k) == js and g.export_updates(k) == ex, k


def test_export_inserts_larger_than_a_block():
    from tests.export_checks import check_export_against_oracle
    from tests.test_export_emu import big_insert_documents
    check_export_against_oracle(big_insert_documents())


# ------------------------------------------------------------------ movable tree (SURVEY 8a row a16, config C5 shape)
def test_tree_known_answer_and_cycles():
    """loro_rust_test.rs:426-444 through the CUDA path, plus two concurrent moves that would close a cycle."""
    d = OracleDoc(1)
    t = d.get_tree("tree")
    root = d.tree_create(t)
    root2 = d.tree_create(t)
    d.tree_move(t, root2, root)
    d.map_set(d.tree_meta(root), "color", "red")
    a, b = OracleDoc(1), OracleDoc(2)
    ta, tb = a.get_tree("t"), b.get_tree("t")
    x = a.tree_create(ta)
    y = a.tree_create(ta)
    workloads.merge(b, a)
    a.tree_move(ta, x, y)
    b.tree_move(tb, y, x)
    workloads.merge(a, b)
    batch = check_batch_against_oracle([d.export_updates(), a.export_updates()])
    assert batch.get_deep_value(0) == {"tree": [
        {"parent": None, "meta": {"color": "red"}, "id": "0@1", "index": 0, "fractional_index": "80", "children": [
            {"parent": "0@1", "meta": {}, "id": "1@1", "index": 0, "children": [], "fractional_index": "80"}]}]}
    v = batch.get_deep_value(1)["t"]
    assert [n["id"] for n in v] == ["1@1"] and [c["id"] for c in v[0]["children"]] == ["0@1"]


@pytest.mark.parametrize("seed", range(3))
def test_tree_random_histories_c5_shape(seed):
    """C5 shape at a size the oracle replays in seconds: a base tree by one peer, then concurrent creates / moves
    (cycles across peers included) / deletes / meta writes by 2-4 peers; state JSON equal to the oracle's."""
    blobs, jsons = [], []
    for k in range(24):
        blob, js, vv, _ = workloads.make_tree_history(seed * 100 + k, n_sites=2 + (seed + k) % 3, n_base=30 + 10 * (k % 8),
                                                      n_ops=120 + 20 * (k % 10), mixed=k % 3 == 0)
        blobs.append(blob)
        jsons.append(js)
    check_batch_against_oracle(blobs, expect_json=jsons)


def test_tree_export_and_large_tree():
    from tests.export_checks import check_export_against_oracle
    import random
    blobs = [workloads.make_tree_history(900 + s, n_sites=2 + s % 3, n_base=40, n_ops=200, mixed=s % 2 == 0)[0] for s in range(12)]
    rnd = random.Random(4)
    a, b = OracleDoc(21), OracleDoc(22)
    ta, tb = a.get_tree("tree"), b.get_tree("tree")
    nodes = []
    for i in range(1500):
        parent = rnd.choice(nodes) if nodes and rnd.random() < 0.7 else None
        nodes.append(a.tree_create(ta, parent, -1 if rnd.random() < 0.6 else 0))
        if i % 7 == 0:
            a.commit()
    workloads.merge(b, a)
    for d, t in ((a, ta), (b, tb)):
        for _ in range(500):
            workloads.random_tree_edit(rnd, d, t, p_create=0.2)
    workloads.merge(a, b)
    blobs.append(a.export_updates())
    check_batch_against_oracle(blobs)
    check_export_against_oracle(blobs)


def test_config_c5_full_size_documents():
    """BASELINE config C5 at the stated per-document size (5,000-node tree + 3 x 1,000 concurrent moves): the
    generator's own merge (expected JSON), the oracle and the CUDA path agree on state and on re-exported bytes."""
    from loro_b200.workload import C5Batch
    from tests.export_checks import check_export_against_oracle
    g = C5Batch(12, want_json=True)
    blobs = g.blobs()
    want = [g.expected_json(i) for i in range(g.n_docs)]
    b = check_batch_against_oracle(blobs, expect_json=want)
    assert b.counters()["atom_ops"] == 12 * 8000
    check_export_against_oracle(blobs[:4])


def test_export_from_version_vector_and_c1_end_to_end():
    """lb_doc_export_updates(from): export(ExportMode::updates(vv)) on the CUDA path, byte-equal to the oracle; config C1
    (A exports updates(vv_B), B imports) driven by the engine."""
    import random
    import loro_b200
    from loro_b200 import api
    from tests.export_checks import check_export_from_versions
    for seed in range(4):
        check_export_from_versions(workloads.make_doc_history(7100 + seed, n_sites=2 + seed % 3, n_ops=300)[0], seed=seed)
    check_export_from_versions(workloads.make_tree_history(41, n_sites=3, n_base=40, n_ops=150, mixed=True)[0], seed=9)
    rnd = random.Random(3)
    a, b = OracleDoc(1), OracleDoc(2)
    la, lb = a.get_list("list"), b.get_list("list")
    for k in range(1000):
        a.list_insert(la, rnd.randint(0, a.seq_len(la)), rnd.randint(-10**6, 10**6))
        b.list_insert(lb, rnd.randint(0, b.seq_len(lb)), rnd.randint(-10**6, 10**6))
        if k % 10 == 9:
            a.commit(); b.commit()
    workloads.merge(a, b)
    batch = loro_b200.import_batch([a.export_updates()], flags=api.LB_FLAG_EXPORT)
    update_for_b = batch.export_updates(0, b.oplog_vv())
    assert update_for_b == a.export_updates(b.oplog_vv())
    b.import_(update_for_b)
    assert b.json_text() == a.json_text() == batch.json_bytes(0)


def test_nested_values_and_floats():
    from tests.export_checks import check_export_against_oracle
    a = OracleDoc(1)
    l, m = a.get_list("l"), a.get_map("m")
    a.list_insert(l, 0, {"b": 1, "a": [1, 2, {"z": None, "y": 2.5}]}, [1, [2, [3]]], 7, 0.1, -1e-7, 1e21, 5e-324)
    a.map_set(m, "k", {"x": {"y": {"z": "deep"}}, "w": [True, False], "aa": {}})
    a.map_set(m, "f", 3.14159)
    blob = a.export_updates()
    check_batch_against_oracle([blob])
    check_export_against_oracle([blob])


def test_config_c4_reduced_and_round_trip():
    """BASELINE config C4 (single rich-text document, 64 concurrent peers) at a size the oracle replays in seconds:
    state JSON and exported bytes equal the oracle's; importing the export again gives the same state hash."""
    import loro_b200
    from loro_b200 import api
    from loro_b200.workload import C4Doc
    from tests.export_checks import check_export_against_oracle
    g = C4Doc(base_chars=100000, n_peers=64, edits=800)
    blob = g.blob(0)
    b = check_batch_against_oracle([blob])
    assert b.counters()["atom_ops"] == g.atom_ops
    check_export_against_oracle([blob])


@pytest.mark.parametrize("seed", range(3))
def test_partially_known_changes_are_trimmed(seed):
    import loro_b200
    from loro_b200 import api
    e1, e2, n = workloads.overlapping_update_blobs(50 + seed)
    assert n > 0
    for blobs in ([e1, e2], [e2, e1]):
        ref = OracleDoc(7)
        for bl in workloads.import_batch_order(blobs):
            ref.import_(bl)
        bt = loro_b200.import_batch(blobs, doc_ids=[1, 1], flags=api.LB_FLAG_EXPORT)
        assert bt.status(0).code == 0
        assert bt.json_bytes(0) == ref.json_text()
        assert bt.oplog_vv(0) == ref.oplog_vv()
        assert bt.export_updates(0) == ref.export_updates()
        frm = {p: c // 2 for p, c in ref.oplog_vv().items()}
        assert bt.export_updates(0, frm) == ref.export_updates(frm)


@pytest.mark.parametrize("seed", range(4))
def test_import_batch_status_of_overlapping_updates(seed):
    """Overlapping, repeated and out-of-order update blobs into one document: state and ImportStatus (success starts,
    per-blob pending hulls) equal to the reference's import_batch fold."""
    from tests.test_engine_emu import test_import_batch_status_of_overlapping_updates as body
    import tests.test_engine_emu as emu
    saved = emu.EMU
    emu.EMU = None          # the real CUDA library
    try:
        body(seed)
    finally:
        emu.EMU = saved


@pytest.mark.parametrize("seed", range(3))
def test_docset_imports_against_existing_documents(seed):
    """lb_docset_import: a stream of update blobs (late, repeated, overlapping) into documents that live in device
    memory between calls; status / JSON / vv / frontiers / exported bytes equal to persistent oracle documents after
    every import."""
    from tests.docset_checks import check_docset_against_oracle
    steps = check_docset_against_oracle(n_docs=12, seed=seed, rounds=8, edits=16)
    assert steps > 5


def test_docset_compaction_equals_recreating_the_document_from_its_export():
    """LB_FLAG_COMPACT: a document without pending changes is kept as its own export; everything it answers afterwards
    equals a reference document re-created with fresh.import(doc.export(all_updates)) at the same points."""
    from tests.docset_checks import check_docset_against_oracle
    assert check_docset_against_oracle(n_docs=8, seed=21, rounds=8, edits=16, compact=True) > 5


def test_docset_updates_that_start_inside_known_changes():
    from tests.docset_checks import check_docset_against_oracle
    assert check_docset_against_oracle(n_docs=8, seed=2, rounds=8, edits=16, stale_inside=True) > 5


def test_host_batch_split_into_overlapping_sub_batches():
    from tests.test_engine_emu import test_host_batch_split_into_overlapping_sub_batches as body
    import tests.test_engine_emu as emu
    saved = emu.EMU
    emu.EMU = None
    try:
        body()
    finally:
        emu.EMU = saved


@pytest.mark.parametrize("which", ["c4_quarter.json", "c4_full.json"])
def test_config_c4_full_size_against_committed_oracle_digests(golden_dir, which):
    """BASELINE config C4 AT STATED SIZE (1 M base chars + 64 peers x 50 k concurrent edits, one document): the oracle
    replays it in minutes, so its answers are committed as digests (tests/golden/c4_full.json, made by
    tests/golden/make_c4_golden.py); the engine's JSON, version vector and exported bytes must hash to the same.
    `c4_quarter.json` is the same generator at 500 k base chars + 64 x 12.5 k edits (4.1 M atom ops)."""
    import json as _json
    import loro_b200
    from loro_b200 import api
    from loro_b200.workload import C4Doc
    path = os.path.join(golden_dir, which)
    if not os.path.exists(path):
        pytest.skip(f"tests/golden/{which} not generated")
    want = _json.load(open(path))
    g = C4Doc(**want["config"])
    blob = g.blob(0)
    xxh = lambda b: oracle.i64s(oracle.codec("xxh32", bytes(b), 0))[0] & 0xFFFFFFFF   # noqa: E731
    assert len(blob) == want["blob_len"] and xxh(blob) == want["blob_xxh32"]           # same generated input
    b = loro_b200.import_batch([blob], flags=api.LB_FLAG_EXPORT)
    st = b.status(0)
    assert st.code == 0 and st.pending is None
    assert b.counters()["atom_ops"] == want["atom_ops"]
    assert b.counters()["state_hash"] == want["state_hash"]
    js = b.json_bytes(0)
    assert len(js) == want["json_len"] and xxh(js) == want["json_xxh32"]
    assert {str(k): v for k, v in b.oplog_vv(0).items()} == want["vv"]
    ex = b.export_updates(0)
    assert len(ex) == want["export_len"] and xxh(ex) == want["export_xxh32"]


def test_library_next_to_the_emulated_build():
    """The emulated test build and the CUDA library in one process, the emulated one used first (as when the whole suite
    runs in one pytest process): each keeps its own host staging rings, and both give the same document."""
    import subprocess
    import sys
    emu = os.path.join(HERE, "emu", "libloro_b200_emu.so")
    subprocess.check_call([os.path.join(HERE, "emu", "build_emu.sh")])
    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import loro_b200\n"
        "from tests import workloads\n"
        "blob = workloads.make_doc_history(5, n_sites=2, n_ops=60)[0]\n"
        "a = loro_b200.import_batch([blob], lib_path=%r)\n"
        "b = loro_b200.import_batch([blob])\n"
        "assert b.status(0).code == 0 and a.json_bytes(0) == b.json_bytes(0)\n"
        "print('ok')\n"
    ) % (os.path.dirname(HERE), emu)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr[-2000:]


def test_plain_c_caller_runs_against_the_library(tmp_path, golden_dir):
    """examples/c/import_and_docset.c (plain C99 against include/loro_b200.h): import_batch of two updates of one document,
    then the same updates one call at a time into a docset document"""
    import subprocess
    import loro_b200
    exe = str(tmp_path / "demo")
    root = os.path.dirname(HERE)
    libdir = os.path.dirname(loro_b200.library_path())
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(root, "include"),
                           os.path.join(root, "examples", "c", "import_and_docset.c"), "-L" + libdir, "-lloro_b200", "-o", exe])
    a, b = OracleDoc(1), OracleDoc(2)
    a.text_insert(a.get_text("text"), 0, "hello")
    a.commit()
    u1 = a.export_updates()
    workloads.merge(b, a)
    b.text_insert(b.get_text("text"), 5, " world")
    b.commit()
    u2 = b.export_updates(a.oplog_vv())
    p1, p2 = str(tmp_path / "u1.bin"), str(tmp_path / "u2.bin")
    open(p1, "wb").write(u1)
    open(p2, "wb").write(u2)
    out = subprocess.run([exe, p1, p2], capture_output=True, text=True, env=dict(os.environ, LD_LIBRARY_PATH=libdir), timeout=120)
    assert out.returncode == 0, out.stderr
    assert out.stdout.count('"text":"hello world"') == 2, out.stdout      # the batch import and the second docset import
    assert '"text":"hello"' in out.stdout and "docset: 1 document(s)" in out.stdout
