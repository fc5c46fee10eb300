#!/usr/bin/env python3
"""bench.py -- merged CRDT ops/sec of the batched import hot path (BASELINE.json metric).

One "step" = one pass of the hot path (decode -> causal scan -> eg-walker / tree merge -> deep JSON -> re-export) over one
batch of synthetic documents.  --config picks the BASELINE.json configuration (SURVEY.md 8d): C3 (default, the one the
metric is quoted on: N docs x 10k mixed List/Map atom ops, 3 concurrent peers), C2 (automerge-paper trace x 4096 docs;
--c2-distinct-peers gives every copy its own peer id), C4 (ONE text document, 1M chars + 64 peers x 50k concurrent
edits: replicas only), C5 (10k docs x 5k-node movable trees with concurrent moves).
`value` is measured with the update blobs already resident in HBM (lb_import_batch_device); `e2e` is the same metric
through the host-buffer path a user calls (loro_b200.import_batch -> lb_import_batch: pinned staging + H2D inside the
timed region, JSON + status + re-exported blobs read back to the host; large batches go as two overlapping sub-batches).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2|C3|C4|C5] [--docs D] [--ops-per-doc 10000]
                  [--dump-outputs DIR]   # what the last timed step returned, as DIR/*.npy (dump_outputs)
  python bench.py --impl reference ...     # the CPU arm: the oracle port of the reference path on host cores

Under torchrun (N>1) every rank imports its own shard of documents (weak scaling: per-GPU work fixed) and
the per-shard summary counters are exchanged with one NCCL all-gather per step.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "merged CRDT ops/sec (batched docs)"
UNIT = "ops/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="C3", choices=["C2", "C3", "C4", "C5"],
                    help="BASELINE.json config: C3 = 100k docs x 10k mixed List/Map ops, 3 peers (the config the metric is quoted on); "
                         "C2 = automerge-paper text trace x 4096 docs; C4 = ONE rich-text doc, 1M chars + 64 peers x 50k concurrent edits "
                         "(does not shard: every GPU runs a replica); C5 = 10k docs x 5k-node movable trees with 3 x 1k concurrent moves")
    ap.add_argument("--c2-distinct-peers", action="store_true",
                    help="C2: document i is typed by peer i + 1 (own peer id and checksum in every copy) instead of byte-identical copies")
    ap.add_argument("--c4-base", type=int, default=1000000)
    ap.add_argument("--c4-peers", type=int, default=64)
    ap.add_argument("--c4-edits", type=int, default=50000)
    ap.add_argument("--docs", type=int, default=0, help="documents per GPU (0 = the config's figure: C3 100k, C2 4096, C5 10k)")
    ap.add_argument("--ops-per-doc", type=int, default=10000)
    ap.add_argument("--peers", type=int, default=3)
    ap.add_argument("--tree-nodes", type=int, default=5000, help="C5: nodes of the base tree")
    ap.add_argument("--tree-moves", type=int, default=1000, help="C5: concurrent moves per peer")
    ap.add_argument("--distinct", type=int, default=0, help="distinct seeded docs generated per GPU; the batch cycles through them (0 = all distinct)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample-docs", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-export", action="store_true", help="skip the re-export phase (import + state only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (see dump_outputs; "
                         "under torchrun, rank 0's documents)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path's outputs; the reference arm has none")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def begin_region(self):
        """nvidia-smi needs about a second before its first line: the sampler starts before the warm-up steps and
        only what arrives after this call (= during the timed region) is reported."""
        self.region0 = len(self.samples)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        region = self.samples[getattr(self, "region0", 0):]
        note = None
        if not region and self.samples:   # timed region shorter than one sampling period: closest samples instead
            region = self.samples[-2:]
            note = "no sample fell inside the timed region; last warm-up samples reported"
        for s in region:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm)}
        if note:
            out["note"] = note
        return out


def default_docs(args, world):
    """Documents per GPU: BASELINE's figure for the config at every N, so that per-GPU work is fixed (weak scaling)."""
    return args.docs or {"C3": 100000, "C2": 4096, "C4": 1, "C5": 10000}[args.config]


class TraceBatch:
    """Config C2: the automerge-paper editing trace (259,778 single-character patches applied to a root Text by one
    peer, a transaction every 10 patches, exported with all_updates) -- the committed fixture
    tests/golden/automerge_trace_blob.bin.gz, made by tests/golden/make_golden.py with the oracle.  Every document
    of the batch is a copy of that blob with its own bytes in HBM."""

    def __init__(self):
        import gzip
        import numpy as np
        blob = gzip.open(os.path.join(ROOT, "tests", "golden", "automerge_trace_blob.bin.gz"), "rb").read()
        self.n_docs = 1
        self.bytes = np.zeros(((len(blob) + 15) & ~15) + 64, dtype=np.uint8)
        self.bytes[:len(blob)] = np.frombuffer(blob, dtype=np.uint8)
        self.offsets = np.zeros(1, dtype=np.uint64)
        self.lens = np.array([len(blob)], dtype=np.uint32)
        self.atom_ops = 0   # taken from the engine's counters (sum of change.atom_len)
        self._blob = blob

    def blob(self, i):
        return self._blob


def peer_id_offsets(blob):
    """byte offsets of every 8-byte peer id in the `peers` tables of a FastUpdates blob's blocks (block_meta_encode.rs:
    the header section starts with ULEB n_peers, then n_peers x u64 LE)"""
    def uleb(i):
        v, sh = 0, 0
        while True:
            c = blob[i]
            i += 1
            v |= (c & 0x7f) << sh
            sh += 7
            if not c & 0x80:
                return v, i
    out, i, n = [], 22, len(blob)
    while i < n:
        ln, i = uleb(i)
        end, j = i + ln, i
        for _ in range(5):
            _, j = uleb(j)
        _, j = uleb(j)            # length prefix of the header section
        npeers, j = uleb(j)
        out += [j + 8 * k for k in range(npeers)]
        i = end
    return out


class TraceBatchDistinctPeers(TraceBatch):
    """Config C2, SURVEY 8d's variant: document i is the same trace typed by peer (i + 1) -- every copy of the blob gets
    its own peer id in every block's peers table and its own checksum, so no two documents share their bytes."""

    def __init__(self, n_docs):
        import struct
        import numpy as np
        import oracle
        super().__init__()
        base = bytearray(self._blob)
        offs = peer_id_offsets(base)
        assert offs and all(base[o:o + 8] == base[offs[0]:offs[0] + 8] for o in offs)   # the trace has one author
        span = (len(base) + 15) & ~15
        self.n_docs = n_docs
        self.bytes = np.zeros(span * n_docs + 64, dtype=np.uint8)
        self.offsets = (np.arange(n_docs, dtype=np.uint64) * np.uint64(span))
        self.lens = np.full(n_docs, len(base), dtype=np.uint32)
        self._blobs = []
        for d in range(n_docs):
            pid = struct.pack("<Q", d + 1)
            for o in offs:
                base[o:o + 8] = pid
            h = oracle.i64s(oracle.codec("xxh32", bytes(base[20:]), 0x4F524F4C))[0] & 0xFFFFFFFF
            base[16:20] = struct.pack("<I", h)
            self.bytes[d * span:d * span + len(base)] = np.frombuffer(bytes(base), dtype=np.uint8)
            self._blobs.append(bytes(base))

    def blob(self, i):
        return self._blobs[i]


def workload_text(args, n_docs, extra=""):
    if args.config == "C2":
        return (f"C2: automerge-paper text trace (259,778 patches -> one FastUpdates blob of 1 peer) replicated x {n_docs} docs/GPU, "
                f"each copy with its own bytes in HBM{' and its own peer id (document i typed by peer i + 1)' if args.c2_distinct_peers else ''} (SURVEY.md 8d){extra}")
    if args.config == "C4":
        return (f"C4: {n_docs} rich-text document(s)/GPU (replicas: a single document does not shard), {args.c4_base} ASCII chars by peer 0 + "
                f"{args.c4_peers} peers x {args.c4_edits} concurrent edits (70 % insert 1-8 chars, 30 % delete 1-8), never synced (SURVEY.md 8d){extra}")
    if args.config == "C5":
        return (f"C5: {n_docs} docs/GPU x movable tree of {args.tree_nodes} nodes (fan-out <= 8) built by peer 0 + {args.peers} peers x "
                f"{args.tree_moves} concurrent moves (random target / parent, cycles across peers included), one FastUpdates blob per doc (SURVEY.md 8d){extra}")
    return (f"C3: {n_docs} docs/GPU x {args.ops_per_doc} mixed List/Map atom ops, {args.peers} concurrent peers, "
            f"one FastUpdates blob per doc (SURVEY.md 8d){extra}")


GEN_CORES = 16   # host cores the generation budget below is sized for


def affordable_distinct(args, world, n_docs):
    """How many DISTINCT documents this rank's share of GEN_CORES host cores can generate in about 90 s
    (~1.2 M generated atom ops/s/core); the batch is filled by cycling through them (every copy has its own bytes
    in HBM; `distinct_docs_per_gpu` in the config says how many there are).  The budget is fixed rather than taken
    from this host's cores, so that the same arguments give the same inputs on every machine."""
    if args.config == "C2" and args.c2_distinct_peers:
        return n_docs
    if args.config in ("C2", "C4"):
        return 1
    if args.distinct:
        return min(args.distinct, n_docs)
    cores = max(1, GEN_CORES // max(1, world))
    if args.config == "C5":   # ~0.7 M generated tree ops/s/core
        return max(64, min(n_docs, int(cores * 0.7e6 * 90 / (args.tree_nodes + args.peers * args.tree_moves))))
    return max(64, min(n_docs, int(cores * 1.2e6 * 90 / args.ops_per_doc)))


def make_workload(args, rank, world, n_docs):
    from loro_b200.workload import C3Batch, C4Doc, C5Batch
    distinct = affordable_distinct(args, world, n_docs)
    threads = max(1, (host_cores() or 1) // max(1, world))
    t0 = time.time()
    if args.config == "C2":
        gen = TraceBatchDistinctPeers(n_docs) if args.c2_distinct_peers else TraceBatch()
    elif args.config == "C4":
        gen = C4Doc(args.c4_base, args.c4_peers, args.c4_edits, seed=rank)
    elif args.config == "C5":
        gen = C5Batch(distinct, n_nodes=args.tree_nodes, n_peers=args.peers, n_moves=args.tree_moves, first_doc=rank * n_docs, threads=threads)
    else:
        gen = C3Batch(distinct, n_ops=args.ops_per_doc, n_peers=args.peers, first_doc=rank * n_docs, threads=threads)
    return gen, distinct, time.time() - t0


def cpu_baseline(args, gen, threads=None):
    """The oracle port of the reference's CPU path on a bounded sample of the same workload."""
    import oracle
    import numpy as np
    threads = threads or (host_cores() or 1)
    n = args.cpu_sample_docs or min(gen.n_docs, max(64, min(4096, threads * 48)))
    if args.config == "C2":
        n = args.cpu_sample_docs or max(1, min(threads, 16))    # one trace import is ~0.26 M ops: a few copies suffice
    if args.config == "C4":
        # the full document takes the restated CPU path ~80 s (one core: a single document has one task), more than the
        # bench may spend: a quarter-size instance of the same generator (500 k base chars, 64 peers x 12.5 k edits, ~35 s)
        from loro_b200.workload import C4Doc
        gen = C4Doc(min(args.c4_base, 500000), min(args.c4_peers, 64), min(args.c4_edits, 12500), seed=0)
        n, threads = 1, 1
        reduced = f" -- REDUCED instance ({gen.config['base_chars']} base chars, {gen.config['n_peers']} peers x {gen.config['edits']} edits)"
    else:
        reduced = ""
    # oracle.bench_import wants contiguous [off[i], off[i+1]) blobs: re-pack exact lengths
    blobs = [gen.blob(i % gen.n_docs) for i in range(n)]
    buf = b"".join(blobs)
    o = [0]
    for b in blobs:
        o.append(o[-1] + len(b))
    r = oracle.bench_import(np.frombuffer(buf, dtype=np.uint8), o, threads=threads, want_json=True,
                            want_export=not args.no_export)
    return {"value": r["ops"] / r["seconds"], "unit": UNIT, "cores": threads, "kind": "port", "ops": r["ops"],
            "sample": f"{n} docs of the same {args.config} workload{reduced} ({r['ops']} atom ops, {r['seconds']:.2f} s), import + deep JSON{"" if args.no_export else " + export(all_updates)"} per doc, one doc per task; "
                      "the CPU arm is the C++ restatement of the reference algorithm (oracle/), not the Rust reference (no cargo in the image)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import oracle
    oracle.build()
    threads = host_cores() or 1
    n = args.cpu_sample_docs or max(64, min(4096, threads * 48))
    if args.config == "C5":
        n = args.cpu_sample_docs or max(64, min(1024, threads * 24))
    if args.config == "C4":
        n = 1
    ns = argparse.Namespace(**vars(args))
    ns.distinct = 0
    gen, _, _ = make_workload(ns, 0, 1, n)
    steps, warm = args.steps, args.warmup
    vals = []
    for s in range(warm + steps):
        cb = cpu_baseline(args, gen, threads)
        if s >= warm:
            vals.append(cb)
    total_ops_per_s = statistics.mean(v["value"] for v in vals)
    ms = 1e3 * (vals[-1]["ops"] / total_ops_per_s)
    for v in vals:
        v.pop("ops", None)
    line = {"impl": "reference", "metric": METRIC, "value": total_ops_per_s, "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int64", "data": "synthetic",
            "config": {"workload": workload_text(args, n, " -- bounded sample of the ours-arm workload")},
            "cpu_baseline": {"value": total_ops_per_s, "unit": UNIT, "cores": vals[-1]["cores"], "kind": "port", "sample": vals[-1]["sample"]},
            "e2e": {"value": total_ops_per_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def host_cores():
    """Cores this process can really use: min(affinity, cgroup cpu.max quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def ncu_traffic(kernel_key, rows):
    """dram bytes per launch for `rows` op rows, scaled from the committed `ncu --set full` capture (profiles/)."""
    try:
        here = os.path.dirname(os.path.abspath(__file__))
        best = None
        for fn in sorted(os.listdir(os.path.join(here, "profiles"))):
            if fn.endswith("_ncu_facts.json"):
                best = os.path.join(here, "profiles", fn)
        f = json.load(open(best))[kernel_key]
        return {"bytes": f["dram_bytes_per_op_row"] * rows, "source": os.path.basename(best) + ": dram__bytes_read+write per op row x rows"}
    except Exception:
        return None


DUMP_DOCS = 64                # documents sampled, with a fixed seed, for the per-document outputs
DUMP_STREAM_BYTES = 6000000   # bytes kept of each per-document byte stream (JSON, re-export), shared by the sample


def dump_outputs(b, out_dir, with_export):
    """--dump-outputs DIR: what the timed path returned to its caller in the last timed step, as .npy files by which two
    builds can be compared (about 50 MB at most).  64-bit values (peer ids, state_hash) are split into two float64
    columns, high and low 32 bits, so that every value is exact.
      counters.npy          [10, 2]  the batch counters, in loro_b200.shard.COUNTER_KEYS order
      docs.npy              [K]      the K = min(n_docs, DUMP_DOCS) sampled documents (fixed seed, ascending)
      status.npy            [K]      ImportStatus code of each
      status_spans.npy      [S, 6]   sample row, 0 = success / 1 = pending, peer hi, peer lo, start, end
      vv.npy, frontiers.npy [V, 4]   sample row, peer hi, peer lo, counter
      json.npy              float32  each sampled document's JSON bytes, back to back, at most DUMP_STREAM_BYTES // K
                                     of each (a prefix); json_offsets.npy [K + 1] delimits them
      json_len.npy          [K]      the length of the whole JSON; json_sha256.npy [K, 32] its SHA-256, byte by byte
      export*.npy                    the same four for the re-exported blob (not with --no-export)"""
    import hashlib
    import numpy as np
    from loro_b200.shard import COUNTER_KEYS

    def words(v):
        return (int(v) >> 32) & 0xFFFFFFFF, int(v) & 0xFFFFFFFF

    c = b.counters()
    out = {"counters": np.array([words(c[k]) for k in COUNTER_KEYS], dtype=np.float64)}
    k = min(b.n_docs, DUMP_DOCS)
    docs = [int(i) for i in np.sort(np.random.default_rng(0).choice(b.n_docs, size=k, replace=False))]
    out["docs"] = np.array(docs, dtype=np.float64)
    status, spans, vv, fr = [], [], [], []
    for r, i in enumerate(docs):
        st = b.status(i)
        status.append(st.code)
        for kind, d in ((0, st.success), (1, st.pending or {})):
            spans += [(r, kind, *words(p), s, e) for p, (s, e) in sorted(d.items())]
        vv += [(r, *words(p), n) for p, n in sorted(b.oplog_vv(i).items())]
        fr += [(r, *words(p), n) for p, n in b.oplog_frontiers(i)]
    out["status"] = np.array(status, dtype=np.float64)
    out["status_spans"] = np.array(spans, dtype=np.float64).reshape(-1, 6)
    out["vv"] = np.array(vv, dtype=np.float64).reshape(-1, 4)
    out["frontiers"] = np.array(fr, dtype=np.float64).reshape(-1, 4)
    cap = DUMP_STREAM_BYTES // k
    for name, get in [("json", b.json_bytes)] + ([("export", b.export_updates)] if with_export else []):
        whole = [get(i) for i in docs]
        kept = [w[:cap] for w in whole]
        out[name] = np.frombuffer(b"".join(kept), dtype=np.uint8).astype(np.float32)
        out[name + "_offsets"] = np.cumsum([0] + [len(x) for x in kept]).astype(np.float64)
        out[name + "_len"] = np.array([len(w) for w in whole], dtype=np.float64)
        out[name + "_sha256"] = np.array([list(hashlib.sha256(w).digest()) for w in whole], dtype=np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    import numpy as np
    import torch
    import loro_b200
    from loro_b200.shard import gather_counters
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    # one rank per GPU: keep the rank's host buffers, the pinned staging ring and the gather threads on the NUMA node
    # of its GPU (the host side limited e2e scaling at 8 ranks in round 1)
    numa_bound = loro_b200.numa_bind(local) if world > 1 else False
    n_docs = default_docs(args, world)
    gen, distinct, gen_s = make_workload(args, rank, world, n_docs)
    # lay the batch out in HBM: cycle through the distinct docs (each copy has its own bytes in HBM)
    idx = np.arange(n_docs) % distinct
    lens = gen.lens[idx].astype(np.uint32)
    src = torch.from_numpy(np.ascontiguousarray(gen.bytes)).to(dev)
    g_offs = gen.offsets.astype(np.uint64)
    if distinct == n_docs:
        d_bytes = src
        offs = g_offs.copy()
    else:
        span = (int(src.numel()) + 15) & ~15            # one full copy of the generated buffer, 16-byte aligned
        reps = (n_docs + distinct - 1) // distinct
        d_bytes = torch.zeros(span * reps + 64, dtype=torch.uint8, device=dev)
        for c in range(reps):
            d_bytes[c * span:c * span + src.numel()] = src
        offs = (g_offs[idx] + (np.arange(n_docs) // distinct).astype(np.uint64) * np.uint64(span)).astype(np.uint64)
        del src

    xflags = 0 if args.no_export else loro_b200.api.LB_FLAG_EXPORT

    def step(keep=False):
        b = loro_b200.import_batch_device(d_bytes.data_ptr(), offs, lens, device=local, flags=xflags, keep=d_bytes)
        c = b.counters()
        if world > 1:
            gather_counters(c, device=dev)  # the one collective of the path: per-shard summary counters (NCCL)
        tm = b.timings()
        if keep:
            return c, tm, b
        b.close()
        return c, tm, None

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        c, tm, _ = step()
    assert c["docs_ok"] == n_docs, c
    atoms_per_step = c["atom_ops"]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.begin_region()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    t_wall = time.time()
    phase = {}
    launches = 0
    for s in range(args.steps):
        # rank 0 keeps the last step's batch open for --dump-outputs (closed below, once the timed region has ended)
        c, tm, last = step(keep=bool(args.dump_outputs) and rank == 0 and s == args.steps - 1)
        launches += tm["kernel_launches"]
        for k in ("frame", "decode", "resolve", "classify", "integrate", "tree", "materialise", "reexport", "total_device",
                  "alloc_host_ms", "host_call_ms", "host_tail_ms"):
            phase[k] = phase.get(k, 0.0) + tm[k]
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall_ms = (time.time() - t_wall) * 1e3
    dev_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    if last is not None:
        dump_outputs(last, args.dump_outputs, with_export=bool(xflags))
        last.close()
    total_atoms = atoms_per_step * world
    value = total_atoms * args.steps / (dev_ms * 1e-3)
    ms_per_step = dev_ms / args.steps

    # ---- e2e: host buffers in, JSON + status out, through the public C-ABI call
    e2e = None
    if not args.no_e2e:
        blob_of = [gen.blob(k) for k in range(distinct)]   # copies of a document share one host buffer
        blobs = [blob_of[int(idx[i])] for i in range(n_docs)]
        h2d = int(lens.sum())
        for _ in range(1):
            b = loro_b200.import_batch(blobs, device=local, flags=xflags)
            b.fetch_json()
            b.close()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.time()
        d2h = 0
        for _ in range(args.steps):
            b = loro_b200.import_batch(blobs, device=local, flags=xflags)   # large batches: overlapping sub-batches (api.MultiBatch)
            b.fetch_json()   # pulls the JSON of every document of the batch to the host
            cc = b.counters()
            d2h = cc["json_bytes"] + n_docs * 256
            if xflags:
                b.fetch_exports()  # pulls every document's re-exported blob to the host
                d2h += b.timings()["export_bytes"]
            b.close()
        torch.cuda.synchronize()
        e_ms = (time.time() - t0) * 1e3
        te = torch.tensor([e_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e = {"value": total_atoms * args.steps / (float(te.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(d2h),
               "host_sub_batches": loro_b200.api.auto_split(blobs)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    n_steps = args.steps
    rows = c["op_rows"]
    dec_ms = phase["decode"] / n_steps
    dec_bytes = tm["decode_bytes_read"] + tm["decode_bytes_written"]
    # the dominant kernel = the one behind the longest phase; algorithmic bytes per SURVEY 8d (DESIGN.md section 6):
    #   list/text integration 52 B per run (= op row); decode blob + SoA bytes; causal scan 20 B/change + 12 B/dep
    #   (deps not counted here); materialise JSON bytes written + as many payload bytes read; re-export rows x 13 B read
    #   + blob bytes written; movable tree 36 B per tree op (ids of subject and parent 24, position ref 4, lamport 4
    #   read; parent link 4 written)
    candidates = {
        "integrate": ("k_seq_integrate", rows * 52, "seq"),
        "decode": ("k_block_count+k_block_decode", dec_bytes, "decode"),
        "tree": ("k_tree_build", tm["tree_ops"] * 36, None),
        "materialise": ("k_json", 2 * c["json_bytes"], None),
        "reexport": ("k_exp_encode+k_exp_changes", rows * 13 + tm["export_bytes"], None),
        "resolve": ("k_doc_tables+k_doc_causal", c["changes"] * 20, None),
    }
    top = max(candidates, key=lambda k: phase.get(k, 0.0))
    kname, abytes, facts_key = candidates[top]
    top_ms = phase[top] / n_steps
    roof = {"bound": "hbm", "kernel": kname, "achieved": abytes / (top_ms * 1e-3) / 1e9, "peak": peak,
            "unit": "GB/s", "peak_source": peak_src, "traffic": None, "algorithmic_bytes_per_launch": abytes,
            "share_of_step": top_ms / (phase["total_device"] / n_steps)}
    roof["frac"] = roof["achieved"] / peak
    tr = ncu_traffic(facts_key, rows) if facts_key else None
    if tr:
        roof["traffic"] = tr["bytes"]
        roof["traffic_source"] = tr["source"]
    dec_roof = {"bound": "hbm", "kernel": "k_block_count+k_block_decode", "achieved": dec_bytes / (dec_ms * 1e-3) / 1e9,
                "peak": peak, "unit": "GB/s", "traffic": None}
    dec_roof["frac"] = dec_roof["achieved"] / peak
    tr = ncu_traffic("decode", rows)
    if tr:
        dec_roof["traffic"] = tr["bytes"]
    try:
        import oracle
        oracle.build()
        cpu = cpu_baseline(args, gen)
        cpu.pop("ops", None)
    except Exception as e:  # the bench must still print its line
        cpu = {"value": None, "unit": UNIT, "cores": host_cores(), "kind": "port", "sample": f"failed: {e}"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic",
        "config": {"workload": workload_text(args, n_docs, "; import -> state JSON" + ("" if args.no_export else " -> re-export(all_updates)")),
                   "name": args.config,
                   "docs_per_gpu": n_docs, "distinct_docs_per_gpu": distinct, "atom_ops_per_step_per_gpu": atoms_per_step,
                   "op_rows_per_gpu": rows, "blob_bytes_per_gpu": int(lens.sum()), "l2": "inputs_larger_than_L2" if lens.sum() > 126e6 else "inputs fit L2",
                   "generator_seconds": round(gen_s, 1), "host_cores": host_cores(), "numa_bound": bool(numa_bound),
                   "device_table_bytes_per_step": int(tm["device_bytes"])},
        "phases_ms": {k: v / n_steps for k, v in phase.items()}, "wall_ms_per_step": wall_ms / n_steps,
        "roofline": roof, "decode_roofline": dec_roof, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": launches, "clocks": clocks,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
