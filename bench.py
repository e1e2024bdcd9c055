#!/usr/bin/env python
"""Benchmark of the GFKB fingerprint-match path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path, same metric
    python bench.py ... --dump-outputs DIR                    # also save the last timed step's results as .npy

Workload (config.workload): BASELINE.json configs[2], the one the metric is quoted on -- a 10M-entry
GFKB of synthetic failures.jsonl-shaped ``signature_text`` rows, a 100k-query batch, the reference's
TF-IDF(1,2-gram) cosine with fused top-k=16.  A *step* is one pass of the whole query batch over the
whole GFKB.  With N > 1 GPUs the 10M rows are sharded over the ranks (strong scaling, total work
fixed): per-shard scan -> one all-gather of partial top-k -> merge.

``value``: queries/s with the index AND the prepared query batch resident in HBM (device work only:
scan + merge [+ all-gather + merge]); ``e2e``: queries/s through the public API from host text
buffers (host featurisation, host->device copies, kernels, device->host read of the result).
Only the ``cpu_baseline`` / ``--impl reference`` legs execute anything under oracle/.

``--dump-outputs DIR`` writes what the last timed step returned: ``scores.npy`` (float32 [Q, k]) and ``rows.npy``
(global row ids as float64 [Q, k], -1 = no row).  The inputs are generated from fixed seeds, so two builds run with
the same arguments can be compared output for output.  Past 64 MB a fixed, seeded sample of the queries is written,
and ``query_index.npy`` (float64) lists the sampled queries.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from untouched

METRIC = "fingerprint-match queries/sec over 10M-entry GFKB"
UNIT = "queries/s"
DUMP_LIMIT_BYTES = 64 << 20


def _count(minimum):
    def parse(s):
        v = int(s)
        if v < minimum:
            raise argparse.ArgumentTypeError(f"must be >= {minimum}, got {v}")
        return v
    return parse


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_count(1), default=3, help="timed steps (resident path; also the end-to-end calls unless --e2e-steps is given)")
    ap.add_argument("--warmup", type=_count(0), default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--queries", type=int, default=100_000)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--e2e-steps", type=_count(1), default=None, help="timed end-to-end calls from host text (default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's top-k (scores.npy float32, rows.npy float64) to DIR")
    ap.add_argument("--cpu-sample-rows", type=int, default=50_000)
    ap.add_argument("--cpu-sample-queries", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary kernels (dense / Jaccard / hash / K1a) of the 1-GPU run")
    ap.add_argument("--shard", default="rows", choices=["rows", "queries", "rows-text"],
                    help="rows: corpus rows sharded over the GPUs by row index (BASELINE configs[2]); rows-text: sharded by ranges of "
                         "the global text order (tighter chunks per shard); queries: index replicated, queries split")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs saves the top-k of the CUDA path; the reference arm computes no top-k")
    if a.e2e_steps is None:
        a.e2e_steps = a.steps
    return a


def dump_outputs(out_dir, scores, rows):
    """scores float32 [Q, k], rows int64 [Q, k] -> DIR/scores.npy, DIR/rows.npy (float64: row ids < 2^53 are exact).
    Above DUMP_LIMIT_BYTES a seeded sample of the queries (in query order) is kept and listed in query_index.npy."""
    import numpy as np

    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    q, k = scores.shape
    per_query = k * (4 + 8)
    budget = DUMP_LIMIT_BYTES - 4096          # room for the .npy headers
    if q * per_query > budget:
        keep = np.sort(np.random.default_rng(0).choice(q, budget // (per_query + 8), replace=False))
        scores, rows = scores[keep], rows[keep]
        np.save(out / "query_index.npy", keep.astype(np.float64))
    np.save(out / "scores.npy", np.ascontiguousarray(scores, dtype=np.float32))
    np.save(out / "rows.npy", np.ascontiguousarray(rows, dtype=np.float64))


def workload_config(a, world):
    return {
        "workload": "BASELINE configs[2]: %d-entry GFKB (synthetic failures.jsonl-shaped signature_text rows, seed 0xC0FFEE), "
                    "%d-query batch (seed 0xFACADE, ~50%% exact repeats of stored rows), TF-IDF(1,2-gram) cosine, fused top-k=%d"
                    % (a.rows, a.queries, a.k),
        "rows": a.rows, "queries": a.queries, "k": a.k,
        "parallelism": ("corpus rows sharded over %d GPU(s); queries replicated; pruning bounds pushed to peer GPUs over NVLink during the scan; 1 all-gather of partial top-k" % world)
                       if getattr(a, "shard", "rows").startswith("rows") else
                       ("index replicated on %d GPU(s); query batch split; 1 all-gather of the results" % world),
        "l2": "inputs larger than L2 (column blocks + dense bound matrix >> 126 MB); no explicit flush",
    }


# --------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU path (sklearn, literal restatement in oracle/)
# --------------------------------------------------------------------------------------------
_SAMPLE = {}


def _ref_one(qtext):
    from oracle import tfidf_oracle as O
    t = time.perf_counter()
    O.score_sklearn(qtext, _SAMPLE["corpus"])
    return time.perf_counter() - t


def _standalone_synth(seed, count, dup_of_seed=0, dup_rows=0):
    """Synthetic rows from oracle/_build/libkvsynth.so (the generator alone, g++-built by __graft_entry__.build()):
    the reference arm creates its inputs without loading the product's CUDA library."""
    import ctypes as C

    import numpy as np

    so = ROOT / "oracle" / "_build" / "libkvsynth.so"
    if so.exists():
        lib = C.CDLL(str(so))
    else:   # not built: compile into a temporary directory, never into the tree
        import tempfile

        with tempfile.TemporaryDirectory(prefix="kvsynth-") as tmp:
            so = Path(tmp) / "libkvsynth.so"
            subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", str(ROOT / "oracle" / "synth_shim.cpp"),
                            "-o", str(so)], check=True)
            lib = C.CDLL(str(so))
    lib.kv_synth_signatures.restype = C.c_int
    lib.kv_synth_signatures.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_uint64, C.c_int64, C.c_char_p, C.c_int64,
                                        C.POINTER(C.c_int64)]
    off = np.zeros(count + 1, dtype=np.int64)
    cap = max(1, count * 320)
    buf = C.create_string_buffer(cap)
    rc = lib.kv_synth_signatures(seed, 0, count, dup_of_seed, dup_rows, buf, cap, off.ctypes.data_as(C.POINTER(C.c_int64)))
    assert rc == 0, "kv_synth_signatures failed"
    raw = buf.raw
    return [raw[off[i]:off[i + 1]].decode("ascii") for i in range(count)]


def cpu_reference_rate(a, n_queries, procs, standalone=False):
    """Queries/s of the reference path on this box's host cores, scaled to the a.rows-entry GFKB.

    Sample: n_queries queries scored (SimilarityEngine.score semantics: TF-IDF refit per query) against
    the first a.cpu_sample_rows rows; the reference is Theta(N) per query (SURVEY section 6), so the rate
    on the full GFKB is rate_sample * sample_rows / rows.  `procs` worker processes run queries in
    parallel (the reference itself is single-threaded Python)."""
    import multiprocessing as mp

    rows = min(a.cpu_sample_rows, a.rows)
    if standalone:
        _SAMPLE["corpus"] = _standalone_synth(0xC0FFEE, rows)
        qs = _standalone_synth(0xFACADE, n_queries, 0xC0FFEE, a.rows)
    else:
        from kakveda_b200 import synth

        _SAMPLE["corpus"] = synth.corpus(rows)
        qs = synth.queries(n_queries, a.rows)
    from oracle import tfidf_oracle as O
    O.score_sklearn(qs[0], _SAMPLE["corpus"][:64])  # import scikit-learn / page it in before the clock starts
    t0 = time.perf_counter()
    if procs > 1:
        with mp.get_context("fork").Pool(procs) as pool:
            per = pool.map(_ref_one, qs)
    else:
        per = [_ref_one(q) for q in qs]
    wall = time.perf_counter() - t0
    rate_sample = len(qs) / wall
    return {"value": rate_sample * rows / a.rows, "wall_s": wall, "per_query_s_on_sample": sum(per) / len(per),
            "sample_rows": rows, "sample_queries": len(qs), "procs": procs}


def cpu_fixed_idf_rate(a, n_queries=256, k=16):
    """The "fair" CPU baseline of SURVEY section 8(d): scikit-learn fitted ONCE on a corpus sample, then one sparse
    product X_q @ X_c^T and a top-k per query batch -- what a CPU service would do if it stopped refitting per query.
    NOT parity with the reference (fixed idf instead of the query-inclusive refit); timed on one core, scaled by
    sample_rows / rows like the reference baseline.  Only the per-batch work is timed (transform + product + top-k)."""
    import numpy as np
    from sklearn.feature_extraction.text import TfidfVectorizer

    from kakveda_b200 import synth

    rows = min(a.cpu_sample_rows, a.rows)
    corpus = synth.corpus(rows)
    qs = synth.queries(n_queries, a.rows)
    vec = TfidfVectorizer(ngram_range=(1, 2), min_df=1)
    xc = vec.fit_transform(corpus)          # l2-normalised rows: the product is the cosine
    xct = xc.T.tocsr()
    t0 = time.perf_counter()
    xq = vec.transform(qs)
    scores = (xq @ xct).toarray()
    kk = min(k, rows)
    idx = np.argpartition(-scores, kk - 1, axis=1)[:, :kk]
    part = np.take_along_axis(scores, idx, axis=1)
    order = np.lexsort((idx, -part), axis=1)
    top = np.take_along_axis(idx, order, axis=1)
    wall = time.perf_counter() - t0
    return {"value": n_queries / wall * rows / a.rows, "unit": UNIT, "cores": 1, "wall_s": wall, "checksum": int(top.sum()),
            "sample": "%d queries x first %d rows: TfidfVectorizer fitted once on the sample, X_q @ X_c^T (scipy CSR) + top-%d; "
                      "fixed idf -- not the reference's per-query refit, no parity claim; rate scaled by %d/%d rows"
                      % (n_queries, rows, kk, rows, a.rows)}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    per_step = max(procs, a.cpu_sample_queries)
    for _ in range(max(0, min(a.warmup, 1))):
        cpu_reference_rate(a, procs, procs, standalone=True)
    t0 = time.perf_counter()
    vals = [cpu_reference_rate(a, per_step, procs, standalone=True) for _ in range(max(1, a.steps))]
    total = time.perf_counter() - t0
    v = sum(x["value"] for x in vals) / len(vals)
    sample = ("%d queries x first %d rows per step with sklearn TfidfVectorizer refit per query "
              "(similarity.py:14-20 restated in oracle/tfidf_oracle.py), %d worker processes; rate scaled by %d/%d rows"
              % (per_step, vals[0]["sample_rows"], procs, vals[0]["sample_rows"], a.rows))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * total / max(1, a.steps), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(a, a.gpus),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": procs, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------------
def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist

    from kakveda_b200 import synth
    from kakveda_b200.dist import ShardedGfkb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    real_stdout = os.dup(1)   # the ONE JSON line goes here; everything else (NCCL's version banner ...) to stderr
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"   # the version banner goes to stdout, where the driver expects ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    log = (lambda *s: print(*s, file=sys.stderr, flush=True)) if rank == 0 else (lambda *s: None)
    cores = os.cpu_count() or 1
    threads = max(1, cores // world)
    os.environ.setdefault("KAKVEDA_B200_THREADS", str(min(64, threads)))  # host sort / stream build inside the library

    # ---- build (excluded from the timed region, reported in config) ----
    t0 = time.perf_counter()
    buf, off = synth.signatures_packed(synth.CORPUS_SEED, 0, a.rows)
    t_gen = time.perf_counter() - t0
    shard = ShardedGfkb(device=local, rank=rank, world=world, mode=a.shard.split("-")[0],
                        order="text" if a.shard.endswith("-text") else "index")
    t0 = time.perf_counter()
    shard.build_packed(buf, off, 0, n_threads=threads)
    t_build = time.perf_counter() - t0
    del buf, off
    lay = shard.index.layout()
    log(f"[bench] rows={a.rows} gen {t_gen:.1f}s build {t_build:.1f}s vocab={len(shard.vocab)} layout={lay}")

    qbuf, qoff = synth.signatures_packed(synth.QUERY_SEED, 0, a.queries, dup_of_seed=synth.CORPUS_SEED, dup_rows=a.rows)
    qfb = shard.vocab.featurize_packed(qbuf, qoff, 0, grow=False, n_threads=threads)
    shard.set_resident(qfb)   # inputs resident in HBM before the timed region

    # ---- guard: the bound kernel's compile-time-specialised instantiation must return what the generic one returns ----
    # Pruning is exact, so both must give bit-identical results on this very batch; if they do not, the specialised one is
    # NOT used for this run and the line says so (the in-run float64 parity check below stays the final gate either way).
    if os.environ.get("KAKVEDA_B200_GENERIC_BOUND"):
        bound_variant = "generic (KAKVEDA_B200_GENERIC_BOUND set)"
    else:
        s_f, r_f = shard.topk_resident(a.k)
        os.environ["KAKVEDA_B200_GENERIC_BOUND"] = "1"
        s_g, r_g = shard.topk_resident(a.k)
        same = bool(torch.equal(r_f, r_g)) and bool(torch.equal(s_f, s_g))
        if max_over_ranks(0.0 if same else 1.0) > 0:
            bound_variant = "generic (the specialised instantiation returned different results on this batch and is NOT used)"
            log("[bench] WARNING: specialised bound kernel disagrees with the generic one; timing the generic one")
        else:
            del os.environ["KAKVEDA_B200_GENERIC_BOUND"]
            bound_variant = "specialised (results bit-identical to the generic instantiation on this batch)"
        del s_f, r_f, s_g, r_g

    # ---- device-resident timing: W warm-up + K timed steps ----
    scan_ms, merge_ms, kern_ms, exch_ms = [], [], [], []
    for _ in range(a.warmup):
        shard.topk_resident(a.k)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        s, r = shard.topk_resident(a.k)
        ms = shard.index.last_timing_ms()
        scan_ms.append(ms[1]); merge_ms.append(ms[2])
        kern_ms.append(shard.index.last_kernel_ms())
        exch_ms.append(getattr(shard, "last_exchange_ms", (0.0, 0.0, 0.0)))
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    step_ms = max_over_ranks(e0.elapsed_time(e1) / a.steps)
    lay = shard.index.layout()
    checksum = int(r.sum().item()) if r.numel() else 0
    kavg = [sum(x[i] for x in kern_ms) / len(kern_ms) for i in range(5)]   # bound0, seed scan, bound1, scan, merge
    local_kernels_ms = sum(kavg)
    # per-rank attribution of a step (max/min over ranks): own kernels, all-gather, global merge
    kmax, kmin = max_over_ranks(local_kernels_ms), -max_over_ranks(-local_kernels_ms)
    gather_ms = max_over_ranks(sum(x[0] for x in exch_ms) / len(exch_ms))
    gmerge_ms = max_over_ranks(sum(x[1] for x in exch_ms) / len(exch_ms))
    thr_exch_ms = max_over_ranks(sum(x[2] for x in exch_ms) / len(exch_ms))

    # ---- parity inside the bench run: sampled queries of THIS batch re-scored by the float64 full scan (K1a) ----
    # For 64 sampled queries every rank checks, on its own rows: (a) each returned (score, row) pair it owns agrees with
    # the float64 score at rtol 1e-5, (b) no row of its shard outside the returned set beats the returned k-th score.
    n_check = min(64, a.queries)
    ok_pairs = bad = 0
    s_h, r_h = s.cpu().numpy(), r.cpu().numpy()
    if a.dump_outputs and rank == 0:   # every rank holds the same merged result
        dump_outputs(a.dump_outputs, s_h, r_h)
    row_map = shard.row_map.cpu().numpy() if getattr(shard, "row_map", None) is not None else None
    base = shard.index.row_base if hasattr(shard.index, "row_base") else 0
    for qi in np.linspace(0, a.queries - 1, n_check).astype(np.int64):
        a0, a1 = int(qfb.indptr[qi]), int(qfb.indptr[qi + 1])
        sc = shard.index.score_features(qfb.ids[a0:a1], qfb.tf[a0:a1], float(qfb.oov[qi]))
        gids = row_map if row_map is not None else (np.arange(len(sc), dtype=np.int64) + base)
        pos = {int(g): i for i, g in enumerate(r_h[qi]) if g >= 0}
        mine = np.nonzero(np.isin(gids, np.fromiter(pos.keys(), dtype=np.int64, count=len(pos))))[0]
        for li in mine:
            want, got = sc[li], float(s_h[qi, pos[int(gids[li])]])
            if abs(want - got) <= 1e-5 * abs(want) + 1e-7:
                ok_pairs += 1
            else:
                bad += 1
        rest = sc.copy()
        rest[mine] = -1.0
        kth = float(s_h[qi, a.k - 1]) if r_h[qi, a.k - 1] >= 0 else -1.0
        if rest.size and rest.max() > kth * (1 + 1e-5) + 1e-7:
            bad += 1
    bad_total = int(max_over_ranks(float(bad)))
    ok_total = ok_pairs
    if world > 1:
        t = torch.tensor([ok_pairs], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        ok_total = int(t.item())
    assert bad_total == 0, f"in-run parity check failed on {bad_total} item(s)"

    # ---- end to end from host text ----
    e2e_steps = a.e2e_steps
    for _ in range(2):  # warm-up (staging and read-back buffers of both parities get pinned here, not in the timed calls)
        shard.topk_packed(qbuf, qoff, a.k)
    barrier()
    t0 = time.perf_counter()
    e2e_calls = []
    for _ in range(e2e_steps):
        tc = time.perf_counter()
        es, er = shard.topk_packed(qbuf, qoff, a.k)
        e2e_calls.append(round((time.perf_counter() - tc) * 1e3, 2))
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / e2e_steps)
    h2d = shard.index.layout()["last_upload_bytes"]
    d2h = a.queries * a.k * 12
    split = getattr(shard, "last_prepare_split_ms", None)
    if world > 1 and split:      # sliced preparation: the rank's slice goes up, the gathered slices come back, the batch goes up
        h2d += split["slice_bytes"]
        d2h += split["slice_bytes"] * world
    assert int(er.sum()) == checksum, "end-to-end result differs from the resident-path result"

    # ---- roofline of the path, SURVEY section 8(d) accounting ----
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    rows_local = lay["rows"]
    bytes_per_row = (lay["block_bytes"] + lay["norm_bytes"] + lay["directory_bytes"]) / max(1, rows_local)
    tiles = lay["last_tiles"]
    names = ["tfidf_bound_kernel(pass 0: seeds)", "tfidf_scan_kernel(seeds)", "tfidf_bound_kernel(pass 1: candidate lists)",
             "tfidf_scan_kernel(candidates)", "merge_topk_kernel"]
    dom = max(range(5), key=lambda i: kavg[i])
    path_s = local_kernels_ms / 1e3
    compulsory = tiles * rows_local * bytes_per_row + lay["last_upload_bytes"] + a.queries * a.k * 12 * lay["last_splits"]
    achieved = compulsory / path_s / 1e9
    traffic = ncu_note = None
    try:  # dram bytes of exactly these launches, from the committed ncu capture (same workload only)
        tr = json.loads((ROOT / "profiles" / "r2_path_traffic.json").read_text())
        if (tr["rows"], tr["queries"], tr["k"], tr["n_gpus"]) == (a.rows, a.queries, a.k, world):
            traffic, ncu_note = tr["traffic_bytes_per_step"], tr.get("note")
    except Exception:
        pass
    pairs_all = a.queries * lay["chunks"]
    roofline = {
        "bound": "hbm", "kernel": "GFKB match path = " + " + ".join(names[:4]), "dominant_kernel": names[dom],
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
        "traffic_source": ("profiles/r2_path_traffic.json (ncu capture of this workload, committed; not re-measured in this run)" if traffic else None),
        "ncu_note": ncu_note,
        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
        "algorithmic_bytes_per_step": compulsory, "bytes_per_row": bytes_per_row,
        "query_tile": 128, "query_tiles": tiles, "partial_lists_per_query": lay["last_splits"],
        "chunks": lay["chunks"], "chunk_rows": 32,
        "kernel_ms": {"bound_pass0": kavg[0], "seed_scan": kavg[1], "bound_pass1": kavg[2], "candidate_scan": kavg[3], "merge": kavg[4],
                      "sum": local_kernels_ms},
        "dominant_kernel_frac": compulsory / (kavg[dom] / 1e3) / 1e9 / peak,
        "pairs_passed_bound_frac": lay["pairs_passed_bound"] / max(1, pairs_all),
        "pairs_scored_per_query": lay["pairs_scored"] / max(1, a.queries),
        "candidate_records": lay["records_written"], "pool_pages_used": lay["pool_pages_used"],
        "unbatched_rate_gbs": a.queries * rows_local * bytes_per_row / path_s / 1e9,
        "note": "algorithmic bytes = query_tiles x rows x bytes_per_row (SURVEY 8(d): each 128-query tile would stream every row "
                "once), divided by the SUM of the path's kernel times of one step (CUDA events on the launching stream, rank 0). "
                "The path does not stream: tensor-core chunk bounds (exact block-max pruning) leave ~0.1% of the (query, chunk) "
                "pairs to the exact scan, so measured DRAM traffic is far below the algorithmic bytes -- see DESIGN.md section 6",
    }
    rank_stats = {"kernels_ms_max": kmax, "kernels_ms_min": kmin, "seed_threshold_exchange_ms": thr_exch_ms, "all_gather_ms": gather_ms,
                  "global_merge_ms": gmerge_ms, "step_ms": step_ms, "unattributed_ms": step_ms - kmax - gather_ms - gmerge_ms - thr_exch_ms}
    parity = {"sampled_queries": int(n_check), "pairs_checked": int(ok_total), "failed": int(bad_total),
              "check": "returned (score,row) pairs vs float64 full scan (K1a) at rtol 1e-5 + no unreturned row of a shard beats the k-th score"}

    # ---- secondary kernels of the path (rank 0): the HBM-bound single-query scan and the hash match ----
    secondary = None
    if rank == 0 and world == 1 and not a.no_secondary:   # single-GPU runs only: keeps the multi-GPU scaling runs short
        from kakveda_b200 import HashIndex
        ix = shard.index
        sc_ms = []
        for i in range(4):
            a0, a1 = int(qfb.indptr[i]), int(qfb.indptr[i + 1])
            ix.score_features(qfb.ids[a0:a1], qfb.tf[a0:a1], float(qfb.oov[i]))
            sc_ms.append(ix.last_score_ms())
        sc_bytes = lay["block_bytes"] + lay["directory_bytes"] + rows_local * (8 + 4 + 8)
        sc_s = min(sc_ms[1:]) / 1e3
        rng = np.random.default_rng(11)
        n_hash = 64_000_000  # 512 MB of fingerprints: larger than L2
        hashes = rng.integers(0, 2**63, size=n_hash, dtype=np.uint64)
        hx = HashIndex(device=local)
        hx.add_hashes(hashes)
        hq = hashes[rng.integers(0, n_hash, size=4096)]
        hx.match_hashes(hq, 4)
        hms = []
        for _ in range(3):
            hx.match_hashes(hq, 4)
            hms.append(hx.last_timing()[0])
        hx.close()
        # K2: synthetic bf16 embeddings generated ON the device (random sign/mantissa, exponent 2^-7..2^0), 1M rows at a time
        from kakveda_b200 import DenseIndex
        dd = 768

        def dense_rows(count, seed):
            g = torch.Generator(device=dev).manual_seed(seed)
            raw = torch.randint(0, 2**16, (count, dd), generator=g, device=dev, dtype=torch.int32)
            bits = (raw & 0x807F) | ((120 + ((raw >> 7) & 7)) << 7)
            return torch.where(bits >= 32768, bits - 65536, bits).to(torch.int16).view(torch.bfloat16).contiguous()

        # (BASELINE configs[1]) 1M x 768, 10k queries, fused top-16
        dn, dq = 1_000_000, 10_000
        dxi = DenseIndex(dd, device=local)
        dxi.add_device(dense_rows(dn, 100))
        dxi.finalize()
        dqs = dense_rows(100_000, 999)
        dms = []
        for _ in range(3):
            dxi.topk_device(dqs[:dq], 16)
            dms.append(dxi.last_timing()[0])
        dsplits = dxi.last_timing()[1]
        # (BASELINE configs[3]) all-pairs on the same 1M rows: every row's 32 nearest OTHER rows (self excluded)
        ams = []
        for _ in range(2):
            ap_s, ap_r = dxi.selfjoin_topk(32, device_out=True)
            ams.append(dxi.last_timing()[0])
        assert not bool((ap_r == torch.arange(dn, device=dev)[:, None]).any())
        del ap_s, ap_r
        # (BASELINE configs[2] read as dense embeddings, 1-GPU variant) 10M x 768 (15.4 GB), 100k queries, fused top-16
        d10 = 10_000_000
        for i in range(1, d10 // dn):
            dxi.add_device(dense_rows(dn, 100 + i))
        dxi.finalize()
        d10ms = []
        for _ in range(2):
            dxi.topk_device(dqs, 16)
            d10ms.append(dxi.last_timing()[0])
        d10splits = dxi.last_timing()[1]
        dxi.close()
        del dqs
        torch.cuda.empty_cache()
        # K3 (BASELINE configs[4] shape at 1 GPU): token-set Jaccard, 1M rows x ~55 distinct tokens (64 Zipf draws over 2^20)
        from kakveda_b200 import JaccardIndex
        jn, jq, jv = 1_000_000, 2048, 1 << 20
        draws = np.minimum(rng.zipf(1.2, size=(jn + jq, 64)) - 1, jv - 1).astype(np.uint32)
        draws.sort(axis=1)
        keep = np.ones(draws.shape, dtype=bool)
        keep[:, 1:] = draws[:, 1:] != draws[:, :-1]
        jindptr = np.concatenate([[0], np.cumsum(keep.sum(axis=1))]).astype(np.int64)
        jids = draws[keep]
        del draws, keep
        jx = JaccardIndex(jv, device=local)
        jx.add_csr(jindptr[: jn + 1], jids[: jindptr[jn]])
        jx.finalize()
        qip = (jindptr[jn:] - jindptr[jn]).astype(np.int64)
        qid = jids[jindptr[jn]:]
        jms = []
        for _ in range(2):
            jx.topk_csr(qip, qid, 16)
            jms.append(jx.last_timing_ms()[1])
        jentries = int(jindptr[jn])
        jx.close()
        # CPU baselines of the extension classes (BASELINE.md section 3.2-3.3), on bounded samples, all host cores for the matmul
        t0 = time.perf_counter()
        cs_rows, cs_q = 200_000, 256
        cdense = torch.randn(cs_rows, dd, dtype=torch.float32)
        cq = torch.randn(cs_q, dd, dtype=torch.float32)
        t0 = time.perf_counter()
        sc_cpu = (cq @ cdense.T)
        torch.topk(sc_cpu, 16, dim=1)
        dense_cpu_s = time.perf_counter() - t0
        dense_cpu_qps_1m = cs_q / dense_cpu_s * cs_rows / dn      # Theta(N) per query: scaled to the 1M-row config
        del cdense, cq, sc_cpu
        jsets = [set(jids[jindptr[i]:jindptr[i + 1]].tolist()) for i in range(20_000)]
        jq_sets = [set(qid[qip[i]:qip[i + 1]].tolist()) for i in range(4)]
        t0 = time.perf_counter()
        for qs_ in jq_sets:
            sorted(((len(qs_ & r_) / max(1, len(qs_ | r_)), -i) for i, r_ in enumerate(jsets)), reverse=True)[:16]
        jac_cpu_s = time.perf_counter() - t0
        jac_cpu_qps_1m = len(jq_sets) / jac_cpu_s * len(jsets) / jn
        del jsets
        # BASELINE configs[0]: 1k-entry GFKB, 128 queries, the reference run IN FULL (128 sequential score() calls)
        from oracle import tfidf_oracle as O
        c1_corpus, c1_q = synth.corpus(1000), synth.queries(128, 1000)
        from kakveda_b200 import GfkbIndex
        c1 = GfkbIndex(device=local)
        c1.add_texts(c1_corpus)
        c1.finalize()
        c1.topk(c1_q, 16)
        t0 = time.perf_counter()
        c1_s, c1_r = c1.topk(c1_q, 16)
        c1_gpu_s = time.perf_counter() - t0
        t0 = time.perf_counter()
        c1_ref = np.array([O.score_sklearn(qq, c1_corpus) for qq in c1_q])
        c1_ref_s = time.perf_counter() - t0
        c1_ok = bool(np.allclose(c1_s, np.take_along_axis(c1_ref, c1_r, axis=1), rtol=1e-5, atol=1e-7))
        c1.close()
        dflops = 2.0 * dn * dq * dd
        tpeak = float(peaks.get("bf16_tflops", 1590.0))
        tsust = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
        secondary = {
            "k2_dense_cosine_1Mx768_10k_queries": {"kernel": "dense_topk_kernel", "ms": min(dms), "flops": dflops,
                                                   "achieved_tflops": dflops / (min(dms) / 1e3) / 1e12,
                                                   "frac_of_bf16_burst_peak": dflops / (min(dms) / 1e3) / 1e12 / tpeak,
                                                   "queries_per_s": dq / (min(dms) / 1e3), "row_splits": int(dsplits),
                                                   "note": "BASELINE configs[1]; tcgen05 cta_group::1 M128 N256 K16, 3-stage TMA ring, 8 epilogue warps, fused top-16; "
                                                           "synthetic bf16 embeddings (random sign/mantissa, exponent 2^-7..2^0); parity unpinned"},
            "k2_dense_cosine_10Mx768_100k_queries_1gpu": {"kernel": "dense_topk_kernel", "ms": min(d10ms), "flops": 2.0 * d10 * 100_000 * dd,
                                                          "achieved_tflops": 2.0 * d10 * 100_000 * dd / (min(d10ms) / 1e3) / 1e12,
                                                          "frac_of_bf16_sustained_peak": 2.0 * d10 * 100_000 * dd / (min(d10ms) / 1e3) / 1e12 / tsust,
                                                          "queries_per_s": 100_000 / (min(d10ms) / 1e3), "row_splits": int(d10splits),
                                                          "note": "BASELINE configs[2] read as 768-d bf16 embeddings (SURVEY 8(d) cfg3, 1-GPU variant): 10M rows = 15.4 GB resident, "
                                                                  "100k-query batch, fused top-16; kernel time only; parity unpinned"},
            "k2_dense_allpairs_1Mx1M_top32": {"kernel": "dense_topk_kernel (self-join, own row excluded)", "ms": min(ams),
                                              "flops": 2.0 * dn * dn * dd, "achieved_tflops": 2.0 * dn * dn * dd / (min(ams) / 1e3) / 1e12,
                                              "frac_of_bf16_sustained_peak": 2.0 * dn * dn * dd / (min(ams) / 1e3) / 1e12 / tsust,
                                              "rows_per_s": dn / (min(ams) / 1e3),
                                              "note": "BASELINE configs[3]: every row's 32 nearest other rows; full N x N (symmetry not exploited); parity unpinned"},
            "k3_jaccard_1M_sets_2048_queries": {"kernel": "jaccard_scan_kernel", "rows": jn, "queries": jq, "ms": min(jms),
                                                "queries_per_s": jq / (min(jms) / 1e3), "avg_tokens_per_row": jentries / jn,
                                                "bytes_per_row": 4.0 * jentries / jn + 4.0,
                                                "note": "K3 jaccard_scan_kernel (dense regime: one warp scores a chunk for the 32 queries of a scan group, byte-packed row counters); "
                                                        "random Zipf token sets have no text structure to prune on; bit-exact vs Python sets in tests; parity unpinned"},
            "cfg0_1k_x_128_reference_in_full": {"gpu_ms_host_text_to_result": c1_gpu_s * 1e3, "reference_ms_128_sequential_score_calls": c1_ref_s * 1e3,
                                                "speedup": c1_ref_s / c1_gpu_s, "top16_scores_match_reference_rtol_1e-5": c1_ok,
                                                "note": "BASELINE configs[0]; GPU time = GfkbIndex.topk() from host strings (featurise, upload, exhaustive scan, read back); "
                                                        "reference = oracle.score_sklearn (similarity.py:14-20) called once per query, 1 core"},
            "cpu_baselines_extension_classes": {
                "dense_fp32_matmul_topk": {"queries_per_s_at_1M_rows": dense_cpu_qps_1m, "sample": "%d queries x %d rows x 768 fp32 torch matmul + topk, all host cores; scaled by rows" % (cs_q, cs_rows),
                                           "cores": os.cpu_count()},
                "jaccard_python_sets": {"queries_per_s_at_1M_rows": jac_cpu_qps_1m, "sample": "4 queries x 20000 sets, Python set ops, 1 core; scaled by rows", "cores": 1}},
            "k1a_score_one_query": {"kernel": "tfidf_score_kernel", "rows": rows_local, "ms": sc_s * 1e3, "bytes": sc_bytes,
                                    "achieved_gbs": sc_bytes / sc_s / 1e9, "frac_of_hbm_peak": sc_bytes / sc_s / 1e9 / peak,
                                    "note": "drop-in SimilarityEngine.score path: float64 scores of every row for one query"},
            "k4_hash_match_4096_queries": {"kernel": "hash_scan_kernel", "rows": n_hash, "ms": min(hms),
                                           "bytes": n_hash * 8, "achieved_gbs": n_hash * 8 / (min(hms) / 1e3) / 1e9,
                                           "frac_of_hbm_peak": n_hash * 8 / (min(hms) / 1e3) / 1e9 / peak,
                                           "note": "8 B/row; random 64-bit fingerprints (parity unpinned)"},
        }

    # ---- secondary configs that need several GPUs (every rank takes part; short: a few seconds each) ----
    secondary_multi = None
    if world > 1 and not a.no_secondary:
        from kakveda_b200.dist import ShardedDense, ShardedJaccard, shard_bounds
        secondary_multi = {}
        tsust = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
        dd, d10, dq = 768, 10_000_000, 100_000

        def dense_rows(count, seed):
            g = torch.Generator(device=dev).manual_seed(seed)
            raw = torch.randint(0, 2**16, (count, dd), generator=g, device=dev, dtype=torch.int32)
            bits = (raw & 0x807F) | ((120 + ((raw >> 7) & 7)) << 7)
            return torch.where(bits >= 32768, bits - 65536, bits).to(torch.int16).view(torch.bfloat16).contiguous()

        # BASELINE configs[2] read as dense embeddings, AS SPECIFIED: 10M x 768 bf16 row-sharded, 100k queries, fused top-16
        lo, hi = shard_bounds(d10, world, rank)
        sd = ShardedDense(dd, device=local, rank=rank, world=world)
        sd.build(dense_rows(hi - lo, 100 + rank), d10)
        dqs = dense_rows(dq, 999)
        sd.topk(dqs, 16)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        ds_, dr_ = sd.topk(dqs, 16)
        ev1.record()
        barrier()
        dms = max_over_ranks(ev0.elapsed_time(ev1))
        kms = max_over_ranks(sd.index.last_timing()[0])
        secondary_multi["k2_dense_cosine_10Mx768_100k_queries_sharded"] = {
            "n_gpus": world, "ms_step_max_over_ranks": dms, "ms_kernel_max_over_ranks": kms, "flops": 2.0 * d10 * dq * dd,
            "achieved_tflops_whole_job": 2.0 * d10 * dq * dd / (dms / 1e3) / 1e12,
            "frac_of_bf16_sustained_peak_x_gpus": 2.0 * d10 * dq * dd / (dms / 1e3) / 1e12 / (tsust * world),
            "queries_per_s": dq / (dms / 1e3), "result_checksum": int(dr_.sum().item()),
            "note": "SURVEY 8(d) cfg3 as specified: rows sharded over the GPUs, queries replicated, K2 per shard, one all-gather of partial top-k + K5; "
                    "step = kernel + exchange + merge (CUDA events, max over ranks); parity unpinned"}
        sd.index.close()
        del sd, dqs, ds_, dr_
        torch.cuda.empty_cache()
        # BASELINE configs[4] AS SPECIFIED (4 GPUs): 5M token sets (Zipf ids over 2^20, ~64 tokens), Q = 10k, top-16
        if world == 4 or os.environ.get("KAKVEDA_BENCH_CFG5") == "1":
            jn, jq, jv, draws = 5_000_000, 10_000, 1 << 20, 112

            def token_sets(count, seed):   # Zipf-like ids by inverse-CDF sampling on the device, sorted + deduplicated per set
                g = torch.Generator(device=dev).manual_seed(seed)
                out_ip, out_ids = [np.zeros(1, dtype=np.int64)], []
                for b0 in range(0, count, 500_000):
                    nb = min(500_000, count - b0)
                    u = torch.rand((nb, draws), generator=g, device=dev, dtype=torch.float64)
                    ids_ = (u.pow(-10.0).floor() - 1).clamp_(0, jv - 1).to(torch.int64)   # P(id >= x) ~ x^-0.1: Zipf(1.1)
                    ids_, _ = ids_.sort(dim=1)
                    keep = torch.ones_like(ids_, dtype=torch.bool)
                    keep[:, 1:] = ids_[:, 1:] != ids_[:, :-1]
                    keep &= keep.cumsum(dim=1) <= 64          # sets are capped at 64 tokens (the scan's per-query table)
                    cnt = keep.sum(dim=1).cpu().numpy()
                    out_ids.append(ids_[keep].to(torch.int32).cpu().numpy().astype(np.uint32))
                    out_ip.append(out_ip[-1][-1] + np.cumsum(cnt))
                return np.concatenate(out_ip).astype(np.int64), np.concatenate(out_ids)

            lo, hi = shard_bounds(jn, world, rank)
            t0 = time.perf_counter()
            lip, lids = token_sets(hi - lo, 7000 + rank)
            qip_, qid_ = token_sets(jq, 424242)
            sj = ShardedJaccard(jv, device=local, rank=rank, world=world)
            sj.build_local_csr(lip, lids, jn)
            t_build = time.perf_counter() - t0
            sj.topk_csr(qip_, qid_, 16)
            barrier()
            t0 = time.perf_counter()
            js, jr, ji, ju = sj.topk_csr(qip_, qid_, 16)
            torch.cuda.synchronize()
            j_e2e = max_over_ranks(time.perf_counter() - t0)
            j_kernel = max_over_ranks(sj.index.last_timing_ms()[1])
            # bit-exact check: this rank's first 100k sets as their own index vs Python sets, 8 queries
            from kakveda_b200 import JaccardIndex
            sub_n = min(100_000, hi - lo)
            sub = JaccardIndex(jv, device=local)
            sub.add_csr(lip[: sub_n + 1], lids[: lip[sub_n]])
            sub.finalize()
            ss, sr, si, su = sub.topk_csr(qip_[:9], qid_[: qip_[8]], 16)
            sub.close()
            rsets = [set(lids[lip[i]:lip[i + 1]].tolist()) for i in range(sub_n)]
            exact = True
            for qi in range(8):
                qs_ = set(qid_[qip_[qi]:qip_[qi + 1]].tolist())
                ref = sorted(((len(qs_ & r_) / max(1, len(qs_ | r_)), -i) for i, r_ in enumerate(rsets)), reverse=True)[:16]
                exact &= [-i for _, i in ref] == sr[qi].tolist()
                exact &= all(len(qs_ & rsets[int(r_)]) == int(si[qi, j]) and len(qs_ | rsets[int(r_)]) == int(su[qi, j]) for j, r_ in enumerate(sr[qi]))
            exact_all = max_over_ranks(0.0 if exact else 1.0) == 0.0
            avg_tokens = float(lip[-1]) / (hi - lo)
            secondary_multi["k3_jaccard_5M_sets_10k_queries"] = {
                "n_gpus": world, "sets": jn, "queries": jq, "avg_tokens_per_set": avg_tokens, "ms_kernels_max_over_ranks": j_kernel,
                "ms_end_to_end_max_over_ranks": j_e2e * 1e3, "queries_per_s_kernels": jq / (j_kernel / 1e3), "queries_per_s_end_to_end": jq / j_e2e,
                "bit_exact_vs_python_sets_top16_of_100k_subsample": bool(exact_all), "shard_build_s": t_build,
                "result_checksum": int(jr.sum()),
                "note": "BASELINE configs[4] / SURVEY 8(d) cfg5: sets row-sharded, K3 dense-regime Jaccard kernel per shard (exact integer counts), "
                        "all-gather of partial top-k + K5, max-reduce of the (inter, union) integers; end to end = host CSR in, merged result on the host; "
                        "sets capped at 64 tokens; parity unpinned (oracle: Python sets)"}
            sj.index.close()

    cpu = None
    if rank == 0 and not a.no_cpu_baseline:
        c = cpu_reference_rate(a, a.cpu_sample_queries, 1)
        cpu = {"value": c["value"], "unit": UNIT, "cores": 1, "kind": "port",
               "sample": "%d queries x first %d rows, sklearn refit per query (oracle.score_sklearn = similarity.py:14-20), "
                         "%.1f s wall; rate scaled by %d/%d rows (reference is Theta(N) per query)"
                         % (c["sample_queries"], c["sample_rows"], c["wall_s"], c["sample_rows"], a.rows)}
        try:  # second, non-parity CPU figure (SURVEY 8(d)): never allowed to break the bench line
            cpu["fixed_idf_sparse_product"] = cpu_fixed_idf_rate(a)
        except Exception as e:  # pragma: no cover
            cpu["fixed_idf_sparse_product"] = {"unavailable": repr(e)}

    if rank == 0:
        cfg = workload_config(a, world)
        cfg.update({"threshold_peers": int(getattr(shard, "n_threshold_peers", 0)), "index_build_s": t_build, "corpus_generate_s": t_gen, "vocab": len(shard.vocab),
                    "universal_features_folded": lay["universal_features"], "host_threads_per_rank": threads,
                    "result_checksum": checksum, "bound_kernel_instantiation": bound_variant})
        line = {
            "metric": METRIC, "value": a.queries / (step_ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks,
            "e2e": {"value": a.queries / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "ms_per_step": e2e_s * 1e3, "rank0_split_ms": getattr(shard, "last_e2e_ms", None),
                    "rank0_ms_per_call": e2e_calls},
            "gpu_launches": int(lay["kernel_launches"] + (1 if world > 1 else 0)) * a.steps,
            "roofline": roofline, "rank_stats": rank_stats, "parity_in_run": parity, "cpu_baseline": cpu, "secondary": secondary, "secondary_multi_gpu": secondary_multi,
        }
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
