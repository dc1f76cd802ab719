#!/usr/bin/env python3
"""Benchmark of the MicrobeCensus hot path on B200: reads/s end-to-end AGS (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c4] [--impl ours|reference] [--dump-outputs DIR]

One step = one pass of the whole hot path over one batch of synthetic reads: read QC -> 6-frame
translation + SEG + seeding + ungapped X-drop -> gapped X-drop -> per-read classification -> per-family
sums (-> NCCL all-reduce for N > 1) -> weighted AGS estimate on the host.

workloads (BASELINE.json configs):  c3 (default, the configuration the metric is quoted on: "reads/sec end-to-end AGS
at 150 bp") = 150 bp paired FASTQ files with -q 5 -m 20 -u 5, 5M reads per GPU (R1 block then R2 block, as the reference
processes paired files one after the other); c2 = 2,000,000 synthetic 100 bp single-end reads, -l 100; c4 = 150 bp with
-d, 12.5M reads per GPU.  Per-GPU work is fixed (weak scaling): rank r owns its block of the deterministic stream
(microbecensus_b200/synth.py).

`value`  = reads/s with the reads resident in HBM when the clock starts (device path only);
`e2e`    = the same through the public host API: pinned host buffers -> libmcx (H2D inside) -> results on host;
`roofline` = the seed+ungapped kernel against measured HBM bandwidth (algorithmic bytes, DESIGN.md section 5);
`cpu_baseline` = the unmodified reference (baseline/_ref: its Python stages + rapsearch_Linux_2.15 -z <cores>)
on a bounded prefix of the same reads, or the CPU oracle port when the reference install is absent.

`--dump-outputs DIR` writes, after the timed steps, what the last step of each arm computed (device_*.npy, e2e_*.npy:
ags, agg_hits in family order, counts = SearchResult.counts_vector(), classified = best subject per read, hits = the
HSPs), so that two builds can be compared output for output on the same seeded reads.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED_DUPS = 20260104
# what the reference's auto_detect_quality_offset (mc.py:174-187) returns for Phred+33 files such as the synthetic FASTQ:
# it subtracts 32, not 33, and the drop-in does the same (run_pipeline detects it per file; the bench states it)
QUAL_OFFSET = 32

WORKLOADS = {
    "c2": dict(name="2M synthetic 100 bp single-end reads, -l 100", config_id=2, reads=2_000_000, L=100, fastq=False,
               qc=dict(min_quality=-5, mean_quality=-5, max_unknown=100)),
    "c3": dict(name="10M synthetic 150 bp paired-end reads with -q 5 -m 20 -u 5", config_id=3, reads=10_000_000, L=150,
               fastq=True, qc=dict(min_quality=5, mean_quality=20, max_unknown=5)),
    "c4": dict(name="100M synthetic 150 bp reads with -d (5 % exact + 1 % reverse-complement duplicates), 12.5M per GPU",
               config_id=4, reads=12_500_000, L=150, fastq=False, dups=True,
               qc=dict(min_quality=-5, mean_quality=-5, max_unknown=100)),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    p.add_argument("--reads-per-gpu", type=int, default=None)
    p.add_argument("--ref-sample", type=int, default=20000, help="reads per step of the CPU reference arm")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed step of each arm computed to DIR/<name>.npy (float64)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs records the GPU arm (--impl ours)")
    return a


# caps of the per-read and per-HSP arrays in a dump: 2 arms x (500k + 160k x 12) float64 values = 39 MB at most
DUMP_READS, DUMP_HITS, DUMP_SEED = 500_000, 160_000, 20260105


def outputs_of_step(eng, markers, ags, res, n_reads):
    """What a caller of one step receives (AGS, per-family sums, the counters) plus the per-read classification and
    the HSPs the step left in the context, as float64 arrays.  Reads and HSPs beyond the caps are a fixed, seeded
    sample of rows (the same rows for the same counts)."""
    import numpy as np

    def sample(a, cap):
        if len(a) <= cap:
            return a
        return a[np.sort(np.random.default_rng(DUMP_SEED).choice(len(a), cap, replace=False))]
    agg = res.agg_hits()
    return {"ags": np.array([ags], np.float64),
            "agg_hits": np.array([agg.get(f, 0.0) for f in markers.fam_names], np.float64),
            "counts": res.counts_vector().astype(np.float64),
            "classified": sample(eng.classified(n_reads), DUMP_READS).astype(np.float64),
            "hits": sample(eng.hits(), DUMP_HITS).astype(np.float64)}


def write_outputs(path, arms):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for arm, arrays in arms.items():
        for name, arr in arrays.items():
            np.save(os.path.join(path, "%s_%s.npy" % (arm, name)), arr)


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm = sorted(int(float(r[1])) for r in self.rows if r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------- CPU reference arm
LAST_M8 = None


def reference_available():
    ref = os.path.join(ROOT, "baseline", "_ref", "microbe_census")
    return all(os.path.exists(os.path.join(ref, p)) for p in ("microbe_census.py", "bin/rapsearch_Linux_2.15", "data/rapdb_2.15"))


def sample_batches(wl, sample_reads):
    """The bounded sample both arms see: the first reads of the workload stream, as the list of files the
    workload names (c3: R1 and R2 of the first sample_reads/2 pairs; otherwise one file)."""
    from microbecensus_b200 import synth
    if wl["config_id"] == 3:
        return list(synth.paired_reads(wl["config_id"], 0, sample_reads // 2, wl["L"]))
    return [synth.reads(wl["config_id"], 0, sample_reads, wl["L"], with_quals=wl["fastq"])]


def run_reference_once(batches, wl, threads, tmpdir):
    """The unmodified reference's hot path (mc.py:611-626) on the sample files: process_seqfile -> search_seqs
    (rapsearch child, -z threads) -> classify_reads -> aggregate_hits -> estimate.
    Returns (seconds, AGS, sampled, agg_hits, best_hits)."""
    import warnings
    warnings.filterwarnings("ignore")
    sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
    from microbe_census import microbe_census as mc
    from microbecensus_b200 import synth
    paths_in = []
    for k, batch in enumerate(batches):
        path = os.path.join(tmpdir, "sample_%d.%s" % (k + 1, "fq" if wl["fastq"] else "fa"))
        if not os.path.exists(path):
            (synth.write_fastq if wl["fastq"] else synth.write_fasta)(batch, path)
        paths_in.append(path)
    os.chmod(os.path.join(ROOT, "baseline", "_ref", "microbe_census", "bin", "rapsearch_Linux_2.15"), 0o755)
    args = {"seqfiles": paths_in, "verbose": False, "nreads": sum(b.n for b in batches), "threads": threads, "read_length": wl["L"]}
    args.update(wl["qc"])
    if wl.get("dups"):
        args["filter_dups"] = True
    t0 = time.perf_counter()
    paths = mc.get_relative_paths(args)
    mc.impute_missing_args(args)
    mc.process_seqfile(args, paths)
    mc.search_seqs(args, paths)
    best = mc.classify_reads(args, paths)
    agg = mc.aggregate_hits(args, paths, best)
    dt_before_cleanup = time.perf_counter() - t0
    global LAST_M8                      # the child's .m8 lines, kept for the parity block (read outside the timed span)
    try:
        LAST_M8 = [l.rstrip("\n") for l in open(paths["tempfile"] + ".m8") if l[0] != "#"]
    except OSError:
        LAST_M8 = None
    t1 = time.perf_counter()
    mc.clean_up(paths)
    ags = mc.estimate_average_genome_size(args, paths, agg)
    return dt_before_cleanup + (time.perf_counter() - t1), ags, args["sampled_reads"], agg, best


def run_oracle_port_once(batches, wl, threads, tmpdir):
    """CPU oracle port (oracle/oracle_cli, pthreads over reads) when the reference install is absent."""
    from microbecensus_b200 import synth
    from microbecensus_b200 import microbe_census as mcb
    import gzip
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "oracle_cli"], stdout=subprocess.DEVNULL)
    fa = os.path.join(tmpdir, "sample.fa")
    batch = mcb.concat_batches(batches)
    synth.write_fasta(batch, fa)
    db = os.path.join(tmpdir, "markers.mcxdb")
    if not os.path.exists(db):
        open(db, "wb").write(gzip.open(os.path.join(ROOT, "microbecensus_b200", "data", "markers.mcxdb.gz")).read())
    env = dict(os.environ, ORACLE_THREADS=str(threads))
    t0 = time.perf_counter()
    subprocess.check_call([os.path.join(ROOT, "oracle", "oracle_cli"), db, fa, str(wl["L"]), "16", "1", "49", os.path.join(tmpdir, "o.m8")],
                          env=env, stderr=subprocess.DEVNULL)
    return time.perf_counter() - t0, None, batch.n, None, None


def cpu_baseline(wl, sample_reads, steps=1, warmup=0):
    cores = os.cpu_count() or 1
    batches = sample_batches(wl, sample_reads)
    kind = "reference" if reference_available() else "port"
    fn = run_reference_once if kind == "reference" else run_oracle_port_once
    times, ags, sampled, agg, best = [], None, sample_reads, None, None
    with tempfile.TemporaryDirectory() as tmp:
        for i in range(warmup + steps):
            dt, ags, sampled, agg, best = fn(batches, wl, cores, tmp)
            if i >= warmup:
                times.append(dt)
    sec = sum(times) / len(times)
    files = "%d file%s" % (len(batches), "s (R1, R2)" if len(batches) == 2 else "")
    return {"value": sampled / sec, "unit": "reads/s", "cores": cores, "kind": kind,
            "sample": "first %d reads of the workload stream in %s; whole reference hot path (process_seqfile, rapsearch -z %d, "
                      "classify_reads, aggregate_hits, estimate)" % (sample_reads, files, cores) if kind == "reference" else
                      "first %d reads; CPU oracle port, %d pthreads" % (sample_reads, cores),
            "seconds_per_step": sec, "ags": ags, "sampled": sampled, "agg_hits": agg, "best_hits": best}


def parity_block(eng, markers, wl, sample_reads, cb):
    """SURVEY 8d "parity reported with every perf run": the GPU arm on the SAME bounded sample the reference arm just
    processed -- per-family agg_hits, per-read classification (discrepant sampled-read ids with the reason) and the AGS
    relative difference (bar: <= 1 %)."""
    import numpy as np
    from microbecensus_b200 import microbe_census as mcb
    L = wl["L"]
    batch = mcb.concat_batches(sample_batches(wl, sample_reads))
    eng.set_params(L, quality_offset=QUAL_OFFSET if wl["fastq"] else None, filter_dups=bool(wl.get("dups")), **wl["qc"])
    eng.push(batch)
    res = eng.search(-1)
    agg = res.agg_hits()
    ags = mcb.estimate_average_genome_size({"read_length": L, "sampled_reads": res.sampled_reads, "verbose": False}, None, agg)
    out = {"sample": "first %d reads of the workload stream (the reference arm's sample)" % sample_reads,
           "sampled_reads": {"gpu": res.sampled_reads, "reference": cb.get("sampled")},
           "ags": {"gpu": ags, "reference": cb.get("ags")}, "ags_rel_diff": None, "ags_within_1pct": None}
    if cb.get("ags"):
        out["ags_rel_diff"] = float(abs(ags - cb["ags"]) / cb["ags"])
        out["ags_within_1pct"] = bool(out["ags_rel_diff"] <= 0.01)
    ref_agg, ref_best = cb.get("agg_hits"), cb.get("best_hits")
    if ref_agg is not None:
        fams = sorted(set(agg) | set(ref_agg))
        diff = {f: [agg.get(f, 0.0), ref_agg.get(f, 0.0)] for f in fams
                if abs(agg.get(f, 0.0) - ref_agg.get(f, 0.0)) > 1e-9 * max(1.0, abs(ref_agg.get(f, 0.0)))}
        out["families_compared"] = len(fams)
        out["families_equal"] = len(fams) - len(diff)
        out["families_differing"] = diff          # family: [gpu, reference]
    if ref_best is not None:
        codes, _ = eng.qc_export(False)
        best = eng.classified(batch.n)
        rank = np.cumsum(codes == 0) - 1          # running index among the sampled reads = the reference's read ids
        ours = {int(rank[i]): (markers.fam_names[markers.fam[s]], int(s)) for i, s in enumerate(best) if s >= 0}
        theirs = {int(k): v for k, v in ref_best.items()}
        disc = []
        for rid in sorted(set(ours) | set(theirs)):
            if rid not in theirs:
                disc.append([rid, "gpu-only", ours[rid][0]])
            elif rid not in ours:
                disc.append([rid, "reference-only", theirs[rid][0]])
            elif ours[rid][0] != theirs[rid][0]:
                disc.append([rid, "family", ours[rid][0], theirs[rid][0]])
            else:
                slen = float(markers.subj_len[ours[rid][1]])
                t = theirs[rid]               # [fam, aln, aln/target_len, score]
                if abs(float(t[1]) / float(t[2]) - slen) > 0.5:
                    disc.append([rid, "tie: same family, equal-score subject of another length", ours[rid][0]])
        out["reads_classified"] = {"gpu": len(ours), "reference": len(theirs), "common": len(set(ours) & set(theirs))}
        out["discrepant_reads"] = disc[:50]
        out["n_discrepant_reads"] = len(disc)
    if LAST_M8 is not None:
        # alignment level (SURVEY 8d (i)): the lines RAPsearch2 wrote for the sample against the GPU's HSPs in the same
        # text layout -- all twelve fields (identity, lengths, coordinates, log E, bits) of every single-HSP line
        from microbecensus_b200.engine import format_m8
        hits = eng.hits()
        codes, _ = eng.qc_export(False)
        rank = np.cumsum(codes == 0) - 1
        names = {int(r): str(int(rank[r])) for r in np.unique(hits[:, 0])} if len(hits) else {}
        mine = set(format_m8(hits, markers, L, names))
        single = [l for l in LAST_M8 if len(l.split("\t")[10].split(".")[-1]) <= 2]      # two-decimal E-values; sum-statistics lines carry six
        found = sum(1 for l in single if l in mine)
        out["m8_lines"] = {"reference": len(LAST_M8), "reference_single_hsp": len(single), "reproduced_character_for_character": found,
                           "gpu": len(mine), "note": "reference lines not reproduced: pairs with several HSPs (sum-statistics E-values) and "
                                                     "reads at RAPsearch2's 500-line cap (DESIGN.md section 2 (b), (c))"}
    return out


# ---------------------------------------------------------------------------------------------- main
def main():
    a = parse()
    wl = WORKLOADS[a.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if a.impl == "reference":
        if rank != 0:
            return 0
        cb = cpu_baseline(wl, a.ref_sample, steps=a.steps, warmup=min(a.warmup, 1))
        line = {"impl": "reference", "metric": "reads/sec end-to-end AGS", "value": cb["value"], "unit": "reads/s",
                "n_gpus": a.gpus, "steps": a.steps, "warmup": min(a.warmup, 1), "ms_per_step": 1e3 * cb["seconds_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                "config": {"workload": wl["name"], "sample_reads_per_step": a.ref_sample, "read_length": wl["L"]},
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "ags": cb["ags"], "sampled_reads": cb["sampled"]}
        print(json.dumps(line))
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    from microbecensus_b200 import synth
    from microbecensus_b200.engine import MarkerSearch, ReadBatch
    from microbecensus_b200.markers import Markers
    from microbecensus_b200 import microbe_census as mcb

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the search has no CPU path")
    torch.cuda.set_device(local)
    numa_node = None
    if world > 1:                                # host buffers next to the GPU that reads them (first touch after binding)
        from microbecensus_b200.affinity import bind_to_gpu_numa_node
        numa_node = bind_to_gpu_numa_node(int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local]) if os.environ.get("CUDA_VISIBLE_DEVICES", "").replace(",", "").isdigit() else local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"            # keeps NCCL's version banner out of stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    n = a.reads_per_gpu or (wl["reads"] // 2 if a.workload == "c3" else wl["reads"])
    L = wl["L"]
    lo, hi = rank * n, (rank + 1) * n

    markers = Markers()
    eng = MarkerSearch(markers, local)
    eng.set_stream(torch.cuda.current_stream().cuda_stream)
    dups = bool(wl.get("dups"))
    eng.set_params(L, quality_offset=QUAL_OFFSET if wl["fastq"] else None, filter_dups=dups and world == 1, **wl["qc"])

    # ---- synthetic shard, generated on the host (untimed), staged in pinned memory
    if a.workload == "c3":
        r1, r2 = synth.paired_reads(wl["config_id"], lo // 2, lo // 2 + n // 2, L)
        batch = mcb.concat_batches([r1, r2])        # files are processed one after the other (mc.py:337)
    else:
        batch = synth.reads(wl["config_id"], lo, hi, L, with_quals=wl["fastq"])
    if dups:                                   # copies of earlier reads of the same shard, 1 in 6 reverse-complemented
        rng = np.random.default_rng(SEED_DUPS + rank)
        mat = batch.bases.reshape(n, L)
        comp = np.zeros(256, np.uint8); comp[[65, 67, 71, 84, 78]] = [84, 71, 67, 65, 78]
        idx = np.flatnonzero(rng.random(n) < 0.06)
        idx = idx[idx > 0]
        src = (rng.random(len(idx)) * idx).astype(np.int64)
        rc = rng.random(len(idx)) < 1.0 / 6.0
        mat[idx[~rc]] = mat[src[~rc]]
        mat[idx[rc]] = comp[mat[src[rc]][:, ::-1]]
    # the reads as they cross the ABI: 2-bit bases + mask bit-planes, lengths, quality bytes (include/mcx.h), in
    # page-locked host memory; and a copy of the same arrays resident in HBM for the device-only arm
    from microbecensus_b200.engine import PackedBatch
    host_batch = PackedBatch.from_batch(batch, pinned=True)
    ascii_bytes = batch.nbytes
    del batch
    as_dev = lambda arr: torch.from_numpy(arr.view(np.int32) if arr.dtype == np.uint32 else arr).to(dev)
    d_packed, d_lens = as_dev(host_batch.packed), as_dev(host_batch.lengths)
    d_quals = as_dev(host_batch.quals) if host_batch.quals is not None else None
    h2d_bytes = host_batch.nbytes
    fam_names = markers.fam_names

    def finish(res):
        """counts -> (all-reduce) -> agg_hits -> AGS, as run_pipeline does after the search"""
        if world > 1:
            v = torch.from_numpy(res.counts_vector()).to(dev)
            dist.all_reduce(v)
            res.load_counts_vector(v.cpu().numpy())
        args = {"read_length": L, "sampled_reads": res.sampled_reads, "verbose": False}
        return mcb.estimate_average_genome_size(args, None, res.agg_hits()), res

    from microbecensus_b200.distributed import sharded_search

    def finish_reduced(res):
        args = {"read_length": L, "sampled_reads": res.sampled_reads, "verbose": False}
        return mcb.estimate_average_genome_size(args, None, res.agg_hits()), res

    def push_dev():
        return eng.push_packed_device(d_packed.data_ptr(), int(d_packed.numel()), d_lens.data_ptr(),
                                      d_quals.data_ptr() if d_quals is not None else 0, host_batch.n_bases, n)

    def step_device():
        if dups:
            eng.dedup_reset()                  # every step is a run of its own: the duplicate filter starts empty
        if dups and world > 1:                 # -d needs the cross-rank exchange of fingerprints
            return finish_reduced(sharded_search(eng, None, lo, nreads=None, filter_dups=True, push=push_dev))
        push_dev()
        return finish(eng.search(-1))

    def step_e2e():
        if dups:
            eng.dedup_reset()
        if dups and world > 1:
            return finish_reduced(sharded_search(eng, host_batch, lo, nreads=None, filter_dups=True))
        eng.push(host_batch)
        return finish(eng.search(-1))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            out = fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stage = {}
        launches = 0
        e0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = fn()
            tm, nl = eng.timings()
            launches += nl
            for k, v in tm.items():
                stage[k] = stage.get(k, 0.0) + v
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        return ms / steps, wall / steps, {k: v / steps for k, v in stage.items()}, launches, out

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_dev, wall_dev, stage_dev, launches, (ags, res) = timed(step_device, a.steps, max(a.warmup, 3))
    clocks = sampler.stop() if sampler else None
    dump = {"device": outputs_of_step(eng, markers, ags, res, n)} if a.dump_outputs and rank == 0 else None
    ms_e2e, wall_e2e, stage_e2e, _, (ags2, res2) = timed(step_e2e, a.steps, 1)
    if dump is not None:
        dump["e2e"] = outputs_of_step(eng, markers, ags2, res2, n)
        write_outputs(a.dump_outputs, dump)
    # device events bracket only GPU work; the step also holds host work (counter read-back, AGS estimate),
    # so the step time is the larger of the two clocks
    t_dev = max(ms_dev / 1e3, wall_dev)
    t_e2e = max(ms_e2e / 1e3, wall_e2e)
    total_reads = res.sampled_reads            # all ranks (after the all-reduce)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm = peaks.get("hbm_gbs")
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if hbm else "fallback 6650 GB/s (B200_PROFILING.md)"
    hbm = hbm or 6650.0
    # ---- roofline of every kernel of the step (DESIGN.md section 5 states the formulas): ALGORITHMIC bytes per launch =
    # per-unit bytes x the units the launch worked on (reads, frames and the queue lengths the library counted), over
    # the kernel's own CUDA-event time inside the timed region.  `roofline` is the entry of the kernel with the
    # largest share of the step.
    per_gpu_reads = total_reads / world
    work = eng.search_counters()                                  # rank 0's last search
    m = [(L - o) // 3 for o in (0, 1, 2)]
    sum_m = 2 * sum(m)                                            # residues of the six frames of a read
    w9, w10 = 2 * sum(max(0, x - 8) for x in m), 2 * sum(max(0, x - 9) for x in m)    # 9- and 10-letter windows per read
    G = (L + 31) // 32
    nwr = max(1, ((L + 2) // 3 - 12 + 1 + 31) // 32)
    R = per_gpu_reads
    algo = {
        "k_frames": R * (12 * G + 12 + sum_m),                                        # packed record, length, offset in; six rows out
        "k_seg": work["seg_frames"] * (2 * sum_m / 6.0 + 8 * nwr + 4),               # row in and out, its two window masks, queue entry
        "k_probe": R * (sum_m + 16 * w9 + 8 * w10) + 12 * work["filter_passes"],      # rows in, one 16 B and one 8 B filter block per window, pass records out
        "k_resolve": work["filter_passes"] * (12 + 8) + work["candidates"] * (4 + 12),  # pass record + table slot in; posting in, candidate out
        "k_seed": work["candidates"] * (12 + 2 * 16 + 8) + work["seeds"] * 16,        # candidate, two 16-residue windows, subject offsets in; seed out
        "k_walk": work["seeds"] * 16 + work["ungapped_hsps"] * 16,                     # seed in, HSP out (the residues walked are L1 / L2 hits)
    }
    k_times = {"k_frames": stage_dev["frames"], "k_seg": stage_dev["seg"], "k_probe": stage_dev["k_probe"],
               "k_resolve": stage_dev["k_resolve"], "k_seed": stage_dev["k_seed"], "k_walk": stage_dev["k_walk"]}
    traffic = {}
    try:
        pj = json.load(open(os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")))
        traffic = {k: v * (per_gpu_reads / pj["reads"]) for k, v in pj["dram_bytes_per_launch"].items()}
        issue = pj.get("issue_active_pct", {})
    except Exception:
        pj, issue = None, {}
    what = {"k_frames": "translation of the six frames, SEG window verdicts",
            "k_seg": "SEG (Wootton-Federhen) of the frames with a low-entropy window, one warp per frame",
            "k_probe": "murphy10 seed-word presence filter: two filter blocks (L2) per window",
            "k_resolve": "word tables and posting lists of the words that passed the filter (HBM), first rejection test",
            "k_seed": "seed growth and acceptance from 16-residue windows",
            "k_walk": "ungapped X-drop walks"}
    kernels = []
    for k, ms_k in k_times.items():
        ach = algo[k] / (ms_k * 1e-3) / 1e9 if ms_k else None
        kernels.append({"kernel": k, "ms": ms_k, "share_of_step": ms_k / (t_dev * 1e3), "algorithmic_bytes": algo[k],
                        "achieved_gbs": ach, "frac_of_hbm": ach / hbm if ach else None, "dram_traffic_bytes": traffic.get(k),
                        "issue_active_pct_ncu": issue.get(k)})
    top = max(kernels, key=lambda r: r["ms"])
    l2_peak = eng.l2_peak()
    block_loads = R * (w9 + w10)
    roofline = {"bound": "hbm", "kernel": "%s (%s)" % (top["kernel"], what[top["kernel"]]),
                "achieved": top["achieved_gbs"], "peak": hbm, "unit": "GB/s", "frac": top["frac_of_hbm"], "traffic": top["dram_traffic_bytes"],
                "peak_source": peak_src, "algorithmic_bytes_per_read": top["algorithmic_bytes"] / R, "kernel_ms": top["ms"],
                "kernel_timing": "CUDA events around the kernel's launches on the library's stream (mcx_timings / mcx_timings_detail)",
                "kernel_share_of_step": top["share_of_step"],
                "issue_active_pct_ncu": top["issue_active_pct_ncu"],
                "note": "integer work bound by issue slots, not by bytes: the HBM fraction is small by construction; "
                        "issue_active_pct_ncu is the share of issue slots used under ncu (profiles/r02_ncu_summary.md)",
                "traffic_source": "profiles/r02_kernel_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum per launch at %d reads, scaled to this step)" % pj["reads"] if pj else None,
                "lookups": {"kernel": "k_probe", "filter_block_loads_per_read": w9 + w10, "block_loads_per_s": block_loads / (stage_dev["k_probe"] * 1e-3),
                            "bytes_per_lookup": "16 (exact word and wildcards 3 / 4) or 8 (wildcards 5 / 6): one 32-byte L2 sector either way",
                            "l2_random_loads_per_s_measured": l2_peak * 1e9,
                            "frac_of_l2_random_rate": block_loads / (stage_dev["k_probe"] * 1e-3) / (l2_peak * 1e9),
                            "note": "upper bound on the loads issued (windows with a stop codon or masked residue are skipped); the "
                                    "microbenchmark issues nothing but scattered 4-byte loads over the same filter"},
                "kernels": kernels}
    # K1 (the kernel SURVEY 8d calls HBM-bound): bytes per read of the survey's table -- 2-bit bases ceil(L/4) + mask
    # ceil(L/8), + L quality bytes when -q/-m are active, one verdict byte written -- over the k_qc launches alone
    k1_bytes = (L + 3) // 4 + (L + 7) // 8 + (L if wl["fastq"] else 0) + 1
    k1_ms = stage_dev.get("k_qc") or 0.0
    n_in = n                                   # reads pushed per GPU (k_qc sees all of them)
    roofline_k1 = {"bound": "hbm", "kernel": "k_qc (trim to -l, unknown-base, mean / minimum quality filters on the packed reads)",
                   "achieved": (n_in * k1_bytes / (k1_ms * 1e-3) / 1e9) if k1_ms else None, "peak": hbm, "unit": "GB/s",
                   "frac": (n_in * k1_bytes / (k1_ms * 1e-3) / 1e9 / hbm) if k1_ms else None, "algorithmic_bytes_per_read": k1_bytes,
                   "kernel_ms": k1_ms, "kernel_timing": "CUDA events around the k_qc launches (mcx_timings[10])",
                   "moved_bytes_per_read": 12 * ((L + 31) // 32) + (L if wl["fastq"] else 0) + 4 + 8 + (8 if wl["fastq"] else 0) + 1}
    gcups = res.gapped_cells / world / (stage_dev["gapped"] * 1e-3) / 1e9 if stage_dev.get("gapped") else None
    # SURVEY 8d: the DPX-bound cell rate = measured DPX issue rate / 3 DPX instructions per affine-gap cell
    dpx = eng.dpx_peak()
    gapped = {"gcups": gcups, "cells_per_step_per_gpu": res.gapped_cells / world, "stage_ms": stage_dev.get("gapped"),
              "dpx_ginstr_per_s": dpx, "dpx_bound_gcups": dpx / 3.0, "frac_of_dpx_bound": (gcups / (dpx / 3.0)) if gcups else None,
              "note": "X-drop extension (RAPsearch2 AlignGapped): k_gap_screen (all extensions until first gain or death, rows in shared memory, DPX viaddmax/vimax3) + k_gap_dp (complete DP of the gainers, direction nibbles) + k_gap_trace; cells = every DP cell once"}

    line = {"metric": "reads/sec end-to-end AGS", "value": total_reads / t_dev, "unit": "reads/s", "n_gpus": world,
            "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": t_dev * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": wl["name"], "reads_per_gpu": n, "read_length": L, "parallelism": "reads sharded x%d, marker index replicated" % world,
                       "l2": "inputs (%d MB per GPU) larger than L2, no flush needed" % (h2d_bytes >> 20),
                       "genome_pack": "%s (%d bp in %d contigs)" % (os.path.basename(synth.genome_pack_path()), len(synth.genome()[0]), len(synth.genome()[2])),
                       "input_layout": "2-bit bases + mask bit-planes (%d B/read), lengths, quality bytes; %d MB instead of %d MB of ASCII" % (
                           4 * 3 * ((L + 31) // 32), h2d_bytes >> 20, ascii_bytes >> 20), "rank0_numa_node": numa_node},
            "e2e": {"value": total_reads / t_e2e, "unit": "reads/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": int(res.counts_vector().nbytes), "ms_per_step": t_e2e * 1e3},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "roofline_k1": roofline_k1,
            "stages_ms": stage_dev, "stages_ms_e2e": stage_e2e,
            "exchange_ms": getattr(eng, "exchange_ms", None) if (dups and world > 1) else None,
            "gapped_gcups": gcups, "gapped": gapped, "ags": ags, "ags_e2e": ags2,
            "counts": {"sampled_reads": res.sampled_reads, "reads_with_hits": res.reads_with_hits,
                       "reads_classified": res.reads_classified, "n_hsp": res.n_hsp, "n_seed_hits": res.n_seed_hits,
                       "n_gapped": res.n_gapped, "gapped_cells": res.gapped_cells, "low_qual": res.low_qual, "dups": res.dups}}
    if world == 1 and not a.no_cpu_baseline:
        try:
            cb = cpu_baseline(wl, a.ref_sample)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            line["cpu_baseline"]["ags_on_sample"] = cb["ags"]
        except Exception as exc:      # the baseline is reporting only; never lose the GPU line over it
            cb = None
            line["cpu_baseline"] = {"value": None, "unit": "reads/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": str(exc)[:200]}
        if cb is not None:
            try:
                line["parity"] = parity_block(eng, markers, wl, a.ref_sample, cb)
            except Exception as exc:
                line["parity"] = {"error": str(exc)[:200]}
    print(json.dumps(line, default=lambda o: o.item() if hasattr(o, "item") else str(o)))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
