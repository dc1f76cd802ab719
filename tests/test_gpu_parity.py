"""CUDA path (through the libmcx C ABI) against the CPU oracle and the golden fixtures.  Needs a B200."""
import gzip
import os

import numpy as np
import pytest

import golden_io
from microbecensus_b200 import microbe_census as mcb, synth
from microbecensus_b200.engine import MarkerSearch, ReadBatch
from oracle_lib import MCX_ORDER

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng(markers):
    e = MarkerSearch(markers, 0)
    yield e
    e.close()


def gpu_vs_oracle(eng, oracle, markers, batch, L, quota=-1):
    eng.set_params(L)
    eng.push(batch)
    res = eng.search(quota)
    hits = eng.hits()
    oh, _ = oracle.search(batch, L, eng.min_report_raw)
    assert hits.shape == oh[:, MCX_ORDER].shape
    assert np.array_equal(hits, oh[:, MCX_ORDER])          # every reported HSP, every field: bit-exact
    oc = oracle.classify(oh, L, markers, batch.n)
    assert res.reads_classified == oc["classified"]
    assert np.array_equal(res.fam_hits, oc["fam_hits"])
    assert np.array_equal(res.fam_aln, oc["fam_aln"])
    assert np.array_equal(res.aln_by_len, oc["aln_by_len"])
    assert np.array_equal(eng.classified(batch.n), oc["best_subject"])
    assert res.n_hsp == len(oh)
    assert res.reads_with_hits == len(set(oh[:, 0].tolist()))
    return res


@pytest.mark.parametrize("fname,L", [("meta.fa.gz", 100), ("meta50.fa.gz", 50), ("long.fa.gz", 500), ("long.fa.gz", 250),
                                     ("long.fa.gz", 150), ("long.fa.gz", 60), ("long.fa.gz", 300), ("ties.fa.gz", 500)])
def test_golden_reads_bit_exact(eng, oracle, markers, fname, L):
    gpu_vs_oracle(eng, oracle, markers, ReadBatch.from_strings(golden_io.read_fasta(fname)), L)


@pytest.mark.parametrize("L,n", [(100, 20000), (150, 8000), (70, 8000), (400, 2000)])
def test_seeded_synthetic_reads_bit_exact(eng, oracle, markers, L, n):
    res = gpu_vs_oracle(eng, oracle, markers, synth.reads(7, 0, n, L), L)
    assert res.reads_classified > 0


def test_large_sample_bit_exact_at_the_metric_length(eng, oracle, markers):
    """200,000 reads of the bench workload's stream at 150 bp (ten times the largest sample above): every HSP, the
    classification of every read and the per-family sums against the oracle, which runs on all host cores (slices of the
    batch on threads; the C calls release the GIL and only read the index)."""
    import concurrent.futures as cf
    n, L = 200_000, 150
    batch = synth.reads(3, 0, n, L)
    eng.set_params(L)
    eng.push(batch)
    res = eng.search(-1)
    hits = eng.hits()
    oracle.search(batch.slice(0, 8), L, eng.min_report_raw)            # one-time table set-up before the threads start
    workers = max(1, min(32, os.cpu_count() or 1))
    cuts = np.linspace(0, n, 4 * workers + 1).astype(np.int64)

    def part(k):
        lo, hi = int(cuts[k]), int(cuts[k + 1])
        oh, _ = oracle.search(batch.slice(lo, hi), L, eng.min_report_raw, cap=400_000)
        oh[:, 0] += lo                                                 # read index within the whole batch
        return oh
    with cf.ThreadPoolExecutor(workers) as ex:
        oh = np.concatenate(list(ex.map(part, range(len(cuts) - 1))))
    assert hits.shape == oh[:, MCX_ORDER].shape
    assert np.array_equal(hits, oh[:, MCX_ORDER])
    oc = oracle.classify(oh, L, markers, n)
    assert res.reads_classified == oc["classified"] > 1000
    assert np.array_equal(res.fam_hits, oc["fam_hits"]) and np.array_equal(res.fam_aln, oc["fam_aln"])
    assert np.array_equal(res.aln_by_len, oc["aln_by_len"])
    assert np.array_equal(eng.classified(n), oc["best_subject"])


@pytest.mark.parametrize("n", [1, 2, 7, 33])
def test_small_batches_bit_exact(eng, oracle, markers, n):
    """Fewer gapped extensions than lanes of a warp: the work-list refill of k_gap_dir / k_seg with lanes that never get work."""
    seqs = golden_io.read_fasta("long.fa.gz")[:n]
    res = gpu_vs_oracle(eng, oracle, markers, ReadBatch.from_strings(seqs), 150)
    assert res.sampled_reads == n


def _full_state(eng, n):
    res = eng.search(-1)
    return res.counts_vector(), eng.hits(), eng.classified(n), eng.qc_export(False)[0]


def test_packed_push_equals_ascii_push(eng, markers, monkeypatch):
    """mcx_push_reads_packed (2-bit + mask bit-planes, the layout of the reads in HBM) against mcx_push_reads (ASCII,
    packed on the device by k_pack_ascii): same verdicts, HSPs, classification and sums -- FASTA and FASTQ with QC,
    fixed-length and ragged reads, reads with N and lower-case characters; then the same packed push cut into many copy
    steps and search chunks (the overlapped path of large inputs), from page-locked buffers."""
    from microbecensus_b200.engine import PackedBatch
    rng = np.random.default_rng(3)
    seqs = golden_io.read_fasta("long.fa.gz")[:1500]
    ragged = [s[:int(k)] for s, k in zip(seqs, rng.integers(100, 400, size=len(seqs)))]
    noisy = ["".join(("N" if u < 0.01 else c.lower() if u < 0.015 else c) for c, u in zip(s, rng.random(len(s)))) for s in ragged]
    quals = ["".join(chr(33 + int(q)) for q in np.clip(np.rint(rng.normal(30, 7, size=len(s))), 2, 41)) for s in noisy]
    for name, batch, kw in (("fasta", ReadBatch.from_strings(seqs), {}),
                            ("ragged", ReadBatch.from_strings(noisy), dict(max_unknown=1)),
                            ("fastq", ReadBatch.from_strings(noisy, quals), dict(quality_offset=33, min_quality=5, mean_quality=25, max_unknown=1))):
        eng.set_params(150, **kw)
        eng.push(batch)
        ref = _full_state(eng, batch.n)
        assert ref[0][0] > 0 and (name == "fasta" or 0 < ref[0][2] < batch.n)          # some reads fail QC, some pass
        for pinned in (False, True):
            eng.push(PackedBatch.from_batch(batch, pinned=pinned))
            got = _full_state(eng, batch.n)
            for a, b in zip(ref, got):
                assert np.array_equal(a, b), (name, pinned)
        monkeypatch.setenv("MCX_COPY_STEPS", "13")
        monkeypatch.setenv("MCX_CHUNK_READS", "100")
        eng.push(PackedBatch.from_batch(batch, pinned=True))
        got = _full_state(eng, batch.n)
        monkeypatch.delenv("MCX_COPY_STEPS"); monkeypatch.delenv("MCX_CHUNK_READS")
        for a, b in zip(ref, got):
            assert np.array_equal(a, b), (name, "chunked")
        for quota in (1, 137, 700):              # -n across chunk boundaries
            monkeypatch.setenv("MCX_CHUNK_READS", "100")
            eng.push(PackedBatch.from_batch(batch)); r1 = eng.search(quota)
            monkeypatch.delenv("MCX_CHUNK_READS")
            eng.push(batch); r2 = eng.search(quota)
            assert np.array_equal(r1.counts_vector(), r2.counts_vector()) and r1.sampled_reads == min(quota, ref[0][0])


def test_500_line_cap_runs(eng, oracle, markers):
    """Reads with more than 500 reportable subjects (RAPsearch2 -v 500): the cap kernel must actually run on the GPU and
    agree with the oracle."""
    seqs = golden_io.read_fasta("cap.fa.gz")
    res = gpu_vs_oracle(eng, oracle, markers, ReadBatch.from_strings(seqs), 100)
    assert res.n_capped_reads > 0


def test_classification_against_reference_golden(eng, markers):
    """GPU classification vs what the reference's classify_reads made of RAPsearch2's own output."""
    for fname, name, L in (("meta.fa.gz", "meta", 100), ("meta50.fa.gz", "meta50", 50)):
        batch = ReadBatch.from_strings(golden_io.read_fasta(fname))
        eng.set_params(L); eng.push(batch); eng.search(-1)
        best = eng.classified(batch.n)
        exp = golden_io.read_json("%s.L%d.json" % (name, L))
        ref_cls = {int(k): v["fam"] for k, v in exp["classified"].items()}
        ours = {int(i): markers.fam_names[markers.fam[s]] for i, s in enumerate(best) if s >= 0}
        assert set(ref_cls) == set(ours)
        assert all(ref_cls[k] == ours[k] for k in ours)


def test_qc_counters_match_reference_and_oracle(eng, oracle, markers):
    recs = golden_io.read_fastq("short.fq.gz")
    batch = ReadBatch.from_strings([r[1] for r in recs], [r[2] for r in recs])
    for case in golden_io.read_json("short.qc.json"):
        o = case["opts"]
        L = case["read_length"]
        eng.set_params(L, quality_offset=case["quality_offset"], min_quality=o.get("min_quality", -5),
                       mean_quality=o.get("mean_quality", -5), max_unknown=o.get("max_unknown", 100))
        eng.push(batch)
        res = eng.search(o.get("nreads", 1000000))
        assert (res.sampled_reads, res.too_short, res.low_qual, res.dups) == (case["sampled"], case["too_short"], case["low_qual"], 0), case
        sampled, code, cnt = oracle.process_reads(batch, L, case["quality_offset"], o.get("min_quality", -5), o.get("mean_quality", -5),
                                                  o.get("max_unknown", 100), o.get("nreads", 1000000))
        assert sampled == res.sampled_reads
        # the searched reads are exactly the oracle's kept reads: same HSPs on that subset
        kept = np.flatnonzero(code == 0)
        sub = ReadBatch.from_strings([recs[i][1] for i in kept])
        oh, _ = oracle.search(sub, L, eng.min_report_raw)
        hits = eng.hits()
        assert len(hits) == len(oh)
        assert np.array_equal(hits[:, 1:], oh[:, MCX_ORDER][:, 1:])
        assert np.array_equal(hits[:, 0], kept[oh[:, 0]])


def test_edge_cases(eng, oracle, markers):
    # empty input
    eng.set_params(100)
    eng.push(ReadBatch.from_strings([]))
    res = eng.search(-1)
    assert res.sampled_reads == 0 and res.n_hsp == 0 and res.reads_classified == 0
    # all too short / unknown bases / lower case / ragged lengths
    good = golden_io.read_fasta("meta.fa.gz")[:40]
    seqs = ["ACGT" * 10, "N" * 100, good[0].lower(), good[1][:50] + "N" + good[1][51:], good[2] + "ACGTACGT", good[3][:99]] + good[4:]
    batch = ReadBatch.from_strings(seqs)
    eng.push(batch)
    res = eng.search(-1)
    assert res.too_short == 2 and res.sampled_reads == len(seqs) - 2
    kept = [s for s in seqs if len(s) >= 100]
    oh, _ = oracle.search(ReadBatch.from_strings(kept), 100, eng.min_report_raw)
    assert res.n_hsp == len(oh)
    # max_unknown filter: the all-N read goes
    eng.set_params(100, max_unknown=10)
    eng.push(batch)
    assert eng.search(-1).low_qual == 1


def test_full_size_invariants(eng, markers):
    """BASELINE config 2 size (2M x 100 bp): size-independent properties instead of an oracle run --
    idempotence, additivity of the integer sums over a split of the reads (checksum of checksums), the -n quota
    equals a search of the prefix, and agreement of the host API with device-resident input."""
    import torch
    n, L = 2_000_000, 100
    batch = synth.reads(2, 0, n, L)
    eng.set_params(L)
    eng.push(batch)
    whole = eng.search(-1)
    again = eng.search(-1)
    assert np.array_equal(whole.counts_vector(), again.counts_vector())
    assert whole.sampled_reads == n and whole.reads_classified > 10000
    parts = []
    for lo, hi in ((0, 700_001), (700_001, n)):
        eng.push(batch.slice(lo, hi))
        parts.append(eng.search(-1).counts_vector())
    total = parts[0] + parts[1]
    assert np.array_equal(total, whole.counts_vector())
    eng.push(batch)
    q = eng.search(700_001)
    assert np.array_equal(q.counts_vector(), parts[0])
    d_b = torch.from_numpy(batch.bases).cuda(); d_o = torch.from_numpy(batch.offsets).cuda()
    eng.push_device(d_b.data_ptr(), 0, d_o.data_ptr(), n, d_b.numel())
    assert np.array_equal(eng.search(-1).counts_vector(), whole.counts_vector())
    ags = mcb.estimate_average_genome_size({"read_length": L, "sampled_reads": n, "verbose": False}, None, whole.agg_hits())
    assert 1.0e6 < ags < 4.0e6


def test_consecutive_device_pushes_of_growing_reads(eng, markers):
    """Device-resident pushes one after the other with a growing read length (the read-length sweep): every push must
    rebuild the record offsets.  (Regression: an error code left behind by cudaEventElapsedTime on a never-recorded event
    made CUB skip the offset scan of the NEXT push without a word; with equal lengths nobody noticed.)"""
    import torch
    n = 30000
    pool = synth.reads(5, 0, n, 120).bases.reshape(n, 120)
    d_pool = torch.from_numpy(pool).cuda()
    for L in (60, 70, 100, 50):
        eng.set_params(L)
        eng.push(ReadBatch(np.ascontiguousarray(pool[:, :L]).reshape(-1), np.arange(n + 1, dtype=np.int64) * L))
        want = eng.search(-1).counts_vector()
        d_b = d_pool[:, :L].contiguous()
        d_o = torch.arange(n + 1, dtype=torch.int64, device="cuda") * L
        torch.cuda.synchronize()
        for _ in range(2):
            eng.push_device(d_b.data_ptr(), 0, d_o.data_ptr(), n, n * L)
            assert np.array_equal(eng.search(-1).counts_vector(), want), L
    # and the same in the packed device layout
    from microbecensus_b200.engine import PackedBatch
    for L in (60, 70, 100):
        eng.set_params(L)
        hb = ReadBatch(np.ascontiguousarray(pool[:, :L]).reshape(-1), np.arange(n + 1, dtype=np.int64) * L)
        eng.push(hb)
        want = eng.search(-1).counts_vector()
        pb = PackedBatch.from_batch(hb)
        d_p = torch.from_numpy(pb.packed.view(np.int32)).cuda(); d_l = torch.from_numpy(pb.lengths.view(np.int32)).cuda()
        torch.cuda.synchronize()
        for _ in range(2):
            eng.push_packed_device(d_p.data_ptr(), int(d_p.numel()), d_l.data_ptr(), 0, pb.n_bases, n)
            assert np.array_equal(eng.search(-1).counts_vector(), want), L


FULL = os.path.join(golden_io.GOLD, "full")


def test_reference_accuracy_test_on_the_gpu_path(markers):
    """The reference's own integration test (tests/test_microbe_census.py:15-25) through the drop-in: run_pipeline on
    tests/data/metagenome.fa.gz with API defaults must land within 1 % of the true AGS of the simulated community
    (3,530,599.61) -- and within 1 % of what the unmodified reference computes on the same file (3,519,110.107,
    tests/golden/full/expected.json, written by tools/make_golden.py full), with its counters: 70,623 reads sampled, the
    same reads classified into the same families (one extra read at the 500-line cap)."""
    exp = golden_io.read_json(os.path.join("full", "expected.json"))["metagenome"]
    args = {"seqfiles": [os.path.join(FULL, "metagenome.fa.gz")]}
    est, out = mcb.run_pipeline(args)
    assert abs(est - 3530599.61) / 3530599.61 < 0.01                       # the reference's own assertion
    assert abs(est - exp["ags"]) / exp["ags"] < 0.01
    assert out["sampled_reads"] == exp["sampled_reads"] == 70623 and out["read_length"] == 100
    eng = mcb.get_engine(0)
    batch = mcb.load_reads(args["seqfiles"][0])
    eng.set_params(100); eng.push(batch); res = eng.search(-1)
    best = eng.classified(batch.n)
    ours = {str(i): markers.fam_names[markers.fam[s]] for i, s in enumerate(best) if s >= 0}
    ref = exp["classified"]
    assert set(ref) <= set(ours) and len(set(ours) - set(ref)) <= 1
    assert all(ours[k] == ref[k] for k in ref)
    # reads with hits: RAPsearch2 prints a few sub-floor sum-statistics lines the GPU path does not (DESIGN.md section 2)
    assert 0 <= exp["reads_with_hits"] - res.reads_with_hits <= 0.01 * exp["reads_with_hits"]
    assert res.n_capped_reads > 0
    # per-family sums: `hits` families identical up to the one extra read, others within the equal-score ties
    agg = res.agg_hits()
    cut = markers.cutoffs(100)
    for f, fam in enumerate(markers.fam_names):
        if int(cut[f]["stat"]) == 0:
            assert abs(agg.get(fam, 0.0) - exp["agg_hits"].get(fam, 0.0)) <= 1.0, fam
        else:
            assert abs(agg.get(fam, 0.0) - exp["agg_hits"].get(fam, 0.0)) <= 0.05 * max(exp["agg_hits"].get(fam, 0.0), 1.0), fam


def test_baseline_config_1_example_fastq(markers, tmp_path):
    """BASELINE.json config 1: microbe_census/example/example.fq.gz with the CLI defaults (-n 2000000), through the CLI
    mirror: offset 32 and 100 bp detected, 8,672 reads sampled, 32 reads classified into the reference's families,
    total_bases 980,306, AGS within 1 % of the reference's 3,051,745.76."""
    import subprocess, sys
    exp = golden_io.read_json(os.path.join("full", "expected.json"))["example_fq"]
    out = tmp_path / "report.txt"
    root = os.path.dirname(os.path.dirname(golden_io.GOLD))
    cp = subprocess.run([sys.executable, os.path.join(root, "scripts", "run_microbe_census.py"), "-v", os.path.join(FULL, "example.fq.gz"), str(out)],
                        capture_output=True, text=True, cwd=root)
    assert cp.returncode == 0, cp.stderr
    assert "\t1328 reads shorter than 100 bp and skipped" in cp.stdout
    assert "\t8672 reads sampled from seqfile" in cp.stdout
    assert "\t32 reads assigned to a marker protein" in cp.stdout
    rep = dict(l.rstrip("\n").split(":\t") for l in open(out) if ":\t" in l)
    assert rep["reads_sampled"] == "8672" and rep["trimmed_length"] == "100" and rep["total_bases"] == "980306"
    ags = float(rep["average_genome_size"])
    assert abs(ags - exp["ags"]) / exp["ags"] < 0.01
    assert abs(float(rep["genome_equivalents"]) - 980306 / ags) < 1e-9
    args = {"seqfiles": [os.path.join(FULL, "example.fq.gz")], "nreads": 2000000}
    est, o = mcb.run_pipeline(args)
    assert est == ags and o["quality_offset"] == 32
    for key, L in (("example_fa_150", 150), ("example_fa_500", 500)):
        e = golden_io.read_json(os.path.join("full", "expected.json"))[key]
        est, o = mcb.run_pipeline({"seqfiles": [os.path.join(FULL, "example.fa.gz")], "read_length": L})
        assert o["sampled_reads"] == e["sampled_reads"] == 2000
        assert abs(est - e["ags"]) / e["ags"] < 0.01


def test_run_pipeline_drop_in(eng, oracle, markers, tmp_path, capsys):
    """run_pipeline(args) on a FASTQ file: same args keys, verbose lines and AGS as the oracle-derived numbers."""
    recs = golden_io.read_fastq("short.fq.gz")
    path = os.path.join(os.path.dirname(golden_io.GOLD), "golden", "short.fq.gz")
    args = {"seqfiles": [path], "verbose": True, "nreads": 2000, "mean_quality": 25}
    est, out = mcb.run_pipeline(args)
    text = capsys.readouterr().out
    assert out["file_type"] == "fastq" and out["quality_offset"] == 32 and out["read_length"] == 100
    batch = ReadBatch.from_strings([r[1] for r in recs], [r[2] for r in recs])
    sampled, code, cnt = oracle.process_reads(batch, 100, 32, -5, 25, 100, 2000)
    assert out["sampled_reads"] == sampled
    assert "\t%d reads shorter than 100 bp and skipped" % cnt["too_short"] in text
    assert "\t%d low quality reads found and skipped" % cnt["low_qual"] in text
    sub = ReadBatch.from_strings([recs[i][1] for i in np.flatnonzero(code == 0)])
    oh, _ = oracle.search(sub, 100, mcb.get_engine(0).min_report_raw)
    oc = oracle.classify(oh, 100, markers, sub.n)
    assert "\t%d reads assigned to a marker protein" % oc["classified"] in text
    from microbecensus_b200.engine import SearchResult

    class Raw:
        pass
    raw = Raw()
    for k in ("too_short", "low_qual", "dups", "reads_with_hits", "n_hsp", "n_seed_hits", "n_gapped", "gapped_cells", "n_capped_reads"):
        setattr(raw, k, 0)
    raw.sampled_reads = sampled; raw.reads_classified = oc["classified"]
    raw.fam_hits = oc["fam_hits"]; raw.fam_aln = oc["fam_aln"]; raw.aln_by_len = oc["aln_by_len"].ravel()
    want = mcb.estimate_average_genome_size({"read_length": 100, "sampled_reads": sampled, "verbose": False}, None,
                                            SearchResult(raw, markers, 100).agg_hits())
    assert est == want
    out["outfile"] = str(tmp_path / "r.txt")
    mcb.report_results(out, est, mcb.count_bases(out))
    assert open(out["outfile"]).read().startswith("Parameters\nmetagenome:\t")


def test_duplicate_filter_matches_oracle(eng, oracle, markers):
    """-d on the device (fingerprint + sort + first-kept-wins) against the oracle's sequential set, with QC and -n"""
    from test_host import dup_batch
    seqs, quals = dup_batch(n=20000, seed=11)
    batch = ReadBatch.from_strings(seqs, quals)
    for opts in (dict(minq=-5, meanq=-5, maxunk=100, nreads=None), dict(minq=3, meanq=21, maxunk=5, nreads=None),
                 dict(minq=-5, meanq=22, maxunk=100, nreads=9000)):
        eng.set_params(100, quality_offset=33, min_quality=opts["minq"], mean_quality=opts["meanq"], max_unknown=opts["maxunk"], filter_dups=True)
        qc = eng.push(batch)
        res = eng.search(-1 if opts["nreads"] is None else opts["nreads"])
        sampled, code, cnt = oracle.process_reads(batch, 100, 33, opts["minq"], opts["meanq"], opts["maxunk"], opts["nreads"], filter_dups=True)
        assert (res.sampled_reads, res.too_short, res.low_qual, res.dups) == (sampled, cnt["too_short"], cnt["low_qual"], cnt["dups"]), opts
        assert res.dups > 300


def test_verdict_export_import_roundtrip(eng, oracle, markers):
    """mcx_qc_export / mcx_qc_import (the hooks the cross-GPU -n / -d logic uses): exported verdicts and fingerprints
    equal the oracle's, and importing verdicts decided elsewhere drives the search."""
    import ctypes
    from test_host import dup_batch
    seqs, quals = dup_batch(n=5000, seed=4)
    batch = ReadBatch.from_strings(seqs, quals)
    eng.set_params(100, quality_offset=33, min_quality=3, mean_quality=21, max_unknown=5)
    eng.push(batch)
    code, fp = eng.qc_export(True)
    _, ocode, _ = oracle.process_reads(batch, 100, 33, 3, 21, 5, None)
    assert np.array_equal(code, ocode)
    for i in range(0, len(seqs), 37):
        buf = (ctypes.c_uint64 * 2)()
        oracle.lib.oc_fingerprint(seqs[i].encode(), len(seqs[i]), buf)
        assert (int(fp[i, 0]), int(fp[i, 1])) == (buf[0], buf[1])
    sampled, dcode, cnt = oracle.process_reads(batch, 100, 33, 3, 21, 5, None, filter_dups=True)
    qc = eng.qc_import(dcode)
    assert qc["kept"] == sampled and qc["dups"] == cnt["dups"]
    res = eng.search(-1)
    assert (res.sampled_reads, res.dups, res.low_qual, res.too_short) == (sampled, cnt["dups"], cnt["low_qual"], cnt["too_short"])


@pytest.mark.gpu
def test_streamed_batches_equal_one_push(eng, markers, tmp_path, monkeypatch):
    """run_pipeline reads the files through libmcxio in batches; the sums of the batches, the -n cut across batch and
    file boundaries and count_bases are those of a single push of everything."""
    seqs = golden_io.read_fasta("meta.fa.gz")
    a, b = tmp_path / "a.fa", tmp_path / "b.fa.gz"
    a.write_text("".join(">r%d\n%s\n" % (i, s) for i, s in enumerate(seqs[:300])))
    import gzip
    with gzip.open(b, "wt") as fh:
        fh.write("".join(">r%d x\n%s\n%s\n" % (i, s[:60], s[60:]) for i, s in enumerate(seqs[300:])))
    results = []
    for per_batch, nreads in (("1000000", None), ("64", None), ("64", 411), ("7", 411)):
        monkeypatch.setenv("MCX_BATCH_READS", per_batch)
        args = {"seqfiles": [str(a), str(b)], "verbose": False, "nreads": nreads, "read_length": 100, "no_equivs": False}
        est, out = mcb.run_pipeline(args)
        results.append((nreads, est, out["sampled_reads"], mcb.count_bases(out)))
    assert results[0][1:] == results[1][1:] and results[2][1:] == results[3][1:]
    assert results[0][2] == len(seqs) and results[2][2] == 411
    assert results[0][3] == sum(len(s) for s in seqs)
    one = ReadBatch.from_strings(seqs)
    eng.set_params(100)
    eng.push(one)
    res = eng.search(411)
    assert mcb.estimate_average_genome_size({"read_length": 100, "sampled_reads": 411, "verbose": False}, None, res.agg_hits()) == results[2][1]


def test_streamed_duplicate_filter_and_threads(eng, oracle, markers, tmp_path, monkeypatch):
    """-d over a file that arrives in many batches (the context remembers the reads kept by earlier batches), parsed by
    several threads (-t): counters and AGS are those of the oracle's sequential set / of one push of everything."""
    n = 20000
    base = synth.reads(9, 0, n, 100, with_quals=True)
    rng = np.random.default_rng(4)
    b, q = base.bases.reshape(n, 100).copy(), base.quals.reshape(n, 100).copy()
    comp = np.zeros(256, np.uint8); comp[[65, 67, 71, 84, 78]] = [84, 71, 67, 65, 78]
    for i in np.flatnonzero(rng.random(n) < 0.08):
        if i >= 10:
            j = int(rng.integers(0, i))
            b[i] = b[j] if rng.random() < 0.8 else comp[b[j][::-1]]
    seqs = [bytes(r).decode() for r in b]
    quals = [bytes(r).decode() for r in q]
    p = tmp_path / "d.fq"
    p.write_text("".join("@r%d\n%s\n+\n%s\n" % (i, s, q) for i, (s, q) in enumerate(zip(seqs, quals))))
    batch = ReadBatch.from_strings(seqs, quals)
    for nreads in (None, 9000):
        sampled, code, cnt = oracle.process_reads(batch, 100, 32, -5, 29, 100, nreads, filter_dups=True)
        assert cnt["dups"] > 500 and cnt["low_qual"] > 50
        eng.set_params(100, quality_offset=32, mean_quality=29, filter_dups=True)
        eng.push(batch)
        one = eng.search(-1 if nreads is None else nreads)
        want = mcb.estimate_average_genome_size({"read_length": 100, "sampled_reads": one.sampled_reads, "verbose": False}, None, one.agg_hits())
        for per_batch, threads in (("1500", 1), ("1500", 4), ("100000", 8)):
            monkeypatch.setenv("MCX_BATCH_READS", per_batch)
            monkeypatch.setenv("MCXIO_WINDOW_BYTES", "300000")
            args = {"seqfiles": [str(p)], "verbose": False, "nreads": nreads, "read_length": 100, "mean_quality": 29, "filter_dups": True, "threads": threads}
            est, out = mcb.run_pipeline(args)
            assert out["sampled_reads"] == sampled == one.sampled_reads, (nreads, per_batch, threads)
            assert est == want, (nreads, per_batch, threads)
    monkeypatch.delenv("MCXIO_WINDOW_BYTES")


@pytest.mark.gpu
def test_m8_dump_matches_rapsearch_lines(eng, markers, tmp_path):
    """args['m8_out']: the m8-compatible dump (SURVEY 8f-3).  On the reference's own reads >= 99 % of RAPsearch2's
    single-HSP lines appear in it character for character, under the query ids process_seqfile assigns."""
    import gzip
    path = os.path.join(golden_io.GOLD, "meta.fa.gz")
    out = tmp_path / "hits.m8"
    mcb.run_pipeline({"seqfiles": [path], "verbose": False, "nreads": None, "read_length": 100, "m8_out": str(out)})
    ours = set(l.rstrip("\n") for l in open(out) if l[0] != "#")
    ref = [l.rstrip("\n") for l in gzip.open(os.path.join(golden_io.GOLD, "meta.L100.m8.gz"), "rt") if l[0] != "#"]
    single = [l for l in ref if len(l.split("\t")[10].split(".")[-1]) <= 2]
    same = sum(l in ours for l in single)
    assert same >= 0.99 * len(single), (same, len(single))


def test_bench_dump_outputs_are_the_last_step(eng, markers, tmp_path):
    """bench.py --dump-outputs: what the last timed step of both arms computed (AGS, per-family sums, counters, the
    classification of every read, the HSPs) as float64 .npy files, equal to one search of the same seeded reads."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(golden_io.GOLD))
    n = 20000
    out = tmp_path / "dump"
    cp = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "c2", "--reads-per-gpu", str(n), "--steps", "2",
                         "--warmup", "0", "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, cwd=str(tmp_path))
    assert cp.returncode == 0, cp.stderr[-2000:]
    assert json.loads(cp.stdout.strip().splitlines()[-1])["steps"] == 2
    got = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert set(got) == {"%s_%s" % (arm, k) for arm in ("device", "e2e") for k in ("ags", "agg_hits", "counts", "classified", "hits")}
    assert all(a.dtype == np.float64 for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64 << 20
    eng.set_params(100)
    eng.push(synth.reads(2, 0, n, 100))
    res = eng.search(-1)
    agg = res.agg_hits()
    ags = mcb.estimate_average_genome_size({"read_length": 100, "sampled_reads": n, "verbose": False}, None, agg)
    assert res.sampled_reads == n and len(got["device_hits"]) > 1000
    for arm in ("device", "e2e"):
        assert got[arm + "_ags"].tolist() == [ags]
        assert got[arm + "_agg_hits"].tolist() == [agg.get(f, 0.0) for f in markers.fam_names]
        assert np.array_equal(got[arm + "_counts"], res.counts_vector())
        assert np.array_equal(got[arm + "_classified"], eng.classified(n))
        assert np.array_equal(got[arm + "_hits"], eng.hits())
