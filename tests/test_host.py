"""Host-side logic: reader, QC semantics, drop-in API pieces, C ABI surface.  No GPU needed."""
import ctypes
import gzip
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import golden_io
from microbecensus_b200 import _lib, microbe_census as mcb
from microbecensus_b200.engine import ReadBatch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_library_exports_every_declared_symbol():
    """libmcx.so loads without a GPU and exports exactly the functions include/mcx.h declares."""
    header = open(os.path.join(ROOT, "include", "mcx.h")).read()
    declared = set(re.findall(r"\b(mcx_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = _lib.load()
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"sm_100a" in lib.mcx_version()


def test_no_cpu_fallback_without_device():
    """On a box without a CUDA device mcx_create fails loudly (MCX_ECUDA); nothing computes on the CPU."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from microbecensus_b200.engine import MarkerSearch
    with pytest.raises(_lib.McxError) as e:
        MarkerSearch()
    assert e.value.code == -2 and "no CPU path" in e.value.msg


def test_product_does_not_touch_the_oracle():
    """The oracle is test infrastructure: nothing under microbecensus_b200/ or scripts/ refers to it."""
    for base in ("microbecensus_b200", "scripts"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".h")):
                    txt = open(os.path.join(dirpath, f)).read()
                    assert "libmcoracle" not in txt and "oracle_lib" not in txt and "mc_oracle.h" not in txt, f
                    assert not re.search(r"^\s*(from|import)\s+oracle", txt, re.M), f


def test_struct_layouts_match_header():
    assert ctypes.sizeof(_lib.Cutoff) == 24
    assert ctypes.sizeof(_lib.Params) == 32 + 24 * 30
    assert ctypes.sizeof(_lib.Hit) == 48
    assert ctypes.sizeof(_lib.Result) == 8 * (11 + 30 + 30 + 30 * 1280)


def _unpack(pb):
    """PackedBatch -> strings ('x' for characters that are neither ACGT nor N), checking the padding bits"""
    out, w = [], 0
    for l in (int(x) for x in pb.lengths):
        G = (l + 31) // 32
        lo, hi, mk = (pb.packed[w + k * G: w + (k + 1) * G] for k in range(3))
        w += 3 * G
        chars = []
        for k in range(l):
            a, b, m = ((int(pl[k // 32]) >> (k % 32)) & 1 for pl in (lo, hi, mk))
            chars.append(("N" if a == 0 else "x") if m else "TCAG"[a | (b << 1)])
        if l % 32:
            assert all(int(pl[-1]) >> (l % 32) == 0 for pl in (lo, hi, mk))
        out.append("".join(chars))
    assert w == pb.packed.size
    return out


def test_packed_read_layout_roundtrip():
    """The 2-bit + mask bit-plane layout of include/mcx.h (mcx_push_reads_packed) as the numpy packer writes it:
    fixed-length and ragged batches, N / lower-case / IUPAC characters, empty reads."""
    from microbecensus_b200.engine import PackedBatch
    rng = np.random.default_rng(5)
    alpha = np.frombuffer(b"ACGTNacgtRY", np.uint8)
    p = np.array([0.23] * 4 + [0.04] + [0.04 / 6] * 6); p /= p.sum()
    for lengths in ([150] * 70, [32] * 5, [64] * 3, [int(x) for x in rng.integers(0, 200, size=150)], [0, 1, 31, 32, 33, 0], []):
        seqs = [alpha[rng.choice(len(alpha), size=l, p=p)].tobytes().decode() for l in lengths]
        quals = ["".join(chr(33 + int(q)) for q in rng.integers(0, 42, size=l)) for l in lengths]
        pb = PackedBatch.from_batch(ReadBatch.from_strings(seqs, quals))
        assert pb.n == len(seqs) and pb.n_bases == sum(lengths)
        assert _unpack(pb) == ["".join(c if c in "ACGTN" else "x" for c in s) for s in seqs]
        assert pb.quals.tobytes().decode() == "".join(quals)
        assert pb.packed.size == sum(3 * ((l + 31) // 32) for l in lengths)


def test_reader_matches_readfq_state_machine(tmp_path):
    """libmcxio and the readfq generator agree, including multi-line FASTA / FASTQ, names with spaces, a missing
    final newline and '+' lines inside FASTA (more cases in tests/test_seqio.py)."""
    cases = {
        "a.fa": ">r1 desc\nACGT\nAC\n>r2\nTTTT\n>r3\n\nGG",
        "b.fq": "@q1\nACGTN\n+\nIIII#\n@q2 x\nAC\n+q2\n!!\n",
        "c.fq": "@q1\nACGT\nAC\n+\nIIII\nII\n@q2\nGG\n+\n@@\n",       # multi-line FASTQ
        "d.fa": ">r1\nAC\n+weird\nGG\n>r2\nTT\n",                       # '+' line inside FASTA
    }
    for name, text in cases.items():
        p = tmp_path / name
        p.write_text(text)
        ft = "fastq" if name.endswith(".fq") else "fasta"
        recs = list(mcb.parse_seqs(open(p)))
        b = mcb.load_reads(str(p), ft)
        assert b.n == len(recs), name
        for i, r in enumerate(recs):
            assert b.bases[b.offsets[i]:b.offsets[i + 1]].tobytes().decode() == r.seq, name
            if r.quality is not None and b.quals is not None:
                assert b.quals[b.offsets[i]:b.offsets[i + 1]].tobytes().decode() == r.quality[:len(r.seq)], name


def test_reader_and_autodetect_match_reference_on_its_own_files():
    """The reference's example and test inputs (copies in tests/golden/full): records, total bases, detected file type,
    read length and quality offset, and count_bases as the unmodified reference reported them (full/expected.json)."""
    exp = golden_io.read_json(os.path.join("full", "expected.json"))
    for key in ("example_fq", "example_fa_500", "metagenome"):
        e = exp[key]
        name = os.path.join("full", e["file"])
        path = os.path.join(golden_io.GOLD, name)
        ft = "fasta" if e["quality_offset"] is None else "fastq"     # the reference detects a quality offset for FASTQ only
        seqs = [r[1] for r in golden_io.read_fastq(name)] if ft == "fastq" else golden_io.read_fasta(name)
        b = mcb.load_reads(path, ft)
        assert b.n == len(seqs)
        assert int(b.offsets[-1]) == sum(len(s) for s in seqs) == e["total_bases"]
        for i in range(0, len(seqs), 97):
            assert b.bases[b.offsets[i]:b.offsets[i + 1]].tobytes().decode() == seqs[i]
        assert mcb.auto_detect_file_type(path) == ft
        if "read_length" not in e["opts"]:          # detected by the reference
            assert mcb.auto_detect_read_length(path, ft) == e["read_length"]
        else:                                       # 500 bp reads only: the longest length the reference supports
            assert mcb.auto_detect_read_length(path, ft) == 500
        if ft == "fastq":
            assert mcb.auto_detect_quality_offset(path) == e["quality_offset"]
        assert mcb.count_bases({"seqfiles": [path], "verbose": False, "file_type": ft}) == e["total_bases"]


def test_oracle_qc_matches_reference_counters(oracle):
    """process_seqfile counters (too short / low quality / sampled, incl. the -n cut) recorded from the
    reference for eight option sets on tests/golden/short.fq.gz."""
    recs = golden_io.read_fastq("short.fq.gz")
    batch = ReadBatch.from_strings([r[1] for r in recs], [r[2] for r in recs])
    for case in golden_io.read_json("short.qc.json"):
        o = case["opts"]
        sampled, code, cnt = oracle.process_reads(batch, case["read_length"], case["quality_offset"], o.get("min_quality", -5),
                                                  o.get("mean_quality", -5), o.get("max_unknown", 100), o.get("nreads", 1000000))
        assert (sampled, cnt["too_short"], cnt["low_qual"]) == (case["sampled"], case["too_short"], case["low_qual"]), case
        kept = [recs[i][1][:case["read_length"]] for i in np.flatnonzero(code == 0)]
        assert kept[:3] == case["first_kept"] and kept[-1] == case["last_kept"]


def test_estimator_reference_numbers():
    """estimate_average_genome_size on agg_hits the reference produced (golden json) returns its AGS."""
    for name in ("meta.L100.json", "meta50.L50.json"):
        exp = golden_io.read_json(name)
        args = {"read_length": exp["read_length"], "sampled_reads": exp["sampled_reads"], "verbose": False}
        ags = mcb.estimate_average_genome_size(args, None, exp["agg_hits"])
        assert abs(ags - exp["ags"]) <= 1e-9 * exp["ags"]


def test_report_format(tmp_path):
    args = {"outfile": str(tmp_path / "o.txt"), "seqfiles": ["a.fq", "b.fq"], "sampled_reads": 10, "read_length": 100,
            "min_quality": -5, "mean_quality": -5, "filter_dups": False, "max_unknown": 100}
    mcb.report_results(args, 1234.5, 100)
    txt = open(args["outfile"]).read().split("\n")
    assert txt[0] == "Parameters" and txt[1] == "metagenome:\ta.fq,b.fq" and txt[2] == "reads_sampled:\t10"
    assert txt[9] == "Results" and txt[10] == "average_genome_size:\t1234.5" and txt[12].startswith("genome_equivalents:\t")


def test_counts_vector_allreduce_two_ranks_gloo(tmp_path):
    """N > 1 path on CPU: two gloo ranks all-reduce their per-shard integer counts; the sum equals the counts of
    the whole and agg_hits/AGS computed from it do not depend on the split."""
    script = tmp_path / "w.py"
    script.write_text('''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, "tests"))
from microbecensus_b200.markers import Markers, report_floor
from microbecensus_b200.engine import ReadBatch, SearchResult
from microbecensus_b200 import microbe_census as mcb
from oracle_lib import Oracle
import golden_io
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
m = Markers(); o = Oracle(m)
seqs = golden_io.read_fasta("meta.fa.gz")[:240]
def counts(ss):
    b = ReadBatch.from_strings(ss)
    h, _ = o.search(b, 100, report_floor(100)); c = o.classify(h, 100, m, b.n)
    class Raw: pass
    raw = Raw()
    for k in ("too_short","low_qual","dups","n_seed_hits","n_gapped","gapped_cells","n_capped_reads"): setattr(raw, k, 0)
    raw.sampled_reads = b.n; raw.reads_classified = c["classified"]; raw.n_hsp = len(h); raw.reads_with_hits = len(set(h[:,0].tolist()))
    raw.fam_hits = c["fam_hits"]; raw.fam_aln = c["fam_aln"]; raw.aln_by_len = c["aln_by_len"].ravel()
    return SearchResult(raw, m, 100)
n = len(seqs); lo, hi = r * n // w, (r + 1) * n // w
part = counts(seqs[lo:hi])
v = torch.from_numpy(part.counts_vector()); dist.all_reduce(v); part.load_counts_vector(v.numpy())
whole = counts(seqs)
assert np.array_equal(part.counts_vector(), whole.counts_vector())
a1 = mcb.estimate_average_genome_size({"read_length":100,"sampled_reads":part.sampled_reads,"verbose":False}, None, part.agg_hits())
a2 = mcb.estimate_average_genome_size({"read_length":100,"sampled_reads":whole.sampled_reads,"verbose":False}, None, whole.agg_hits())
assert a1 == a2
dist.destroy_process_group()
''' % (ROOT, ROOT))
    subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                           "--master-port", "29517", str(script)], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=600)


def dup_batch(n=3000, L=100, seed=5):
    """reads with injected exact and reverse-complement duplicates, ragged lengths, N's and varied qualities"""
    rng = np.random.default_rng(seed)
    comp = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
    seqs, quals = [], []
    for i in range(n):
        u = rng.random()
        if i > 10 and u < 0.08:
            s = seqs[int(rng.integers(0, i))]
        elif i > 10 and u < 0.12:
            s = "".join(comp[c] for c in reversed(seqs[int(rng.integers(0, i))]))
        else:
            ln = int(rng.choice([L - 20, L, L + 7, L + 30]))
            s = "".join(rng.choice(list("ACGT"), ln))
            if rng.random() < 0.05:
                s = s[:5] + "N" * 12 + s[17:]
        seqs.append(s)
        lowq = 2 if rng.random() < 0.2 else 12
        quals.append("".join(chr(33 + int(q)) for q in rng.integers(lowq, 41, len(s))))
    return seqs, quals


def reference_loop(seqs, quals, L, qoff, minq, meanq, maxunk, dups, nreads):
    """process_seqfile (mc.py:328-367) re-typed over in-memory records: the known answer for the -d semantics"""
    comp = {"A": "T", "T": "A", "G": "C", "C": "G", "N": "N"}
    seen, kept, too_short, low_qual, ndup = set(), [], 0, 0, 0
    for i, (s, q) in enumerate(zip(seqs, quals)):
        if len(s) < L:
            too_short += 1; continue
        if dups and (s in seen or "".join(comp[c] for c in s[::-1]) in seen):
            ndup += 1; continue
        t = s[:L]
        ph = [ord(c) - qoff for c in q[:L]]
        if 100 * t.count("N") / float(len(t)) > maxunk or float(np.mean(ph)) < meanq or min(ph) < minq:
            low_qual += 1; continue
        kept.append(i)
        if dups:
            seen.add(s)
        if len(kept) == nreads:
            break
    return kept, too_short, low_qual, ndup


def test_oracle_duplicate_filter_matches_reference_semantics(oracle):
    seqs, quals = dup_batch()
    batch = ReadBatch.from_strings(seqs, quals)
    for opts in (dict(minq=-5, meanq=-5, maxunk=100, nreads=10**9), dict(minq=3, meanq=21, maxunk=5, nreads=10**9),
                 dict(minq=-5, meanq=22, maxunk=100, nreads=1500)):
        kept, ts, lq, nd = reference_loop(seqs, quals, 100, 33, opts["minq"], opts["meanq"], opts["maxunk"], True, opts["nreads"])
        sampled, code, cnt = oracle.process_reads(batch, 100, 33, opts["minq"], opts["meanq"], opts["maxunk"], opts["nreads"], filter_dups=True)
        assert sampled == len(kept) and list(np.flatnonzero(code == 0)) == kept
        assert (cnt["too_short"], cnt["low_qual"], cnt["dups"]) == (ts, lq, nd)
        assert nd > 60


def test_sharded_quota_and_duplicates_equal_the_whole(oracle):
    """Cross-GPU logic on CPU: three contiguous shards + shard_quota + resolve_duplicates reproduce the verdicts and
    counters of one pass over everything (oracle = reference loop) for -d with QC and a -n cut."""
    from microbecensus_b200.distributed import shard_quota, resolve_duplicates
    seqs, quals = dup_batch(n=4000, seed=21)
    whole = ReadBatch.from_strings(seqs, quals)
    fp = np.zeros((len(seqs), 2), np.uint64)
    for i, s in enumerate(seqs):
        buf = (ctypes.c_uint64 * 2)()
        oracle.lib.oc_fingerprint(s.encode(), len(s), buf)
        fp[i] = (buf[0], buf[1])
    bounds = [0, 1100, 2900, 4000]
    for nreads in (None, 1700, 2500):
        sampled, code, cnt = oracle.process_reads(whole, 100, 33, 3, 21, 5, nreads, filter_dups=True)
        # per shard: local QC without -d
        local = []
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            _, c, _ = oracle.process_reads(whole.slice(lo, hi), 100, 33, 3, 21, 5, None, filter_dups=False)
            local.append(c)
        allc = np.concatenate(local)
        ok = np.flatnonzero(allc == 0)
        resolved = [resolve_duplicates(c, fp[lo:hi], lo, fp[ok], ok) for c, (lo, hi) in zip(local, zip(bounds[:-1], bounds[1:]))]
        kept = [int((c == 0).sum()) for c in resolved]
        quotas = [shard_quota(kept, nreads, r) for r in range(3)]
        tot = {"sampled": 0, "too_short": 0, "low_qual": 0, "dups": 0}
        for c, q in zip(resolved, quotas):
            if q == 0:
                continue
            if q < 0:
                upto = len(c)
                tot["sampled"] += int((c == 0).sum())
            else:
                upto = int(np.flatnonzero(c == 0)[q - 1]) + 1
                tot["sampled"] += q
            tot["too_short"] += int((c[:upto] == 1).sum()); tot["low_qual"] += int((c[:upto] == 2).sum()); tot["dups"] += int((c[:upto] == 3).sum())
        assert tot == {"sampled": sampled, "too_short": cnt["too_short"], "low_qual": cnt["low_qual"], "dups": cnt["dups"]}, (nreads, tot, cnt)
        searched = np.concatenate(resolved)
        assert np.array_equal(np.flatnonzero(searched == 0)[:sampled], np.flatnonzero(code == 0))


def test_host_module_does_not_import_torch():
    """A single-GPU run goes numpy + ctypes only: importing torch costs more than searching a million reads."""
    out = subprocess.run([sys.executable, "-c", "import sys; sys.path.insert(0, %r); import microbecensus_b200.microbe_census; "
                          "print('torch' in sys.modules)" % ROOT], capture_output=True, text=True)
    assert out.stdout.strip() == "False", out.stdout + out.stderr


def test_exchange_duplicates_two_ranks_gloo(tmp_path):
    """-d across ranks (all-to-all routed by fingerprint, owner-side sort and marks, all-to-all back) on two and three
    gloo ranks on CPU: every rank ends with the verdicts `resolve_duplicates` gives with all passing fingerprints in hand."""
    script = tmp_path / "w.py"
    script.write_text('''
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %r)
from microbecensus_b200.distributed import exchange_duplicates, resolve_duplicates
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
rng = np.random.default_rng(7)
n = 6000
fp = rng.integers(0, 2**63, size=(n, 2), dtype=np.int64).astype(np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, 2)).astype(np.uint64)
for i in rng.choice(np.arange(50, n), 900, replace=False):      # duplicates of earlier reads, some of them chains
    fp[i] = fp[rng.integers(0, i)]
codes = rng.choice(np.array([0, 0, 0, 0, 1, 2], np.uint8), n)
ok = np.flatnonzero(codes == 0)
bounds = [k * n // w for k in range(w + 1)]
lo, hi = bounds[r], bounds[r + 1]
got = exchange_duplicates(codes[lo:hi], fp[lo:hi], lo)
want = resolve_duplicates(codes[lo:hi], fp[lo:hi], lo, fp[ok], ok)
assert np.array_equal(got, want), (r, int((got != want).sum()))
assert (want == 3).sum() > 50
empty = exchange_duplicates(codes[:0], fp[:0], 0) if r == 0 else exchange_duplicates(codes[lo:hi], fp[lo:hi], lo)
dist.destroy_process_group()
''' % ROOT)
    for nproc, port in ((2, "29518"), (3, "29519")):
        subprocess.check_call([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=%d" % nproc, "--master-addr", "127.0.0.1",
                               "--master-port", port, str(script)], stdout=subprocess.DEVNULL, timeout=600)


def test_marker_blob_equals_reference_maps():
    """find_opt_pars / read_dic (mc.py:61-88): every cut-off, coefficient and weight per (read length, family) and the
    family and length of every subject in the packed blob equal the reference's own *.map files -- line by line where the
    reference tree is mounted, by the committed digest of those lines (tools/marker_digest.py) elsewhere."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import marker_digest as md
    from microbecensus_b200.markers import Markers
    m = Markers()
    ours = md.lines_from_blob(m)
    want, n = open(os.path.join(ROOT, "tests", "golden", "marker_maps.sha256")).read().split()
    assert len(ours) == int(n) == 3 * 600 + m.n_subj
    assert md.digest(ours) == want
    if os.path.isdir("/root/reference/microbe_census/data"):
        theirs = md.lines_from_reference("/root/reference", set(m.names))
        assert theirs == ours


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the driver's CPU arm): one JSON line with the metric, unit and config of the GPU arm, the
    reference's own functions and rapsearch child on a bounded sample, no GPU and none of this package's search code."""
    import json
    if not os.path.exists(os.path.join(ROOT, "baseline", "_ref", "microbe_census", "data", "rapdb_2.15")):
        pytest.skip("reference install (baseline/_ref) not present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-sample", "400"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-400:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "reads/sec end-to-end AGS" and line["unit"] == "reads/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["gpu_launches"] == 0
    assert line["config"]["read_length"] == 150 and "150 bp" in line["config"]["workload"]
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
