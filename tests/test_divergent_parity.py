"""The CUDA path against the oracle on divergent homologs of the markers (tests/homologs.py) at every supported read
length, the gapped stage's hand-offs forced down to the fallback kernel, and k_qc on ragged FASTQ at the boundaries of
its tests.  The tests marked gpu need a B200; the others check the generators and the references on the CPU.

The golden and synthetic reads of test_gpu_parity.py either miss the markers or match them almost exactly; here the
reads carry substitutions up to 40 %, indels, subject ends, low-complexity stretches and ambiguous bases, and every
test also checks that the input still reaches the paths it exists for (floors at about half of what a B200 run of
these seeds shows)."""
import concurrent.futures as cf
import os

import numpy as np
import pytest

from homologs import homolog_reads
from microbecensus_b200.engine import MarkerSearch, PackedBatch, ReadBatch
from microbecensus_b200.markers import LOG10_KN
from oracle_lib import MCX_ORDER, OC_HIT_FIELDS

READ_LENGTHS = sorted(LOG10_KN)
F = {k: OC_HIT_FIELDS.index(k) for k in OC_HIT_FIELDS}


@pytest.fixture(scope="module")
def eng(markers):
    e = MarkerSearch(markers, 0)
    yield e
    e.close()


def oracle_hits(oracle, batch, L, min_raw):
    """oracle.search on slices of the batch on threads (the C calls release the GIL and only read the index)"""
    workers = max(1, min(32, os.cpu_count() or 1))
    oracle.search(batch.slice(0, min(8, batch.n)), L, min_raw)        # one-time table set-up before the threads start
    cuts = np.linspace(0, batch.n, 4 * workers + 1).astype(np.int64)

    def part(k):
        lo, hi = int(cuts[k]), int(cuts[k + 1])
        oh, _ = oracle.search(batch.slice(lo, hi), L, min_raw, cap=1500 * (hi - lo) + 20000)
        oh[:, 0] += lo
        return oh
    with cf.ThreadPoolExecutor(workers) as ex:
        return np.concatenate(list(ex.map(part, range(len(cuts) - 1))))


def search_vs_oracle(eng, oracle, markers, batch, L):
    """gpu_vs_oracle of test_gpu_parity with the oracle on threads: every HSP with all 12 fields, the sums, aln_by_len,
    the best subject of every read, n_hsp and reads_with_hits.  -> (result, oracle hits, oracle classification)"""
    eng.set_params(L)
    eng.push(batch)
    res = eng.search(-1)
    hits = eng.hits()
    oh = oracle_hits(oracle, batch, L, eng.min_report_raw)
    assert hits.shape == oh[:, MCX_ORDER].shape
    bad = np.flatnonzero((hits != oh[:, MCX_ORDER]).any(axis=1)) if hits.shape == oh[:, MCX_ORDER].shape else []
    assert len(bad) == 0, ("first differing HSP", L, hits[bad[0]].tolist(), oh[bad[0], MCX_ORDER].tolist())
    oc = oracle.classify(oh, L, markers, batch.n)
    assert res.reads_classified == oc["classified"]
    assert np.array_equal(res.fam_hits, oc["fam_hits"])
    assert np.array_equal(res.fam_aln, oc["fam_aln"])
    assert np.array_equal(res.aln_by_len, oc["aln_by_len"])
    assert np.array_equal(eng.classified(batch.n), oc["best_subject"])
    assert res.n_hsp == len(oh)
    assert res.reads_with_hits == len(set(oh[:, 0].tolist()))
    return res, oh, oc


def coverage(oh, oc, markers, L):
    """what the input reached: HSPs with gap openings, at a subject's ends and at a frame's ends; reads classified, and
    reads with hits that were not classified"""
    slen = markers.subj_len[oh[:, F["subject"]]]
    mlen = (L - oh[:, F["frame"]] % 3) // 3
    hit_reads = np.unique(oh[:, F["read"]])
    return {"gapo1": int((oh[:, F["gapo"]] >= 1).sum()), "gapo2": int((oh[:, F["gapo"]] >= 2).sum()),
            "subject_ends": int(((oh[:, F["t0"]] == 0) | (oh[:, F["t1"]] == slen - 1)).sum()),
            "frame_ends": int(((oh[:, F["q0"]] == 0) | (oh[:, F["q1"]] == mlen - 1)).sum()),
            "classified": int(oc["classified"]),
            "hits_unclassified": int((oc["best_subject"][hit_reads] < 0).sum())}


# floors of coverage() per read length for homolog_reads(markers, 1, 3000, L): half of the counts observed (the oracle's,
# which the GPU path equals), in the order of COVERAGE_KEYS
COVERAGE_KEYS = ("gapo1", "gapo2", "subject_ends", "frame_ends", "classified", "hits_unclassified")
FLOORS = {50: (265, 0, 1513, 16324, 204, 104), 60: (703, 1, 1714, 29926, 279, 133), 70: (1563, 10, 2001, 33732, 335, 155),
          80: (3933, 97, 5920, 44833, 429, 198), 90: (5923, 145, 5673, 52692, 498, 209),
          100: (10226, 392, 6530, 60291, 560, 241), 110: (12618, 846, 8461, 69277, 637, 232),
          120: (14838, 1103, 8455, 74210, 693, 263), 130: (18471, 1784, 10637, 79773, 728, 283),
          140: (23780, 2155, 12441, 86759, 788, 284), 150: (25307, 3062, 12528, 95424, 809, 323),
          175: (36692, 5094, 14582, 110724, 955, 287), 200: (50674, 8500, 20734, 124836, 1069, 239),
          225: (58732, 10681, 19533, 140972, 1153, 220), 250: (68219, 12217, 25537, 143729, 1171, 226),
          300: (92201, 21153, 44099, 155728, 1274, 145), 350: (104705, 25814, 55456, 150065, 1299, 132),
          400: (123254, 32020, 89267, 145070, 1309, 137), 450: (137996, 37048, 105719, 133261, 1300, 138),
          500: (139531, 38737, 130934, 125279, 1310, 125)}
# ... and of the gapped stage's work at the same lengths: extensions (n_gapped), extensions handed to k_gap_dp, and
# extensions whose live window outgrew k_gap_dp's ring and went to k_gap_dir without any knob (a B200 run of these
# seeds saw 1 at 140 and 250 bp, 21 / 1 / 2 / 6 / 9 at 300 / 350 / 400 / 450 / 500 bp)
GAP_FLOORS = {50: (4322, 275), 60: (12097, 713), 70: (21218, 1667), 80: (37610, 4235), 90: (50109, 7072),
              100: (68028, 12166), 110: (82704, 15983), 120: (104821, 17820), 130: (129378, 24740), 140: (157285, 30624),
              150: (182622, 33916), 175: (247186, 51354), 200: (311604, 69963), 225: (377106, 88112), 250: (418412, 103943),
              300: (542979, 150961), 350: (637848, 180985), 400: (735712, 222625), 450: (810884, 253185), 500: (837392, 261782)}
NATURAL_WIDE = {300: 10, 450: 3, 500: 4}


def test_read_lengths_are_the_supported_ones(markers):
    assert READ_LENGTHS == markers.read_lengths


def test_homolog_reads_are_seeded_and_mixed(markers):
    """same seed, same reads; both strands, reads longer and shorter than L, ambiguous and lower-case bases"""
    a, b = homolog_reads(markers, 9, 400, 150), homolog_reads(markers, 9, 400, 150)
    assert np.array_equal(a.bases, b.bases) and np.array_equal(a.offsets, b.offsets)
    assert not np.array_equal(homolog_reads(markers, 10, 400, 150).bases, a.bases)
    lens = np.diff(a.offsets)
    assert (lens < 150).any() and (lens > 150).any() and (lens == 150).sum() > 300
    for c in b"NRYKacgt":
        assert (a.bases == c).any(), chr(c)


@pytest.mark.parametrize("qoff,L,minq,meanq,maxunk", [(33, 100, 10, 25, 5), (64, 250, -5, 3, 2), (33, 150, 0, 30, 2)])
def test_qc_float64_reference_equals_oracle_on_the_boundaries(oracle, markers, qoff, L, minq, meanq, maxunk):
    """the oracle's integer form of the QC tests against mc.py's float64 arithmetic, on reads whose statistics sit on and
    one unit off every boundary"""
    batch = ragged_fastq(markers, 5, L, qoff, minq, meanq, maxunk)
    want = qc_reference(batch, L, qoff, minq, meanq, maxunk)
    _, ocode, _ = oracle.process_reads(batch, L, qoff, minq, meanq, maxunk, None)
    assert np.array_equal(ocode, want)
    on = 0
    for r in range(batch.n):
        a = int(batch.offsets[r])
        if batch.offsets[r + 1] - a >= L:
            q = batch.quals[a:a + L].astype(np.int64) - qoff
            on += int(q.sum()) in (meanq * L, meanq * L - 1) or int(q.min()) in (minq, minq - 1)
    assert on > batch.n // 4 and (batch.quals == 255).any() and (batch.quals < qoff).any()


@pytest.mark.gpu
@pytest.mark.parametrize("L", READ_LENGTHS)
def test_divergent_homologs_bit_exact_at_every_read_length(eng, oracle, markers, L):
    batch = homolog_reads(markers, 1, 3000, L)
    res, oh, oc = search_vs_oracle(eng, oracle, markers, batch, L)
    cov = coverage(oh, oc, markers, L)
    work = eng.search_counters()
    print("coverage L=%d %s n_gapped=%d counters=%s" % (L, cov, res.n_gapped, work))
    for k, v in zip(COVERAGE_KEYS, FLOORS[L]):
        assert cov[k] >= v, (L, k, cov)
    assert cov["classified"] > 0 and cov["hits_unclassified"] > 0 and cov["gapo1"] > 0
    assert res.too_short > 0
    assert res.n_gapped >= GAP_FLOORS[L][0] and work["gap_dp_extensions"] >= GAP_FLOORS[L][1], (L, res.n_gapped, work)
    assert work["gap_wide_extensions"] >= NATURAL_WIDE.get(L, 0), (L, work)


@pytest.mark.gpu
def test_large_divergent_sample_bit_exact_at_150(eng, oracle, markers):
    """100,000 homolog reads at 150 bp, the metric length of the benchmark"""
    L = 150
    batch = homolog_reads(markers, 2, 100_000, L)
    res, oh, oc = search_vs_oracle(eng, oracle, markers, batch, L)
    cov = coverage(oh, oc, markers, L)
    work = eng.search_counters()
    print("coverage large L=150 %s n_gapped=%d counters=%s" % (cov, res.n_gapped, work))
    # floors: half of what a B200 run of this seed saw (1,757,842 / 206,284 / 729,945 / 6,553,682 / 56,081 / 20,273;
    # 12,026,814 extensions, 2,325,109 to k_gap_dp, 15 to k_gap_dir)
    for k, v in zip(COVERAGE_KEYS, (878921, 103142, 364972, 3276841, 28040, 10136)):
        assert cov[k] >= v, (k, cov)
    assert res.n_gapped >= 6_013_407 and work["gap_dp_extensions"] >= 1_162_554 and work["gap_wide_extensions"] >= 7, work


# ---------------------------------------------------------------------------------------------------------------------
# the gapped stage's hand-offs: screen -> k_gap_dp -> k_gap_dir

FORCE = {"MCX_GAP_SCREEN_ROWS": 1, "MCX_GAP_SCREEN_COLS": 1, "MCX_GAP_DP_COLS": 1}


def _full_state(eng, n):
    res = eng.search(-1)
    return res.counts_vector(), eng.hits(), eng.classified(n), eng.qc_export(False)[0]


def _fresh_search(markers, batch, L):
    eng = MarkerSearch(markers, 0)
    try:
        eng.set_params(L)
        eng.push(batch)
        return _full_state(eng, batch.n), eng.search_counters()
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [100, 150, 500])
def test_forced_gapped_handoffs_equal_default_and_oracle(oracle, markers, monkeypatch, L):
    """Every extension that survives the first row of the screening pass goes to k_gap_dp, and every one of those to the
    wide-window fallback k_gap_dir (its score pass and its statistics pass): same counts, HSPs, classification and QC
    verdicts as the default search, and both equal the oracle."""
    batch = homolog_reads(markers, 3, 3000, L)
    ref, work = _fresh_search(markers, batch, L)
    for k, v in FORCE.items():
        monkeypatch.setenv(k, str(v))
    got, forced = _fresh_search(markers, batch, L)
    for k in FORCE:
        monkeypatch.delenv(k)
    print("hand-offs L=%d default %s forced %s" % (L, work, forced))
    # a B200 run of this seed: 126,153 / 361,120 / 1,764,897 extensions through k_gap_dir at 100 / 150 / 500 bp, i.e.
    # every extension handed to k_gap_dp (19,872 / 69,256 / 562,966 of them by default, 0 / 0 / 4 of those wide)
    assert forced["gap_wide_extensions"] == forced["gap_dp_extensions"] >= {100: 63076, 150: 180560, 500: 882448}[L], forced
    assert forced["gap_dp_extensions"] > work["gap_dp_extensions"]
    for name, a, b in zip(("counts", "hits", "classified", "qc codes"), ref, got):
        assert a.shape == b.shape and np.array_equal(a, b), name
    eng = MarkerSearch(markers, 0)
    try:
        search_vs_oracle(eng, oracle, markers, batch, L)
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------------------------------
# k_qc on ragged FASTQ

def qc_reference(batch, L, qoff, minq, meanq, maxunk):
    """mc.py:265-279 (with the too-short test of :342) in float64: %N of seq[:L] as a float, numpy.mean of the trimmed
    qualities"""
    code = np.zeros(batch.n, np.uint8)
    for r in range(batch.n):
        a, b = int(batch.offsets[r]), int(batch.offsets[r + 1])
        if b - a < L:
            code[r] = 1
            continue
        seq = batch.bases[a:a + L]
        q = batch.quals[a:a + L].astype(np.int64) - qoff
        if 100 * int((seq == ord("N")).sum()) / L > maxunk or np.mean(q) < meanq or q.min() < minq:
            code[r] = 2
    return code


def ragged_fastq(markers, seed, L, qoff, minq, meanq, maxunk, n=3000):
    """Reads of 40-600 bp (quality starts on every residue mod 16, the last read ending at the buffer end off a 16-byte
    boundary), most at or next to a boundary of the QC tests over their first L bases: sum(q) = meanq L or one less,
    min(q) = minq or one less, 100 nN = maxunk L or the next N; bytes below the offset and 0xff among the qualities."""
    rng = np.random.default_rng([seed, L, qoff])
    hom = _homolog_strings(markers, L)
    lens = rng.integers(40, 601, size=n)
    lens[-1] = max(L + 3, int(lens[-1]))
    if (lens.sum() % 16) == 0:
        lens[-1] += 1
    seqs, quals = [], []
    nN_on = maxunk * L // 100
    assert nN_on * 100 == maxunk * L
    for r, ln in enumerate(lens):
        ln = int(ln)
        src = hom[r % len(hom)]
        s = np.frombuffer((src * (ln // len(src) + 1))[:ln].encode(), np.uint8).copy()
        q = np.full(ln, meanq, np.int64)                         # relative qualities; the first L decide
        kind = int(rng.integers(0, 8))
        m = min(ln, L)
        if kind == 7:                                            # anything, with bytes below the offset and 0xff
            q = rng.integers(-qoff, 256 - qoff, size=ln)
        else:
            # spread without moving the sum: +d at one place, -d at another (staying >= minq)
            for _ in range(int(rng.integers(0, 6))):
                i, j = rng.integers(0, m, size=2)
                d = int(rng.integers(0, max(1, q[j] - minq)))
                if i != j and q[i] + d <= 255 - qoff:
                    q[i] += d; q[j] -= d
            if kind == 1:
                q[int(rng.integers(0, m))] -= 1                  # sum one below meanq L
            elif kind == 2:                                      # min exactly minq, sum kept
                i, j = rng.choice(m, size=2, replace=False)
                q[j] += q[i] - minq; q[i] = minq
            elif kind == 3:                                      # min one below minq, sum kept
                i, j = rng.choice(m, size=2, replace=False)
                q[j] += q[i] - (minq - 1); q[i] = minq - 1
            q = np.clip(q, -qoff, 255 - qoff)
            if ln > L:                                           # past the trim: anything
                q[L:] = rng.integers(-qoff, 256 - qoff, size=ln - L)
        k_n = {4: nN_on, 5: nN_on + 1}.get(kind, int(rng.integers(0, 2)))
        if kind in (4, 5):
            s[:m][s[:m] == ord("N")] = ord("A")
        if k_n and m >= k_n:
            s[rng.choice(m, size=k_n, replace=False)] = ord("N")
        for p in rng.integers(0, ln, size=int(rng.integers(0, 3))):   # not unknown bases: lower case, IUPAC
            s[p] = ord(rng.choice(["n", "R", "Y", "a"]))
        seqs.append(s)
        quals.append((q + qoff).astype(np.uint8))
    offs = np.zeros(n + 1, np.int64)
    offs[1:] = np.cumsum(lens)
    return ReadBatch(np.concatenate(seqs), offs, np.concatenate(quals))


_HOM = {}


def _homolog_strings(markers, L):
    """400 homolog reads as upper-case ACGTN strings (the bases of the ragged reads)"""
    if L not in _HOM:
        b = homolog_reads(markers, 4, 400, L)
        _HOM[L] = [bytes(b.bases[b.offsets[i]:b.offsets[i + 1]]).decode().upper().replace("R", "A").replace("Y", "C")
                   .replace("K", "G") for i in range(b.n)]
    return _HOM[L]


@pytest.mark.gpu
@pytest.mark.parametrize("qoff,L,minq,meanq,maxunk", [(33, 100, 10, 25, 5), (64, 250, -5, 3, 2), (33, 150, 0, 30, 2)])
def test_k_qc_boundaries_on_ragged_fastq(eng, oracle, markers, qoff, L, minq, meanq, maxunk):
    import torch
    batch = ragged_fastq(markers, 5, L, qoff, minq, meanq, maxunk)
    want = qc_reference(batch, L, qoff, minq, meanq, maxunk)
    _, ocode, _ = oracle.process_reads(batch, L, qoff, minq, meanq, maxunk, None)
    assert np.array_equal(ocode, want)
    assert (want == 0).sum() > 200 and (want == 2).sum() > 200 and (want == 1).sum() > 100
    eng.set_params(L, quality_offset=qoff, min_quality=minq, mean_quality=meanq, max_unknown=maxunk)
    pb = PackedBatch.from_batch(batch)
    d_p = torch.from_numpy(pb.packed.view(np.int32)).cuda()
    d_l = torch.from_numpy(pb.lengths.view(np.int32)).cuda()
    d_q = torch.from_numpy(pb.quals).cuda()
    torch.cuda.synchronize()
    for name, push in (("ascii", lambda: eng.push(batch)), ("packed", lambda: eng.push(pb)),
                       ("packed device", lambda: eng.push_packed_device(d_p.data_ptr(), int(d_p.numel()), d_l.data_ptr(),
                                                                        d_q.data_ptr(), pb.n_bases, batch.n))):
        push()
        code = eng.qc_export(False)[0]
        bad = np.flatnonzero(code != want)
        assert len(bad) == 0, (name, "read", int(bad[0]), int(code[bad[0]]), int(want[bad[0]]))
        res = eng.search(-1)
        assert (res.sampled_reads, res.too_short, res.low_qual) == ((want == 0).sum(), (want == 1).sum(), (want == 2).sum())
        # the searched reads are exactly the kept ones: the oracle's HSPs on that subset
        kept = np.flatnonzero(want == 0)
        sub = ReadBatch.from_strings([bytes(batch.bases[batch.offsets[i]:batch.offsets[i + 1]]).decode() for i in kept])
        oh = oracle_hits(oracle, sub, L, eng.min_report_raw)
        hits = eng.hits()
        assert len(hits) == len(oh) > 0, name
        assert np.array_equal(hits[:, 1:], oh[:, MCX_ORDER][:, 1:]), name
        assert np.array_equal(hits[:, 0], kept[oh[:, 0]]), name
