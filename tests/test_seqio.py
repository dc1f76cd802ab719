"""libmcxio (C++ FASTA/FASTQ reader, include/mcxio.h) against the readfq generator it restates
(mc.py:294-325, mirrored by microbecensus_b200.microbe_census.parse_seqs) and against what the reference's own
parse_seqs / count_bases returned (tests/golden).  No GPU needed."""
import bz2
import gzip
import io
import json
import os
import random
import re

import numpy as np
import pytest

from microbecensus_b200 import microbe_census as mcb, seqio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

CASES = {
    "multi-line fasta, names with spaces, no final newline": ">r1 desc\nACGT\nAC\n>r2\nTTTT\n>r3\n\nGG",
    "fastq, '+name' lines": "@q1\nACGTN\n+\nIIII#\n@q2 x\nAC\n+q2\n!!\n",
    "multi-line fastq, quality starting with @": "@q1\nACGT\nAC\n+\n@III\nII\n@q2\nGG\n+\n@@\n",
    "'+' line inside fasta": ">r1\nAC\n+weird\nGG\n>r2\nTT\n",
    "crlf": "@q1\r\nACGT\r\n+\r\nIIII\r\n@q2\r\nGG\r\n+\r\n##\r\n",
    "lone cr": ">r1\rACGT\rAC\r>r2\rTT\r",
    "quality longer than sequence": "@q1\nACGT\n+\nIIIIIIII\n@q2\nGG\n+\n##\n",
    "quality spread over more lines than the sequence": "@q1\nACGTAC\n+\nII\nII\nII\n@q2\nGG\n+\n##\n",
    "truncated quality at eof": "@q1\nACGT\n+\nIIII\n@q2\nGGGG\n+\n##",
    "eof right after '+'": "@q1\nACGT\n+\nIIII\n@q2\nGGGG\n+\n",
    "junk before the first record": "junk\n\n>r1\nAC\n",
    "empty sequence": ">r1\n>r2\nAC\n@q\n\n+\n\n@q2\nA\n+\nI\n",
    "header only, no newline": ">",
    "header with one character": "@q1\nAC\n+\nII\n>",
    "empty file": "",
    "only newlines": "\n\n\n",
    "fasta then fastq": ">r1\nACGT\n@q1\nGG\n+\nII\n>r2\nT\n",
    "last line without newline loses a character": ">r1\nACGT",
}


def records(text):
    return [(r.seq, r.quality) for r in mcb.parse_seqs(io.StringIO(text, newline=None))]


def check(batch, recs, label):
    assert batch.n == len(recs), label
    any_q = any(q is not None for _, q in recs)
    assert (batch.quals is not None) == any_q, label
    for i, (seq, qual) in enumerate(recs):
        lo, hi = int(batch.offsets[i]), int(batch.offsets[i + 1])
        assert batch.bases[lo:hi].tobytes().decode() == seq, (label, i)
        if any_q:
            want = qual[:len(seq)] if qual is not None else "~" * len(seq)
            assert batch.quals[lo:hi].tobytes().decode() == want, (label, i)


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "mcxio.h")).read()
    declared = set(re.findall(r"\b(mcxio_[a-z0-9_]+)\s*\(", header))
    assert declared == set(seqio.EXPORTS), declared ^ set(seqio.EXPORTS)
    lib = seqio.load()
    for name in declared:
        assert getattr(lib, name) is not None


@pytest.mark.parametrize("label", sorted(CASES))
def test_known_shapes(label, tmp_path):
    text = CASES[label]
    recs = records(text)
    rd = seqio.SeqFile.from_bytes(text.encode())
    check(rd.next_batch(), recs, label)
    assert rd.eof and rd.records_total == len(recs) and rd.bases_total == sum(len(s) for s, _ in recs)
    # the same through a file, plain / gzip / bzip2
    for ext, opener in ((".txt", open), (".gz", gzip.open), (".bz2", bz2.open)):
        p = tmp_path / ("x" + ext)
        with opener(p, "wb") as fh:
            fh.write(text.encode())
        with seqio.SeqFile(str(p)) as f:
            check(f.next_batch(), recs, label + ext)


def check_packed(parts, recs, label):
    """batches of SeqFile.next_packed against the readfq records: bit-planes decoded back to letters"""
    from test_host import _unpack
    seqs = [s for p in parts for s in _unpack(p)]
    assert seqs == ["".join(c if c in "ACGTN" else "x" for c in s) for s, _ in recs], label
    any_q = any(q is not None for _, q in recs)
    if any_q and seqs:
        quals = b"".join(p.quals.tobytes() for p in parts if p.quals is not None).decode()
        want = "".join((q[:len(s)] if q is not None else "~" * len(s)) for s, q in recs)
        if all(p.quals is not None for p in parts if p.n):
            assert quals == want, label


@pytest.mark.parametrize("label", sorted(CASES))
def test_packed_reader_known_shapes(label, tmp_path, monkeypatch):
    """mcxio_next_packed (parallel pieces of a plain file, each checked against the sequential state machine's position;
    packed output) on the same shapes, with pieces of a few bytes so that every guess / re-parse path runs."""
    text = CASES[label]
    recs = records(text)
    p = tmp_path / "x.txt"
    p.write_bytes(text.encode())
    for env in ({}, {"MCXIO_PIECE_BYTES": "7", "MCXIO_MARGIN_BYTES": "5", "MCXIO_WINDOW_BYTES": "23"},
                {"MCXIO_PIECE_BYTES": "3", "MCXIO_MARGIN_BYTES": "64"}):
        for k in ("MCXIO_PIECE_BYTES", "MCXIO_MARGIN_BYTES", "MCXIO_WINDOW_BYTES"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        for threads in (1, 3, 8):
            with seqio.SeqFile(str(p)) as f:
                parts = []
                for _ in range(10000):
                    if f.eof:
                        break
                    parts.append(f.next_packed(2, threads))
                assert f.eof and f.records_total == len(recs) and f.bases_total == sum(len(s) for s, _ in recs), (label, env, threads)
            check_packed(parts, recs, (label, env, threads))
    with gzip.open(tmp_path / "x.gz", "wb") as fh:
        fh.write(text.encode())
    with seqio.SeqFile(str(tmp_path / "x.gz")) as f:
        parts = [f.next_packed(None, 4)]
    check_packed(parts, recs, label + ".gz")


def test_packed_reader_large_random_files(tmp_path, monkeypatch):
    """FASTQ with '@' / '+' / '>' quality lines, multi-line FASTA, ragged lengths: the threaded reader returns the records
    of the sequential one whatever the piece size, and skip_packed / skip_rest walk the same batches."""
    from microbecensus_b200.engine import PackedBatch
    rng = random.Random(11)
    fq = "".join("@r%d d\n%s\n+\n%s\n" % (i, "".join(rng.choice("ACGTN") for _ in range(n)), "".join(rng.choice("@+>I#5") for _ in range(n)))
                 for i, n in enumerate(rng.randrange(1, 160) for _ in range(6000)))
    fa = "".join(">s%d\n%s\n" % (i, "\n".join("".join(rng.choice("ACGTacgtN") for _ in range(rng.randrange(1, 70))) for _ in range(rng.randrange(1, 4))))
                 for i in range(5000))
    for name, text in (("a.fq", fq), ("a.fa", fa)):
        p = tmp_path / name
        p.write_bytes(text.encode())
        with seqio.SeqFile(str(p)) as f:
            ref = PackedBatch.from_batch(f.next_batch(None))
        for env in ({}, {"MCXIO_PIECE_BYTES": "4000", "MCXIO_MARGIN_BYTES": "1500", "MCXIO_WINDOW_BYTES": "50000"},
                    {"MCXIO_PIECE_BYTES": "200", "MCXIO_MARGIN_BYTES": "100", "MCXIO_WINDOW_BYTES": "3000"}):
            for k in ("MCXIO_PIECE_BYTES", "MCXIO_MARGIN_BYTES", "MCXIO_WINDOW_BYTES"):
                monkeypatch.delenv(k, raising=False)
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            for threads in (2, 8):
                with seqio.SeqFile(str(p)) as f:
                    parts, skipped = [], 0
                    turn = 0
                    while not f.eof:
                        if turn % 3 == 2:
                            skipped += f.skip_packed(700, threads)       # a batch another rank would own
                            parts.append(None)
                        else:
                            parts.append(f.next_packed(700, threads))
                        turn += 1
                    assert f.records_total == ref.n and f.bases_total == ref.n_bases
                # replay: the kept batches are contiguous runs of the reference, the skipped ones fill the holes
                pos, woff = 0, np.concatenate([[0], np.cumsum(3 * ((ref.lengths.astype(np.int64) + 31) // 32))])
                with seqio.SeqFile(str(p)) as f2:
                    k = 0
                    while not f2.eof:
                        b = f2.next_packed(700, threads)
                        if parts[k] is not None:
                            assert np.array_equal(parts[k].lengths, b.lengths) and np.array_equal(parts[k].packed, b.packed)
                        assert np.array_equal(b.lengths, ref.lengths[pos:pos + b.n])
                        assert np.array_equal(b.packed, ref.packed[woff[pos]:woff[pos + b.n]])
                        if ref.quals is not None:
                            assert b.quals is not None
                        pos += b.n
                        k += 1
                    assert pos == ref.n and k == len(parts)


def test_batches_and_skip_rest(tmp_path):
    rng = random.Random(7)
    text = "".join("@r%d\n%s\n+\n%s\n" % (i, "".join(rng.choice("ACGTN") for _ in range(n)), "I" * n)
                   for i, n in enumerate(rng.randrange(1, 200) for _ in range(5000)))
    recs = records(text)
    p = tmp_path / "r.fq.gz"
    with gzip.open(p, "wb") as fh:
        fh.write(text.encode())
    with seqio.SeqFile(str(p)) as f:
        got = []
        while not f.eof and len(got) < 1234:
            b = f.next_batch(500)
            got.extend(b.bases[b.offsets[i]:b.offsets[i + 1]].tobytes().decode() for i in range(b.n))
        assert got == [s for s, _ in recs[:len(got)]] and len(got) == 1500
        n, total = f.skip_rest()                     # count_bases folded into the same pass
        assert n == len(recs) and total == sum(len(s) for s, _ in recs)
    assert mcb.count_bases({"seqfiles": [str(p)], "verbose": False}) == total


def test_random_line_soup():
    """Random sequences of line kinds and terminators: the C++ state machine and readfq yield the same records."""
    rng = random.Random(20260101)
    kinds = [">h", "@h x", "+", "+h", "ACGT", "ACGTNNAC", "IIII", "@@@@", "", "G", ">", "@"]
    for trial in range(400):
        text = "".join(rng.choice(kinds) + rng.choice(["\n", "\n", "\n", "\r\n", "\r"]) for _ in range(rng.randrange(1, 40)))
        if rng.random() < 0.3:
            text = text.rstrip("\r\n")
        recs = records(text)
        check(seqio.SeqFile.from_bytes(text.encode()).next_batch(), recs, repr(text))


def test_chunk_boundaries(tmp_path):
    """A file larger than the reader's 8 MB chunks, with CRLF terminators falling on chunk boundaries."""
    line = "ACGT" * 25
    n = 90000                                        # ~ 19 MB
    text = "".join(">r%d\r\n%s\r\n%s\r\n" % (i, line, line[:37]) for i in range(n))
    p = tmp_path / "big.fa"
    p.write_bytes(text.encode())
    with seqio.SeqFile(str(p)) as f:
        b = f.next_batch()
    assert b.n == n and int(b.offsets[-1]) == n * 137
    assert (np.diff(b.offsets) == 137).all()
    assert b.bases[:137].tobytes().decode() == line + line[:37]
    assert b.bases[-137:].tobytes().decode() == line + line[:37]


def test_corrupt_gzip_is_an_error(tmp_path):
    p = tmp_path / "bad.fq.gz"
    raw = gzip.compress(b"@q\nACGT\n+\nIIII\n" * 1000)
    p.write_bytes(raw[:len(raw) // 2])
    with seqio.SeqFile(str(p)) as f:
        with pytest.raises(seqio.SeqIOError):
            f.next_batch()


def test_against_the_reference_generator():
    """The records of the reference's own generator on every shape (tests/golden/readfq_cases.json), and its count_bases
    on its example and test inputs (copies and totals in tests/golden/full)."""
    gold = json.load(open(os.path.join(GOLD, "readfq_cases.json")))["cases"]
    assert set(gold) == set(CASES)
    for label, text in CASES.items():
        assert gold[label]["text"] == text, label
        want = [(s, q) for s, q in gold[label]["records"]]
        check(seqio.SeqFile.from_bytes(text.encode()).next_batch(), want, label)
    exp = json.load(open(os.path.join(GOLD, "full", "expected.json")))
    for key in ("example_fq", "example_fa_500", "metagenome"):
        with seqio.SeqFile(os.path.join(GOLD, "full", exp[key]["file"])) as f:
            n, total = f.skip_rest()
        assert total == exp[key]["total_bases"], key
