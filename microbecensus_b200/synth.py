"""Synthetic reads for the benchmark configurations of BASELINE.json (SURVEY.md 8d).

Reads are drawn uniformly (by length) from the genomes in data/genomes.pack, random strand, 0.1 %
substitution errors.  Read i of a configuration depends only on (seed, i // BLOCK, i % BLOCK): blocks of
BLOCK reads are generated independently, so any shard [lo, hi) of the stream is reproduced exactly by
whichever rank owns it.  Qualities (FASTQ configurations): per-base Q ~ normal(mean falling 34 -> 24
along the read, sd 6) clipped to [2, 41]; in 2 % of the reads 1 % of the bases become 'N'.
"""
import os
import struct

import numpy as np

from .engine import ReadBatch

_HERE = os.path.dirname(os.path.abspath(__file__))
BLOCK = 1 << 18
SEED = 20260101
_genome = None


def genome_pack_path():
    """data/genomes30.pack (all 30 training genomes of the reference, 84.8 Mbp, SURVEY 8d; written by
    `tools/build_genome_pack.py --all` from a reference checkout, kept out of git) if present, else the committed
    ten-genome data/genomes.pack; $MCX_GENOME_PACK overrides."""
    if os.environ.get("MCX_GENOME_PACK"):
        return os.environ["MCX_GENOME_PACK"]
    full = os.path.join(_HERE, "data", "genomes30.pack")
    return full if os.path.isfile(full) else os.path.join(_HERE, "data", "genomes.pack")


def genome():
    """(bases as uint8 codes 0..3, contig start offsets, contig lengths)"""
    global _genome
    if _genome is None:
        blob = open(genome_pack_path(), "rb").read()
        assert blob[:8] == b"MCXGEN01"
        n = struct.unpack_from("<i", blob, 8)[0]
        lens = np.frombuffer(blob, np.int64, n, 12)
        packed = np.frombuffer(blob, np.uint8, offset=12 + 8 * n)
        total = int(lens.sum())
        b = np.empty((len(packed), 4), np.uint8)
        for k in range(4):
            b[:, k] = (packed >> (2 * k)) & 3
        _genome = (b.reshape(-1)[:total].copy(), np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64), lens.copy())
    return _genome


_ASCII = np.frombuffer(b"ACGT", np.uint8)


def _block(config_id, block, n, L, with_quals, insert=None):
    """reads [block*BLOCK, block*BLOCK + n) of the stream -> (bases (n, L) uint8 ASCII, quals or None)"""
    g, starts, lens = genome()
    rng = np.random.Generator(np.random.Philox(key=SEED + config_id, counter=[0, 0, 0, block]))
    span = L if insert is None else insert
    # uniform over positions where a window of `span` fits inside one contig
    room = lens - span + 1
    cum = np.cumsum(room)
    u = rng.integers(0, cum[-1], size=BLOCK)
    ci = np.searchsorted(cum, u, side="right")
    pos = starts[ci] + (u - (cum[ci] - room[ci]))
    strand = rng.integers(0, 2, size=BLOCK).astype(bool)
    err = rng.random((BLOCK, 2))            # reserved streams keep later draws aligned for any n
    idx = pos[:n, None] + np.arange(L)[None, :]
    fwd = g[idx]
    if insert is not None:                  # mate from the other end of the fragment, reverse strand
        idx2 = pos[:n, None] + (insert - 1 - np.arange(L))[None, :]
        rev_mate = 3 - g[idx2]
        return fwd, rev_mate, rng
    rc = 3 - g[pos[:n, None] + (L - 1 - np.arange(L))[None, :]]
    codes = np.where(strand[:n, None], rc, fwd)
    return codes, err, rng


def _finish(codes, rng, n, L, with_quals):
    sub = rng.random((n, L)) < 0.001
    shift = rng.integers(1, 4, size=(n, L), dtype=np.uint8)
    codes = np.where(sub, (codes + shift) & 3, codes).astype(np.uint8)
    bases = _ASCII[codes]
    quals = None
    if with_quals:
        mean = np.linspace(34.0, 24.0, L)[None, :]
        q = np.clip(np.rint(rng.normal(mean, 6.0, size=(n, L))), 2, 41).astype(np.uint8)
        quals = q + 33
        noisy = rng.random(n) < 0.02
        nmask = (rng.random((n, L)) < 0.01) & noisy[:, None]
        bases = np.where(nmask, np.uint8(ord("N")), bases)
    return bases, quals


def reads(config_id, lo, hi, L, with_quals=False):
    """Reads lo..hi-1 of configuration `config_id` as a ReadBatch of fixed-length reads."""
    out_b, out_q = [], []
    i = lo
    while i < hi:
        block, first = divmod(i, BLOCK)
        take = min(hi - i, BLOCK - first)
        codes, _, rng = _block(config_id, block, first + take, L, with_quals)
        b, q = _finish(codes, rng, first + take, L, with_quals)
        out_b.append(b[first:first + take]); out_q.append(None if q is None else q[first:first + take])
        i += take
    n = hi - lo
    bases = np.concatenate(out_b).reshape(-1) if out_b else np.zeros(0, np.uint8)
    quals = np.concatenate(out_q).reshape(-1) if with_quals and out_q else None
    offs = np.arange(n + 1, dtype=np.int64) * L
    return ReadBatch(bases, offs, quals)


def paired_reads(config_id, lo, hi, L, insert=400):
    """Two batches (R1, R2): R2 is the reverse-complement mate from an `insert`-bp fragment."""
    r1b, r1q, r2b, r2q = [], [], [], []
    i = lo
    while i < hi:
        block, first = divmod(i, BLOCK)
        take = min(hi - i, BLOCK - first)
        fwd, mate, rng = _block(config_id, block, first + take, L, True, insert=insert)
        b1, q1 = _finish(fwd, rng, first + take, L, True)
        b2, q2 = _finish(mate, rng, first + take, L, True)
        r1b.append(b1[first:first + take]); r1q.append(q1[first:first + take])
        r2b.append(b2[first:first + take]); r2q.append(q2[first:first + take])
        i += take
    n = hi - lo
    offs = np.arange(n + 1, dtype=np.int64) * L
    return (ReadBatch(np.concatenate(r1b).reshape(-1), offs, np.concatenate(r1q).reshape(-1)),
            ReadBatch(np.concatenate(r2b).reshape(-1), offs.copy(), np.concatenate(r2q).reshape(-1)))


def write_fasta(batch, path):
    L = int(batch.offsets[1] - batch.offsets[0]) if batch.n else 0
    with open(path, "wb") as fh:
        mat = batch.bases.reshape(batch.n, L)
        for i in range(batch.n):
            fh.write(b">%d\n" % i + mat[i].tobytes() + b"\n")


def write_fastq(batch, path):
    L = int(batch.offsets[1] - batch.offsets[0]) if batch.n else 0
    with open(path, "wb") as fh:
        b = batch.bases.reshape(batch.n, L); q = batch.quals.reshape(batch.n, L)
        for i in range(batch.n):
            fh.write(b"@%d\n" % i + b[i].tobytes() + b"\n+\n" + q[i].tobytes() + b"\n")
