"""Reads that are divergent homologs of the marker proteins (numpy only).  Test infrastructure.

The seeded synthetic reads of `synth.reads` are cut from the training genomes with 0.1 % substitutions: a read that
hits a marker matches it almost exactly, so the decisions that only matter on divergent homologs (one-substitution
seed words, the seed acceptance test near its threshold, X-drop stops, gapped extensions with real gaps, SEG masks
inside an alignment, alignments that reach a subject's ends) rarely reach a comparison with the oracle.  Each read
made here back-translates a window of a marker subject with:

- synonymous codons drawn at random (the five off-frames are not degenerate), no stop codons;
- either strand and a 0-2 nt prefix, so that hits land in all six frames;
- a per-read amino-acid substitution rate of 0, 10, 20, 30 or 40 %, replacements drawn with weights 2^(s/2) of the
  BLOSUM62 score s (similar residues are likely, as in real homologs);
- 0-3 codon-preserving indels of 1-20 residues anywhere in the window (some long enough to carry an extension past the
  screening pass's 32 rows or 48 columns);
- windows that start before residue 0 or run past the last residue of the subject (random residues in the overhang),
  and short subjects wholly inside a read;
- in about 20 % of reads an 8-40 residue homopolymer or period-2/3 repeat at the start, middle or end of the
  homologous part (the SEG hard mask falls inside hits, also segments longer than 25);
- in about 5 % of reads N, IUPAC letters (R, Y, K) and lower case bases inside the read;
- windows over the subjects' X residues, chosen on purpose (back-translated as random codons);
- reads longer than L (trimmed by the search) and a few shorter than L (too short) in the same batch.

The same (markers, seed, n, L) always gives the same reads.
"""
import numpy as np

from microbecensus_b200.engine import ReadBatch

AA = "ARNDCQEGHILKMFPSTWYV"
# BLOSUM62 in the order above (only the weights of the substitutions depend on it)
_B62 = np.array([
    [4, -1, -2, -2, 0, -1, -1, 0, -2, -1, -1, -1, -1, -2, -1, 1, 0, -3, -2, 0],
    [-1, 5, 0, -2, -3, 1, 0, -2, 0, -3, -2, 2, -1, -3, -2, -1, -1, -3, -2, -3],
    [-2, 0, 6, 1, -3, 0, 0, 0, 1, -3, -3, 0, -2, -3, -2, 1, 0, -4, -2, -3],
    [-2, -2, 1, 6, -3, 0, 2, -1, -1, -3, -4, -1, -3, -3, -1, 0, -1, -4, -3, -3],
    [0, -3, -3, -3, 9, -3, -4, -3, -3, -1, -1, -3, -1, -2, -3, -1, -1, -2, -2, -1],
    [-1, 1, 0, 0, -3, 5, 2, -2, 0, -3, -2, 1, 0, -3, -1, 0, -1, -2, -1, -2],
    [-1, 0, 0, 2, -4, 2, 5, -2, 0, -3, -3, 1, -2, -3, -1, 0, -1, -3, -2, -2],
    [0, -2, 0, -1, -3, -2, -2, 6, -2, -4, -4, -2, -3, -3, -2, 0, -2, -2, -3, -3],
    [-2, 0, 1, -1, -3, 0, 0, -2, 8, -3, -3, -1, -2, -1, -2, -1, -2, -2, 2, -3],
    [-1, -3, -3, -3, -1, -3, -3, -4, -3, 4, 2, -3, 1, 0, -3, -2, -1, -3, -1, 3],
    [-1, -2, -3, -4, -1, -2, -3, -4, -3, 2, 4, -2, 2, 0, -3, -2, -1, -2, -1, 1],
    [-1, 2, 0, -1, -3, 1, 1, -2, -1, -3, -2, 5, -1, -3, -1, 0, -1, -3, -2, -2],
    [-1, -1, -2, -3, -1, 0, -2, -3, -2, 1, 2, -1, 5, 0, -2, -1, -1, -1, -1, 1],
    [-2, -3, -3, -3, -2, -3, -3, -3, -1, 0, 0, -3, 0, 6, -4, -2, -2, 1, 3, -1],
    [-1, -2, -2, -1, -3, -1, -1, -2, -2, -3, -3, -1, -2, -4, 7, -1, -1, -4, -3, -2],
    [1, -1, 1, 0, -1, 0, 0, 0, -1, -2, -2, 0, -1, -2, -1, 4, 1, -3, -2, -2],
    [0, -1, 0, -1, -1, -1, -1, -2, -2, -1, -1, -1, -1, -2, -1, 1, 5, -2, -2, 0],
    [-3, -3, -4, -4, -2, -2, -3, -2, -2, -3, -2, -3, -1, 1, -4, -3, -2, 11, 2, -3],
    [-2, -2, -2, -3, -2, -1, -2, -3, 2, -1, -1, -2, -1, 3, -3, -2, -2, 2, 7, -1],
    [0, -3, -3, -3, -1, -2, -2, -3, -3, 3, 1, -2, 1, -1, -2, -2, 0, -3, -1, 4]])
_SUB_P = np.where(np.eye(20, dtype=bool), 0.0, 2.0 ** (_B62 / 2.0))
_SUB_P /= _SUB_P.sum(axis=1, keepdims=True)
_SUB_CUM = np.cumsum(_SUB_P, axis=1)

# standard genetic code, codons in TCAG order; synonymous codons of every residue (X = any sense codon)
_BASES = "TCAG"
_CODE = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
_CODONS = [a + b + c for a in _BASES for b in _BASES for c in _BASES]
SYN = [[c for c, aa in zip(_CODONS, _CODE) if aa == AA[k]] for k in range(20)]
SYN.append([c for c, aa in zip(_CODONS, _CODE) if aa != "*"])
_COMP = str.maketrans("ACGTRYKN", "TGCAYRMN")
X_CODE = 20


def _low_complexity(rng):
    """an 8-40 residue homopolymer or period-2 / period-3 repeat (residue codes)"""
    n = int(rng.integers(8, 41))
    period = int(rng.choice([1, 2, 3]))
    unit = rng.integers(0, 20, size=period)
    return list(np.resize(unit, n))


def _substitute(rng, res, rate):
    out = []
    for a in res:
        if a < 20 and rate > 0 and rng.random() < rate:
            a = int(np.searchsorted(_SUB_CUM[a], rng.random() * _SUB_CUM[a, -1], side="right"))
            a = min(a, 19)
        out.append(int(a))
    return out


def _one_read(rng, markers, x_subjects, L):
    na = L // 3 + 3                                  # residues the read needs (prefix and trimming included)
    # ---- subject and window start
    u = rng.random()
    if u < 0.08 and len(x_subjects):                 # a window over a database X
        s = int(rng.choice(x_subjects))
        o, n = int(markers.off[s]), int(markers.subj_len[s])
        xs = np.flatnonzero(markers.res[o:o + n] == X_CODE)
        st = int(rng.choice(xs)) - int(rng.integers(0, na))
    elif u < 0.16:                                   # a short subject wholly inside the read
        short = np.flatnonzero(markers.subj_len <= na - 8)
        s = int(rng.choice(short)) if len(short) else int(rng.integers(0, markers.n_subj))
        n = int(markers.subj_len[s])
        st = -int(rng.integers(1, max(2, na - n)))
    else:
        s = int(rng.integers(0, markers.n_subj))
        n = int(markers.subj_len[s])
        v = rng.random()
        if v < 0.12:
            st = -int(rng.integers(1, 25))           # starts before residue 0
        elif v < 0.24:
            st = n - na + int(rng.integers(1, 25))   # runs past the last residue
        else:
            st = int(rng.integers(0, max(1, n - na + 1)))
    o = int(markers.off[s])
    sub = markers.res[o:o + n]
    rate = float(rng.choice([0.0, 0.1, 0.2, 0.3, 0.4]))
    # ---- indels: positions along the window (in residues of the read), deletions skip subject residues
    events = {}
    for _ in range(int(rng.integers(0, 4))):
        ln = int(rng.integers(1, 21)) if rng.random() < 0.6 else int(rng.integers(12, 21))
        events[int(rng.integers(2, na - 2))] = ("ins" if rng.random() < 0.5 else "del", ln)
    res, pos, k = [], st, 0
    while len(res) < na:
        ev = events.pop(k, None)
        if ev is not None:
            if ev[0] == "ins":
                res.extend(int(x) for x in rng.integers(0, 20, size=ev[1]))
            else:
                pos += ev[1]
        res.append(int(sub[pos]) if 0 <= pos < n else int(rng.integers(0, 20)))
        pos += 1
        k += 1
    res = _substitute(rng, res[:na], rate)
    # ---- low-complexity stretch at the start, middle or end
    if rng.random() < 0.2:
        lc = _low_complexity(rng)
        where = int(rng.integers(0, 3))
        at = 0 if where == 0 else (na - len(lc)) // 2 if where == 1 else na - len(lc)
        at = max(0, at)
        res[at:at + len(lc)] = lc
        res = res[:na]
    # ---- back-translation, phase, length, strand
    dna = "".join(SYN[a][int(rng.integers(0, len(SYN[a])))] for a in res)
    prefix = "".join(_BASES[int(b)] for b in rng.integers(0, 4, size=int(rng.integers(0, 3))))
    w = rng.random()
    ln = L - int(rng.integers(1, 30)) if w < 0.03 else L + int(rng.integers(1, 7)) if w < 0.15 else L
    seq = (prefix + dna)[:ln]
    if rng.random() < 0.5:
        seq = seq[::-1].translate(_COMP)
    if rng.random() < 0.05:                          # N, IUPAC letters and lower case inside codons of the hit
        b = list(seq)
        for p in rng.integers(0, len(b), size=int(rng.integers(1, 5))):
            b[p] = str(rng.choice(["N", "R", "Y", "K", b[p].lower()]))
        seq = "".join(b)
    return seq


def homolog_reads(markers, seed, n, L, with_quals=False):
    """n reads of about L bp (see the module doc) as a ReadBatch; qualities 2..41 at offset 33 if asked for."""
    rng = np.random.default_rng([seed, L])
    x_subjects = np.unique(np.searchsorted(markers.off, np.flatnonzero(markers.res == X_CODE), side="right") - 1)
    seqs = [_one_read(rng, markers, x_subjects, L) for _ in range(n)]
    quals = None
    if with_quals:
        quals = ["".join(chr(33 + int(q)) for q in rng.integers(2, 42, size=len(s))) for s in seqs]
    return ReadBatch.from_strings(seqs, quals)
