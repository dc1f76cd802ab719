"""Host-side driver of libmcx: one MarkerSearch = one GPU context with the marker index resident.

Mirrors the seam of the reference pipeline (microbe_census.py:611-620): reads in, sampled_reads +
agg_hits out.  All computation happens in the CUDA library; this module only moves arrays.
"""
import ctypes as C

import numpy as np

from . import _lib
from .markers import Markers, min_raw_for_bits, report_floor, STAT_NAMES


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


class ReadBatch:
    """Reads as the library wants them: concatenated ASCII bases (+ qualities) and n+1 offsets."""

    def __init__(self, bases, offsets, quals=None):
        self.bases = np.ascontiguousarray(bases, dtype=np.uint8)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.quals = None if quals is None else np.ascontiguousarray(quals, dtype=np.uint8)
        self.n = len(self.offsets) - 1

    @classmethod
    def from_strings(cls, seqs, quals=None):
        offs = np.zeros(len(seqs) + 1, np.int64)
        if len(seqs):
            offs[1:] = np.cumsum([len(s) for s in seqs])
        b = np.frombuffer("".join(seqs).encode("ascii", "replace"), np.uint8) if len(seqs) else np.zeros(0, np.uint8)
        q = None
        if quals is not None:
            q = np.frombuffer("".join(quals).encode("ascii", "replace"), np.uint8) if len(quals) else np.zeros(0, np.uint8)
        return cls(b, offs, q)

    def slice(self, lo, hi):
        o = self.offsets[lo:hi + 1]
        b0, b1 = int(o[0]), int(o[-1])
        return ReadBatch(self.bases[b0:b1], o - b0, None if self.quals is None else self.quals[b0:b1])

    @property
    def nbytes(self):
        return self.bases.nbytes + self.offsets.nbytes + (0 if self.quals is None else self.quals.nbytes)


_CODE_LUT = np.full(256, 5, np.uint8)        # T C A G = 0..3 (the codon table's order), N = 4, anything else = 5
for _c, _v in ((84, 0), (67, 1), (65, 2), (71, 3), (78, 4)):
    _CODE_LUT[_c] = _v


def pinned_empty(n, dtype):
    """numpy array of n items in page-locked memory from libmcx (mcx_host_alloc); the owner object frees it."""
    lib = _lib.load()
    dt = np.dtype(dtype)
    ptr = C.c_void_p(0)
    _lib.check(lib, None, lib.mcx_host_alloc(C.byref(ptr), max(int(n), 1) * dt.itemsize))
    buf = (C.c_uint8 * (max(int(n), 1) * dt.itemsize)).from_address(ptr.value)
    arr = np.frombuffer(buf, dtype=dt, count=int(n))
    return arr, _PinnedOwner(lib, ptr)


class _PinnedOwner:
    def __init__(self, lib, ptr):
        self.lib, self.ptr = lib, ptr

    def __del__(self):
        try:
            if self.ptr:
                self.lib.mcx_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


class PackedBatch:
    """Reads in the layout they have in HBM (include/mcx.h, mcx_push_reads_packed): per read of l bases 3 * ceil(l / 32)
    uint32 words -- lo[G], hi[G], mask[G] bit-planes of the 2-bit base codes -- plus the lengths and, for FASTQ, the
    quality bytes of all reads back to back."""

    def __init__(self, packed, lengths, quals=None, n_bases=None):
        self.packed = np.ascontiguousarray(packed, dtype=np.uint32)
        self.lengths = np.ascontiguousarray(lengths, dtype=np.uint32)
        self.quals = None if quals is None else np.ascontiguousarray(quals, dtype=np.uint8)
        self.n = len(self.lengths)
        self.n_bases = int(self.lengths.sum(dtype=np.int64)) if n_bases is None else int(n_bases)
        self._owners = []

    @property
    def nbytes(self):
        return self.packed.nbytes + self.lengths.nbytes + (0 if self.quals is None else self.quals.nbytes)

    @classmethod
    def from_batch(cls, batch, pinned=False):
        """Pack an ASCII ReadBatch (numpy; the C++ reader of libmcxio packs while it parses)."""
        lens = np.diff(batch.offsets).astype(np.int64)
        n = len(lens)
        G = (lens + 31) // 32
        woff = np.zeros(n + 1, np.int64)
        np.cumsum(3 * G, out=woff[1:])
        alloc = (lambda k, dt: pinned_empty(k, dt)) if pinned else (lambda k, dt: (np.empty(k, dt), None))
        packed, o1 = alloc(int(woff[-1]), np.uint32)
        lengths, o2 = alloc(n, np.uint32)
        lengths[:] = lens
        base0 = int(batch.offsets[0]) if n else 0
        if n and (lens == lens[0]).all() and lens[0] > 0:
            L, g = int(lens[0]), int(G[0])
            out = packed.reshape(n, 3, g)
            step = max(1, (1 << 24) // max(L, 1))
            for lo_r in range(0, n, step):               # blocks keep the temporaries small
                hi_r = min(n, lo_r + step)
                code = _CODE_LUT[batch.bases[base0 + lo_r * L: base0 + hi_r * L]].reshape(hi_r - lo_r, L)
                pad = np.zeros((hi_r - lo_r, g * 32), np.uint8)
                for plane, bits in enumerate((((code & 1) & (code < 4)) | (code == 5), ((code >> 1) & 1) & (code < 4), code >= 4)):
                    pad[:, :L] = bits
                    out[lo_r:hi_r, plane, :] = np.packbits(pad.reshape(-1, g, 32), axis=-1, bitorder="little").view("<u4").reshape(-1, g)
        elif n:
            total = int(batch.offsets[-1]) - base0
            code = _CODE_LUT[batch.bases[base0: base0 + total]]
            rd = np.repeat(np.arange(n), lens)
            pos = np.arange(total, dtype=np.int64) - np.repeat(batch.offsets[:-1] - base0, lens)
            word, bit = woff[rd] + pos // 32, (pos % 32).astype(np.uint64)
            g_rd = G[rd]
            acc = np.zeros(int(woff[-1]), np.float64)
            for plane, bits in enumerate((((code & 1) & (code < 4)) | (code == 5), ((code >> 1) & 1) & (code < 4), code >= 4)):
                sel = bits.astype(bool)
                acc += np.bincount(word[sel] + plane * g_rd[sel], weights=np.left_shift(np.uint64(1), bit[sel]).astype(np.float64),
                                   minlength=len(acc))
            packed[:] = acc.astype(np.uint64).astype(np.uint32)
        quals = None
        o3 = None
        if batch.quals is not None:
            nb = int(batch.offsets[-1]) - base0 if n else 0
            quals, o3 = alloc(nb, np.uint8)
            quals[:] = batch.quals[base0: base0 + nb]
        pb = cls(packed, lengths, quals, n_bases=int(lens.sum()))
        pb._owners = [o for o in (o1, o2, o3) if o is not None]
        return pb


class SearchResult:
    def __init__(self, raw, markers, read_length):
        self.sampled_reads = int(raw.sampled_reads)
        self.too_short = int(raw.too_short)
        self.low_qual = int(raw.low_qual)
        self.dups = int(raw.dups)
        self.reads_with_hits = int(raw.reads_with_hits)
        self.reads_classified = int(raw.reads_classified)
        self.n_hsp = int(raw.n_hsp)
        self.n_seed_hits = int(raw.n_seed_hits)
        self.n_gapped = int(raw.n_gapped)
        self.gapped_cells = int(raw.gapped_cells)
        self.n_capped_reads = int(raw.n_capped_reads)
        self.fam_hits = np.array(raw.fam_hits, np.int64)
        self.fam_aln = np.array(raw.fam_aln, np.int64)
        self.aln_by_len = np.array(raw.aln_by_len, np.int64).reshape(_lib.N_FAM, _lib.LEN_BINS)
        self._markers = markers
        self.read_length = read_length

    def counts_vector(self):
        """Everything additive, as one int64 vector (what a multi-GPU run all-reduces)."""
        head = np.array([self.sampled_reads, self.too_short, self.low_qual, self.dups, self.reads_with_hits,
                         self.reads_classified, self.n_hsp, self.n_seed_hits, self.n_gapped, self.gapped_cells,
                         self.n_capped_reads], np.int64)
        return np.concatenate([head, self.fam_hits, self.fam_aln, self.aln_by_len.ravel()])

    def load_counts_vector(self, v):
        v = np.asarray(v, np.int64)
        (self.sampled_reads, self.too_short, self.low_qual, self.dups, self.reads_with_hits, self.reads_classified,
         self.n_hsp, self.n_seed_hits, self.n_gapped, self.gapped_cells, self.n_capped_reads) = (int(x) for x in v[:11])
        nf = _lib.N_FAM
        self.fam_hits = v[11:11 + nf].copy()
        self.fam_aln = v[11 + nf:11 + 2 * nf].copy()
        self.aln_by_len = v[11 + 2 * nf:].reshape(nf, _lib.LEN_BINS).copy()

    def agg_hits(self):
        """{family id: weighted count} as aggregate_hits returns it (microbe_census.py:462-472).

        `hits` families count reads, `aln` families sum alignment lengths, `cov` families sum
        aln/target_len, formed here as sum over subject lengths of (integer sum of aln)/length in
        ascending length order -- independent of read order and of the number of GPUs."""
        cut = self._markers.cutoffs(self.read_length)
        out = {}
        for f, name in enumerate(self._markers.fam_names):
            if self.fam_hits[f] == 0:
                continue
            stat = int(cut[f]["stat"])
            if stat == 0:
                out[name] = float(self.fam_hits[f])
            elif stat == 2:
                out[name] = float(self.fam_aln[f])
            else:
                total = 0.0
                row = self.aln_by_len[f]
                for ln in np.nonzero(row)[0]:
                    total += float(row[ln]) / float(ln)
                out[name] = total
        return out


class MarkerSearch:
    """GPU context: marker residues + seed index on the device, ready to search batches of reads."""

    def __init__(self, markers=None, device=0):
        self.markers = markers if isinstance(markers, Markers) else Markers(markers)
        self.lib = _lib.load()
        m = self.markers
        self._db = _lib.Db(m.n_subj, m.off.ctypes.data, m.res.ctypes.data, m.fam.ctypes.data)
        self.ctx = C.c_void_p(0)
        self.device = int(device)
        rc = self.lib.mcx_create(C.byref(self.ctx), C.byref(self._db), int(device))
        if rc != 0:
            _lib.check(self.lib, None, rc)
        try:                                     # batches of the file reader now come in page-locked memory
            from . import seqio
            seqio.use_pinned_buffers(self.lib)
        except OSError:
            pass
        self.read_length = None
        self._batch = None

    def close(self):
        if self.ctx:
            self.lib.mcx_destroy(self.ctx)
            self.ctx = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        _lib.check(self.lib, self.ctx, rc)

    def set_params(self, read_length, quality_offset=None, min_quality=-5, mean_quality=-5, max_unknown=100,
                   filter_dups=False, min_report_raw=None):
        m = self.markers
        cut = m.cutoffs(read_length)
        raws = m.raw_cutoffs(read_length)
        p = _lib.Params()
        p.read_length = int(read_length)
        p.has_quality = 0 if quality_offset is None else 1
        p.quality_offset = int(quality_offset or 0)
        p.min_quality, p.mean_quality, p.max_unknown = int(min_quality), int(mean_quality), int(max_unknown)
        p.filter_dups = 1 if filter_dups else 0
        floor = report_floor(read_length) if min_report_raw is None else int(min_report_raw)
        p.min_report_raw = min(floor, min(raws))
        for f in range(_lib.N_FAM):
            p.cut[f].min_cov = float(cut[f]["min_cov"])
            p.cut[f].max_aaid = float(cut[f]["max_aaid"])
            p.cut[f].min_raw = int(raws[f])
            p.cut[f].stat = int(cut[f]["stat"])
        self._ck(self.lib.mcx_set_params(self.ctx, C.byref(p)))
        self.read_length = int(read_length)
        self.min_report_raw = int(p.min_report_raw)

    def set_stream(self, cuda_stream):
        """Run on the caller's stream (int handle of a cudaStream_t)."""
        self._ck(self.lib.mcx_set_stream(self.ctx, C.c_void_p(int(cuda_stream))))

    def push(self, batch):
        """Queue the host -> device copy of the reads (ReadBatch = ASCII, PackedBatch = the device layout).  Nothing is
        waited for: the search consumes the reads as they arrive.  `qc()` gives the verdict counts over all pushed reads
        (and waits for all of them)."""
        self._batch = batch  # the copies are asynchronous: keep the arrays alive
        if isinstance(batch, PackedBatch):
            self._ck(self.lib.mcx_push_reads_packed(self.ctx, _ptr(batch.packed), int(batch.packed.size), _ptr(batch.lengths),
                                                    _ptr(batch.quals), int(batch.n_bases), batch.n))
        else:
            self._ck(self.lib.mcx_push_reads(self.ctx, _ptr(batch.bases), _ptr(batch.quals), _ptr(batch.offsets), batch.n))

    def push_device(self, d_bases_ptr, d_quals_ptr, d_offsets_ptr, n, total_bytes):
        """ASCII reads already in device memory"""
        self._ck(self.lib.mcx_push_reads_dev(self.ctx, C.c_void_p(d_bases_ptr), C.c_void_p(d_quals_ptr or 0),
                                             C.c_void_p(d_offsets_ptr), int(n), int(total_bytes)))

    def push_packed_device(self, d_packed_ptr, n_words, d_lengths_ptr, d_quals_ptr, n_bases, n):
        """packed reads already in device memory (the buffers stay the caller's)"""
        self._ck(self.lib.mcx_push_reads_packed_dev(self.ctx, C.c_void_p(d_packed_ptr), int(n_words), C.c_void_p(d_lengths_ptr),
                                                    C.c_void_p(d_quals_ptr or 0), int(n_bases), int(n)))

    def qc(self):
        q = _lib.Qc()
        self._ck(self.lib.mcx_qc_counts(self.ctx, C.byref(q)))
        return {"n_reads": q.n_reads, "kept": q.kept, "too_short": q.too_short, "low_qual": q.low_qual, "dups": q.dups}

    def qc_export(self, with_fingerprints=False):
        """(codes uint8[n], fingerprints uint64[n, 2] or None) of the pushed reads"""
        n = self.qc()["n_reads"]
        code = np.zeros(max(n, 1), np.uint8)
        fp = np.zeros((max(n, 1), 2), np.uint64) if with_fingerprints else None
        self._ck(self.lib.mcx_qc_export(self.ctx, _ptr(code), _ptr(fp)))
        return code[:n], (None if fp is None else fp[:n])

    def qc_device(self, with_fingerprints=True):
        """(pointer to the n verdict bytes, pointer to the n 24-byte fingerprint records or 0, n) in device memory"""
        dc, df, n = C.c_void_p(0), C.c_void_p(0), C.c_int64(0)
        self._ck(self.lib.mcx_qc_device(self.ctx, C.byref(dc), C.byref(df) if with_fingerprints else None, C.byref(n)))
        return dc.value or 0, df.value or 0, n.value

    def qc_refresh(self):
        """rebuild the kept list after the verdicts were rewritten in device memory"""
        self._ck(self.lib.mcx_qc_refresh(self.ctx))
        return self.qc()

    def dedup_reset(self):
        """forget the fingerprints kept by earlier pushes (start of a run with -d)"""
        self._ck(self.lib.mcx_dedup_reset(self.ctx))

    def dedup_begin(self, world, first_index):
        """-d across ranks, step 1 (mcx_dedup_begin): (device pointer to the records grouped by owner rank, records per owner)"""
        d_send = C.c_void_p(0)
        counts = (C.c_int64 * int(world))()
        self._ck(self.lib.mcx_dedup_begin(self.ctx, int(world), int(first_index), C.byref(d_send), counts))
        return d_send.value or 0, [int(c) for c in counts]

    def dedup_owner(self, d_recv_ptr, m):
        """step 2 (mcx_dedup_owner): device pointer to the m mark bytes of the records this rank owns"""
        d_marks = C.c_void_p(0)
        self._ck(self.lib.mcx_dedup_owner(self.ctx, C.c_void_p(d_recv_ptr or 0), int(m), C.byref(d_marks)))
        return d_marks.value or 0

    def dedup_finish(self, d_marks_back_ptr):
        """step 3 (mcx_dedup_finish): verdicts rewritten, counters of all pushed reads"""
        self._ck(self.lib.mcx_dedup_finish(self.ctx, C.c_void_p(d_marks_back_ptr or 0)))
        return self.qc()

    def qc_import(self, code):
        code = np.ascontiguousarray(code, np.uint8)
        self._ck(self.lib.mcx_qc_import(self.ctx, _ptr(code)))
        return self.qc()

    def search(self, quota=-1):
        self._ck(self.lib.mcx_search(self.ctx, -1 if quota is None else int(quota)))
        raw = _lib.Result()
        self._ck(self.lib.mcx_result_get(self.ctx, C.byref(raw)))
        return SearchResult(raw, self.markers, self.read_length)

    def hits(self):
        n = C.c_int64(0)
        self._ck(self.lib.mcx_get_hits(self.ctx, C.c_void_p(0), 0, C.byref(n)))
        arr = np.zeros((max(n.value, 1), 12), np.int32)
        self._ck(self.lib.mcx_get_hits(self.ctx, _ptr(arr), n.value, C.byref(n)))
        return arr[:n.value]

    def classified(self, n):
        out = np.full(int(n), -1, np.int32)
        self._ck(self.lib.mcx_get_classified(self.ctx, _ptr(out), int(n)))
        return out

    def dpx_peak(self):
        """1e9 DPX thread-instructions per second this GPU issues (viaddmax_s32 / vimax3_s32_relu microbenchmark)."""
        v = C.c_double(0.0)
        self._ck(self.lib.mcx_dpx_peak(self.ctx, C.byref(v)))
        return v.value

    def l2_peak(self):
        """1e9 random 4-byte loads (32-byte L2 sectors) per second over the 32 MB presence filter (microbenchmark)."""
        v = C.c_double(0.0)
        self._ck(self.lib.mcx_l2_peak(self.ctx, C.byref(v)))
        return v.value

    def search_counters(self):
        """queue lengths of the last search (include/mcx.h mcx_search_counters)"""
        out = (C.c_int64 * 8)()
        self._ck(self.lib.mcx_search_counters(self.ctx, C.byref(out)))
        return dict(zip(("seg_frames", "filter_passes", "candidates", "seeds", "ungapped_hsps", "gap_dp_extensions",
                         "gap_wide_extensions"), (int(x) for x in out[:7])))

    def timings(self):
        ms = (C.c_float * 12)()
        launches = C.c_int64(0)
        self._ck(self.lib.mcx_timings(self.ctx, C.byref(ms), C.byref(launches)))
        names = ("h2d", "qc", "probe", "gapped", "sort", "classify", "d2h", "extend", "frames", "seg", "k_qc", "dedupe")
        out = {k: float(ms[i]) for i, k in enumerate(names)}
        det = (C.c_float * 4)()
        self._ck(self.lib.mcx_timings_detail(self.ctx, C.byref(det)))
        out.update({k: float(det[i]) for i, k in enumerate(("k_probe", "k_resolve", "k_seed", "k_walk"))})
        return out, int(launches.value)


HIT_FIELDS = ("read", "subject", "frame", "score", "aln", "ident", "mism", "gapo", "q0", "q1", "t0", "t1")


def dna_coords(L, frame, q0, q1):
    """aa range (0-based inclusive) on a frame -> 1-based q.start/q.end on the read, as RAPsearch2 prints them."""
    a0, a1 = q0 + 1, q1 + 1
    if frame < 3:
        return 3 * (a0 - 1) + frame + 1, 3 * a1 + frame
    o = frame - 3
    return L - o - 3 * (a0 - 1), L - o - 3 * a1 + 1


def format_m8(hits, markers, read_length, read_names=None):
    """m8 lines in RAPsearch2's layout (the file search_seqs leaves for parse_rapsearch, mc.py:391-398): -b 0
    subject coordinates, identity with six significant digits, log10 E and bit score with two decimals."""
    from .markers import bits_printed, log10_evalue_printed
    lines = []
    for h in hits:
        d = dict(zip(HIT_FIELDS, (int(x) for x in h)))
        qs, qe = dna_coords(read_length, d["frame"], d["q0"], d["q1"])
        name = str(d["read"]) if read_names is None else read_names[d["read"]]
        lines.append("%s\t%s\t%g\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%s\t%s" % (
            name, markers.names[d["subject"]], 100.0 * d["ident"] / d["aln"], d["aln"], d["mism"], d["gapo"],
            qs, qe, d["t0"], d["t1"], "%g" % log10_evalue_printed(d["score"], read_length), "%g" % bits_printed(d["score"])))
    return lines
