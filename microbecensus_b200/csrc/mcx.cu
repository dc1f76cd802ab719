// mcx.cu -- libmcx.so: translated marker-gene search of MicrobeCensus on one B200 (sm_100a).
//
// One context = one GPU.  The hot path is a chain of hand-written kernels with compaction between every two stages
// whose per-item work varies (no CPU fallback anywhere):
//
//   k_qc          read QC on the 2-bit packed reads   mc.py:265-279, 342-356     one warp per read, HBM-bound
//   k_fingerprint / k_fp_keys / k_mark_dups   -d: 128-bit strand-canonical fingerprints, radix sort, marks (mc.py:333-355);
//                 mcx_dedup_begin / _owner / _finish are the same steps split around the cross-GPU exchange
//   k_frames      6-frame translation (RAPsearch2 BuildQHash) + the verdict of every 12-window against both SEG cut-offs
//                 one thread per (read, frame); frames go to a global frame store, frames with a low window to the SEG queue
//   k_seg         full SEG (Seg::segseq / Seg::trim) for the frames with such a window (34 % at 150 bp), one warp per frame,
//                 frames drawn from the queue by resident blocks
//   k_probe       murphy10 seed words against the presence filter (Searching / FindSeeds): two filter blocks per window,
//                 passing words queued
//   k_resolve     word tables + posting lists of the queued words, one lane per word; every posting that survives the
//                 first rejection test is queued as a candidate
//   k_seed        seed growth and acceptance (ExtendSeq2Set), one thread per candidate, residues from register windows
//   k_walk        ungapped X-drop walks (AlignFwd / AlignBwd), one thread per accepted seed; duplicate HSPs dropped
//   k_gap_list / k_gap_screen / k_gap_dp / k_gap_trace / k_gap_finish   gapped X-drop extension (AlignSeqs / AlignGapped /
//                 CalRes): work list sorted by size, screening pass (DPX) for all extensions, complete DP + traceback
//                 for those that gain, HSP records + sort keys; k_gap_dir: fallback for windows wider than the ring
//   k_cls_groups / _cap / _cap_apply / _filter / _sum   HSP de-duplication per (read, subject), the 500-line cap, the
//                 three cutoffs, best hit per read and the per-family integer sums    mc.py:400-472
// plus CUB scans/sorts for compaction and ordering.  mc.py = /root/reference/microbe_census/
// microbe_census.py; RAPsearch2 = the v2.15 binary it runs at mc.py:375 (behaviour pinned in DESIGN.md
// and restated independently by oracle/mc_oracle.c, against which tests/ check every stage bit for bit).
#include "../../include/mcx.h"
#include "mcx_tables.h"

#include <cuda_runtime.h>
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <climits>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

using namespace mcx;

// ------------------------------------------------------------------------------------------------
// device-side constants
// ------------------------------------------------------------------------------------------------
__constant__ mcx_cutoff c_cut[MCX_N_FAM];
// Look-up tables live in global memory and are staged in shared memory by the blocks that index them per lane:
// constant-bank reads with a per-lane index are serialised (k_extend once spent 11 % of its time filling its
// BLOSUM62 copy from a __constant__ array, k_frames 11 % on the codon table).
__device__ __align__(16) int8_t g_blosum[21 * 32];
__device__ double g_lnfac[256];       // ln(i!)
__device__ double g_ln20[256];        // i * ln 20

// murphy10 letters of residues 0..15 / 16..20, one nibble each (built from MURPHY10 at compile time)
constexpr unsigned long long pack_m10(int first, int last) {
    unsigned long long v = 0;
    for (int a = first; a <= last; ++a) v |= (unsigned long long)MURPHY10_CE[a] << (4 * (a - first));
    return v;
}
constexpr unsigned long long M10_LO = pack_m10(0, 15);
constexpr unsigned long long M10_HI = pack_m10(16, 20);

__device__ __forceinline__ int red_of(int a) {
    return a < 16 ? (int)((M10_LO >> (4 * a)) & 15) : (int)((M10_HI >> (4 * (a - 16))) & 15);
}
__device__ __forceinline__ bool red_eq(int a, int b) {
    int x = red_of(a);
    return x < 10 && x == red_of(b);
}

struct DevDB {
    int n_subj;
    const int32_t *off;
    const uint8_t *res;
    const uint8_t *fam;
    const uint2 *htab;             // N_PAT open-addressing tables of 2^hbits slots, one after the other: x = word code
    int hbits;                     // (0xffffffff = empty), y = 25-bit posting start | 7-bit (count - 1)
    const uint32_t *post;          // (subject << 11 | position), bits 26..29 = a murphy10 letter of the subject (build_index), bit 31 = last posting of the word
    const uint4 *filt_a;           // presence filter (below): 2^FILT_BITS blocks for the exact word and the wildcards at 3 / 4,
    const uint2 *filt_b;           // and as many for the wildcards at 5 / 6; absorbs ~96 % of the probes in L2
};

// presence filter, blocked by what the five words of a window have in common.  All five patterns fix the letters
// 0,1,2,7,8; the exact word and the wildcards at 3 / 4 also share 5,6 (group A, 7 letters), the wildcards at 5 / 6 share
// 3,4,9 (group B, 8 letters).  The block address is a hash of the group's shared letters, so ONE 16-byte load answers
// the three group-A words of a window and ONE 8-byte load the two group-B words: two L1 / L2 requests per lane and
// window instead of five (the loop was bound by the rate of scattered requests, not by bytes; profiles/).  Inside a
// block every pattern owns its word(s) -- exact: one bit in word 0 and one in word 3; wildcard 3 / 4: two bits of word
// 1 / 2; wildcard 5 / 6: two bits of word 0 / 1 of the B block -- so no lane selects a register by a computed index.
// Bit positions come from the letters outside the shared set, the pattern and the address hash.  Measured on the
// marker set with translated synthetic reads (6.0 M distinct words): 1.2 % false positives at 2^21 blocks (the
// one-word-per-key filter before: 1.3 %), 2.1 % at 2^20.  The filter only ever says "maybe": results cannot change.
#ifndef MCX_FILT_BITS
#define MCX_FILT_BITS 21
#endif
constexpr int FILT_BITS = MCX_FILT_BITS;       // log2(blocks) of each of the two arrays: 2^21 x (16 + 8) bytes = 48 MB
// `lo` = reduced letters 0..7 of the window as nibbles, `hi` = letters 8, 9
__host__ __device__ __forceinline__ uint32_t filt_hash_a(uint32_t lo, uint32_t hi) {
    uint32_t h = (lo & 0xFFF00FFFu) * 0x9E3779B1u; h ^= h >> 15;
    h = (h + (hi & 0xFu) * 0x85EBCA77u) * 0xC2B2AE3Du; h ^= h >> 13;
    return h;
}
__host__ __device__ __forceinline__ uint32_t filt_hash_b(uint32_t lo, uint32_t hi) {
    uint32_t h = (lo & 0xF00FFFFFu) * 0x9E3779B1u; h ^= h >> 15;
    h = (h + (hi & 0xFFu) * 0x85EBCA77u + 0x68E31DA4u) * 0xC2B2AE3Du; h ^= h >> 13;
    return h;
}
__host__ __device__ __forceinline__ uint32_t filt_block(uint32_t h) { return h >> (32 - FILT_BITS); }
// the letters of pattern p that are not in its group's shared set
__host__ __device__ __forceinline__ uint32_t filt_free(int p, uint32_t lo, uint32_t hi) {
    return p == 0 ? (lo >> 12) & 0xFFu                          // letters 3, 4
         : p == 1 ? ((lo >> 16) & 0xFu) | (hi & 0xF0u)            // 4, 9
         : p == 2 ? ((lo >> 12) & 0xFu) | (hi & 0xF0u)            // 3, 9
         : p == 3 ? (lo >> 24) & 0xFu                             // 6
                  : (lo >> 20) & 0xFu;                            // 5
}
__host__ __device__ __forceinline__ void filt_bits(int p, uint32_t lo, uint32_t hi, uint32_t h, uint32_t &b1, uint32_t &b2) {
    const uint32_t x = ((filt_free(p, lo, hi) | ((uint32_t)(p + 1) << 8)) ^ (h << 11)) * 0x2C1B3C6Du;   // one round is enough: 1.2 % false positives, as with two
    b1 = 1u << (x >> 27); b2 = 1u << ((x >> 22) & 31u);
}

struct Surv {                      // ungapped HSP that reached the report floor
    int32_t read;
    int subject, frame, q0, q1, ident, t0, score;
    uint32_t gframe;               // row of the frame store (within the chunk the survivor came from, < 2^24)
};
// in memory: 16 bytes, one 128-bit access.  x read | y gframe(24) ident(8) | z subject(15) t0(11) frame(3) | w q0(8) q1(8) score(16)
__device__ __forceinline__ uint4 surv_pack(const Surv &v) {
    uint4 p;
    p.x = (uint32_t)v.read; p.y = v.gframe | ((uint32_t)v.ident << 24);
    p.z = (uint32_t)v.subject | ((uint32_t)v.t0 << 15) | ((uint32_t)v.frame << 26);
    p.w = (uint32_t)v.q0 | ((uint32_t)v.q1 << 8) | ((uint32_t)(uint16_t)(int16_t)v.score << 16);
    return p;
}
__device__ __forceinline__ Surv surv_unpack(const uint4 p) {
    Surv v;
    v.read = (int32_t)p.x; v.gframe = p.y & 0xffffffu; v.ident = (int)(p.y >> 24);
    v.subject = (int)(p.z & 0x7fffu); v.t0 = (int)((p.z >> 15) & 0x7ffu); v.frame = (int)((p.z >> 26) & 7u);
    v.q0 = (int)(p.w & 0xffu); v.q1 = (int)((p.w >> 8) & 0xffu); v.score = (int)(int16_t)(uint16_t)(p.w >> 16);
    return v;
}

struct __align__(16) SortKey {     // (read, subject, score desc, aln desc | ungapped q0, frame, q0, q1, t0, t1, ident)
    unsigned long long k1, k2;
};
struct SortKeyLess {
    __device__ __forceinline__ bool operator()(const SortKey &a, const SortKey &b) const {
        return a.k1 < b.k1 || (a.k1 == b.k1 && a.k2 < b.k2);
    }
};

// ------------------------------------------------------------------------------------------------
// frame construction: translation + SEG hard mask.  Frames live in shared memory, one row per thread
// with a stride of an odd number of 32-bit words: "every lane touches residue k of its own frame" and
// "all lanes touch consecutive residues of one frame" (cooperative extension) are both conflict-free.
// ------------------------------------------------------------------------------------------------
#define FR(k) fr[(k)]
__host__ __device__ inline int frame_stride(int maxm) { int w = (maxm + 3) / 4; return 4 * (w | 1); }

__device__ __forceinline__ int base_code(uint8_t c) {  // T C A G -> 0..3, anything else 4; branch-free
    const int idx = (c >> 1) & 3;                          // A 0, C 1, T 2, G 3 for the four upper-case letters
    const bool valid = ((0x47544341u >> (8 * idx)) & 0xffu) == (uint32_t)c;
    return valid ? (int)((0x3012u >> (4 * idx)) & 3u) : 4;
}

// SEG window test in integers.  The entropy of a window is a function of its sorted letter counts only, and for a
// fixed number of counted residues `tot` it is monotone in G = sum over letters of g(count), g(c) = c log2 c:
// H = log2 tot - G / tot.  G is kept in 2^-24 fixed point and updated as the window slides (one table value per
// residue entering or leaving); "H <= cut" becomes "G >= thr[tot]".  upload_tables() derives thr[tot] from the
// double-precision sums the reference forms (seg.c entropy(): -(c/tot) log2(c/tot), highest count first) over every
// partition of tot <= 12 and refuses to start unless the integer test separates them exactly, so the verdicts are
// those of the floating-point code and of the oracle.  (First version: nibble-packed count histogram + FP64 sum in
// descending-count order for every window with < 8 distinct letters -- 24 % of k_frames' instructions at 6 of 32
// lanes active.)
constexpr int SEG_TAB = 176;       // entries of ln(i!) / i ln 20 staged per block (window lengths <= MAX_FRAME)
struct SegTab { int dg[16]; int2 thr[16]; };    // dg[c] = g(c+1) - g(c); thr[tot] = (locut, hicut) thresholds on G
__device__ SegTab g_segtab;

struct WinG {                       // composition of a <= 12-residue window
    unsigned long long lo, hi;      // counts of letters 0..15 / 16..19, one nibble each
    int G, tot;
    __device__ __forceinline__ void clear() { lo = hi = 0; G = 0; tot = 0; }
    __device__ __forceinline__ void add(int a, const SegTab &T) {
        if (a >= 20) return;
        int c;
        if (a < 16) { c = (int)((lo >> (4 * a)) & 15); lo += 1ull << (4 * a); }
        else { c = (int)((hi >> (4 * (a - 16))) & 15); hi += 1ull << (4 * (a - 16)); }
        G += T.dg[c];
        ++tot;
    }
    __device__ __forceinline__ void sub(int a, const SegTab &T) {
        if (a >= 20) return;
        int c;
        if (a < 16) { c = (int)((lo >> (4 * a)) & 15); lo -= 1ull << (4 * a); }
        else { c = (int)((hi >> (4 * (a - 16))) & 15); hi -= 1ull << (4 * (a - 16)); }
        G -= T.dg[c - 1];
        --tot;
    }
    __device__ __forceinline__ bool low(const SegTab &T) const { return G >= T.thr[tot].x; }    // entropy <= locut
    __device__ __forceinline__ bool high(const SegTab &T) const { return G >= T.thr[tot].y; }   // entropy <= hicut
};

// seg.c getprob() = lnass + lnperm - len*ln20 from the histogram of letter counts: nc[c] = number of letters
// occurring c times.  Walking c downwards visits the counts in exactly the order of seg.c's sorted state vector,
// so the floating-point operations (and their order) are those of the reference and of the oracle.
// nc is the calling lane's column of a [count][32 lanes] byte table in shared memory (stride 32); the entries read
// are reset to zero on the way.  Subtracting ln(1!) = 0 leaves a double unchanged, so counts of one are skipped.
__device__ double seg_getprob(uint8_t *nc, int maxc, int len, const double *lnfac, const double *ln20) {
    double lnperm = lnfac[len], lnass = lnfac[20];
    int nz = 0;
    for (int c = maxc; c >= 1; --c) {
        const int n = nc[c * 32];
        if (!n) continue;
        nc[c * 32] = 0;
        if (c > 1) { const double lf = lnfac[c]; for (int r = 0; r < n; ++r) lnperm -= lf; }
        if (n > 1) lnass -= lnfac[n];
        nz += n;
    }
    if (nz > 0 && nz < 20) lnass -= lnfac[20 - nz];
    return lnass + lnperm - ln20[len];
}
// Windows of at most 20 residues: getprob() depends only on (window length, multiset of letter counts), and there are
// only 10,979 such classes.  upload_tables() evaluates every one of them on the host with the floating-point sequence
// above and stores the results in an open-addressing table keyed by (length, signature), signature = sum over the
// letters of z[count] with 21 fixed pseudo-random words (checked to be unique per class).  A window then costs one
// table value per letter present and one lookup instead of the histogram and ~20 dependent FP64 subtractions.
constexpr int SEGP_MAXLEN = 20;
constexpr int SEGP_SLOTS = 1 << 15;
struct SegProbSlot { unsigned long long key; double prob; };     // key = len << 32 | signature; ~0 = empty
__device__ SegProbSlot g_segprob[SEGP_SLOTS];
__device__ uint32_t g_segz[32];
__host__ __device__ __forceinline__ uint32_t segp_slot(unsigned long long key) {
    return (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 49) & (SEGP_SLOTS - 1);
}
__device__ __forceinline__ double seg_prob_lookup(uint32_t sig, int len) {
    const unsigned long long key = ((unsigned long long)len << 32) | sig;
    uint32_t sl = segp_slot(key);
    for (;;) {
        const SegProbSlot e = g_segprob[sl];
        if (e.key == key) return e.prob;
        sl = (sl + 1) & (SEGP_SLOTS - 1);
    }
}

// ------------------------------------------------------------------------------------------------
// Read store.  Reads live in HBM as 2-bit bases + a mask, in bit-planes of 32 bases: the record of a read of `len`
// bases is 3 G words, G = ceil(len / 32): lo[G], hi[G], mask[G].  Base code T C A G = 0..3 (bit k of lo / hi = low /
// high bit of base k's code; complement = hi flipped); a mask bit marks a base that is not an upper-case ACGT, and under
// it lo = 0 means 'N' (what mc.py:269 counts), lo = 1 any other character.  Bits past `len` are zero in all planes.
// 60 bytes per 150 bp read instead of 150 (SURVEY 8d K1: 57 B of bases + mask); qualities stay bytes (only read when
// -q / -m are active).  Host buffers arrive in this layout through mcx_push_reads_packed; ASCII pushes are packed on
// the device by k_pack_ascii, so every kernel below has one input format.
// ------------------------------------------------------------------------------------------------
struct ReadStore {
    const uint32_t *pk;            // records
    const int64_t *woff;           // n + 1 word offsets of the records
    const uint32_t *len;           // n lengths
    const uint8_t *quals;          // qualities of all reads, one byte per base, or nullptr
    const int64_t *qoff;           // n + 1 byte offsets into quals (prefix sums of len)
    int64_t qbytes;                // bytes readable at quals
};

struct GroupsOf { __host__ __device__ __forceinline__ int64_t operator()(uint32_t len) const { return 3 * (int64_t)((len + 31u) >> 5); } };
struct LenOf { __host__ __device__ __forceinline__ int64_t operator()(uint32_t len) const { return (int64_t)len; } };

__global__ void k_lens_from_offsets(const int64_t *__restrict__ offs, int64_t n, uint32_t *__restrict__ len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) len[i] = (uint32_t)(offs[i + 1] - offs[i]);
    else if (i == n) len[i] = 0;
}

// ASCII -> bit-planes, one warp per read, one base per lane and three ballots per 32 bases (compatibility path of
// mcx_push_reads / mcx_push_reads_dev; the packed pushes skip it)
__global__ void k_pack_ascii(const uint8_t *__restrict__ bases, const int64_t *__restrict__ offs, int64_t n,
                             const int64_t *__restrict__ woff, uint32_t *__restrict__ pk) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n) return;
    const int64_t b = offs[r];
    const int len = (int)(offs[r + 1] - b);
    const int G = (len + 31) >> 5;
    uint32_t *rec = pk + woff[r];
    for (int g = 0; g < G; ++g) {
        const int k = 32 * g + lane;
        int lo = 0, hi = 0, mk = 0;
        if (k < len) {
            const uint8_t c = bases[b + k];
            const int code = base_code(c);
            if (code < 4) { lo = code & 1; hi = code >> 1; }
            else { mk = 1; lo = (c != 'N'); }
        }
        const uint32_t wl = __ballot_sync(0xffffffffu, lo), wh = __ballot_sync(0xffffffffu, hi), wm = __ballot_sync(0xffffffffu, mk);
        if (lane == 0) { rec[g] = wl; rec[G + g] = wh; rec[2 * G + g] = wm; }
    }
}

// ------------------------------------------------------------------------------------------------
// K1: read QC (mc.py:342 too short on the untrimmed length; mc.py:265-279 on seq[:L], qual[:L]).
// Eight lanes per read.  Unknown bases: popcount of mask & ~lo & ~hi over the first L bases.  Qualities: the L bytes
// of a read are fetched as aligned 128-bit pieces (a warp request = the contiguous qualities of its four reads), summed
// with dp4a and minimised with the per-byte SIMD minimum; the bytes of a piece outside [start, start + L) are blanked.
// HBM-bound: 4 ceil(L/32) * 3 + L (+ 20 of lengths / offsets) bytes per read, one code byte written.
// The reference's float comparisons are exact in integers (see oracle oc_read_qc).
// codes: 0 keep, 1 too short, 2 low quality (3 duplicate: k_mark_dups; 4 = not examined)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t byte_range_mask(int lo, int hi) {      // bytes [lo, hi) of a word as 0xff, 0 <= lo, hi <= 4
    if (hi <= lo) return 0u;
    const uint32_t up = hi >= 4 ? 0xffffffffu : ((1u << (8 * hi)) - 1u);
    const uint32_t dn = lo <= 0 ? 0u : ((1u << (8 * lo)) - 1u);
    return up & ~dn;
}
__global__ void __launch_bounds__(256) k_qc(ReadStore S, int64_t r0, int64_t r1, int L, int qoff, int minq, int meanq,
                                            int maxunk, uint8_t *__restrict__ code) {
    const int64_t r = r0 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3);
    const int sub = threadIdx.x & 7;
    const bool live = r < r1;
    const int len = live ? (int)S.len[r] : 0;
    const bool ok = live && len >= L;
    int nN = 0;
    uint32_t sum = 0, mn = 0xffffffffu;
    if (ok) {
        const int G = (len + 31) >> 5, GL = (L + 31) >> 5;
        const uint32_t *__restrict__ rec = S.pk + S.woff[r];
        for (int g = sub; g < GL; g += 8) {
            uint32_t m = __ldg(rec + 2 * G + g);
            if (m) {
                if (32 * g + 32 > L) m &= (1u << (L - 32 * g)) - 1u;
                nN += __popc(m & ~__ldg(rec + g) & ~__ldg(rec + G + g));
            }
        }
        if (S.quals) {
            const int64_t start = S.qoff[r], end = start + L;
            for (int64_t p = (start & ~15ll) + 16 * sub; p < end; p += 128) {
                if (p >= start && p + 16 <= end) {
                    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(S.quals + p));
                    sum = __dp4a(v.x, 0x01010101u, sum); sum = __dp4a(v.y, 0x01010101u, sum);
                    sum = __dp4a(v.z, 0x01010101u, sum); sum = __dp4a(v.w, 0x01010101u, sum);
                    mn = __vminu4(mn, __vminu4(__vminu4(v.x, v.y), __vminu4(v.z, v.w)));
                } else {
                    uint32_t w[4];
                    if (p >= 0 && p + 16 <= S.qbytes) {
                        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(S.quals + p));
                        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
                    } else {                                   // the piece sticks out of the buffer: bytes
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            w[q] = 0;
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const int64_t a = p + 4 * q + c;
                                if (a >= start && a < end) w[q] |= (uint32_t)S.quals[a] << (8 * c);
                            }
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int64_t a = p + 4 * q;
                        const uint32_t vm = byte_range_mask((int)max(start - a, (int64_t)0), (int)min(end - a, (int64_t)4));
                        sum = __dp4a(w[q] & vm, 0x01010101u, sum);
                        mn = __vminu4(mn, w[q] | ~vm);
                    }
                }
            }
        }
    }
    // the eight lanes of a read are neighbours: three butterfly steps
#pragma unroll
    for (int s = 1; s < 8; s <<= 1) {
        nN += __shfl_xor_sync(0xffffffffu, nN, s);
        sum += __shfl_xor_sync(0xffffffffu, sum, s);
        mn = __vminu4(mn, __shfl_xor_sync(0xffffffffu, mn, s));
    }
    if (live && sub == 0) {
        int c = 0;
        if (!ok) c = 1;
        else if (100 * nN > maxunk * L) c = 2;
        else if (S.quals) {
            const uint32_t m2 = __vminu4(mn, mn >> 16);
            const int minb = (int)(__vminu4(m2, m2 >> 8) & 0xffu);
            if ((int)sum - qoff * L < meanq * L || minb - qoff < minq) c = 2;
        }
        code[r] = (uint8_t)c;
    }
}

// -d (mc.py:345, 355): the reference keeps the set of whole untrimmed strings of the reads it has written and
// skips a read whose string or reverse complement is in it.  Restated with a 128-bit polynomial fingerprint that is
// canonical over strands (same definition as the oracle's oc_fingerprint): a read that is long enough is a
// duplicate iff an earlier KEPT read has the same fingerprint.  Per fingerprint group in index order: everything
// after the first kept read is a duplicate; reads before it keep their QC verdict.
struct FpKey { unsigned long long a, b; uint32_t idx; uint32_t pad; };
#define FP_B1 0x9E3779B97F4A7C15ull
#define FP_B2 0xC2B2AE3D27D4EB4Full
#define FP_LEN 0xD6E8FEB86659FD93ull
// character codes of the fingerprint: A 1, C 2, G 3, T 4 (complement = 5 - c), N 5, other 6 + (c & 0x7f).  The packed
// store does not keep which "other" character a base was; under -d the reference raises KeyError on them
// (mc.py:288), so every character that can reach the duplicate test is one of ACGTN.  Others hash as 6.
__host__ __device__ __forceinline__ unsigned long long fp_of_code(int code2, int masked, int lo) {   // base code T C A G = 0..3
    if (masked) return lo ? 6ull : 5ull;
    return code2 == 0 ? 4ull : code2 == 1 ? 2ull : code2 == 2 ? 1ull : 3ull;
}
__host__ __device__ __forceinline__ unsigned long long fp_comp(unsigned long long c) { return (c >= 1 && c <= 4) ? 5 - c : c; }
// Four bases at a time: the forward hash is a Horner scheme from the left, f = f B^4 + TF[nibbles], the hash of the
// reverse complement a Horner scheme from the right, r = r B^4 + TR[nibbles]; TF / TR hold the contribution of every
// combination of four unmasked bases, indexed by (hi nibble << 4 | lo nibble).  One thread per read; groups with a
// masked base and the ragged last nibble go base by base.
struct FpTab { unsigned long long f1[256], f2[256], r1[256], r2[256]; };
__device__ FpTab g_fptab;
__global__ void __launch_bounds__(128) k_fingerprint(ReadStore S, int64_t n, FpKey *__restrict__ keys) {
    __shared__ FpTab T;
    for (int k = threadIdx.x; k < (int)(sizeof(FpTab) / 8); k += 128) reinterpret_cast<unsigned long long *>(&T)[k] = reinterpret_cast<const unsigned long long *>(&g_fptab)[k];
    __syncthreads();
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int len = (int)S.len[r];
    const int G = (len + 31) >> 5;
    const uint32_t *__restrict__ rec = S.pk + S.woff[r];
    constexpr unsigned long long B1_4 = FP_B1 * FP_B1 * FP_B1 * FP_B1, B2_4 = FP_B2 * FP_B2 * FP_B2 * FP_B2;
    unsigned long long f1 = 0, f2 = 0, r1 = 0, r2 = 0;
    for (int g = 0; g < G; ++g) {                               // forward
        const uint32_t lo = __ldg(rec + g), hi = __ldg(rec + G + g), m = __ldg(rec + 2 * G + g);
        const int nb = min(32, len - 32 * g);
        int k = 0;
        if (m == 0)
            for (; k + 4 <= nb; k += 4) {
                const uint32_t ix = (((hi >> k) & 15u) << 4) | ((lo >> k) & 15u);
                f1 = f1 * B1_4 + T.f1[ix]; f2 = f2 * B2_4 + T.f2[ix];
            }
        for (; k < nb; ++k) {
            const unsigned long long c = fp_of_code((int)(((hi >> k) & 1u) << 1 | ((lo >> k) & 1u)), (int)((m >> k) & 1u), (int)((lo >> k) & 1u));
            f1 = f1 * FP_B1 + c; f2 = f2 * FP_B2 + c;
        }
    }
    for (int g = G - 1; g >= 0; --g) {                          // reverse complement, from the last base down
        const uint32_t lo = __ldg(rec + g), hi = __ldg(rec + G + g), m = __ldg(rec + 2 * G + g);
        const int nb = min(32, len - 32 * g);
        int k = nb;
        if (m == 0) {
            for (; k & 3; --k) {
                const unsigned long long c = fp_comp(fp_of_code((int)(((hi >> (k - 1)) & 1u) << 1 | ((lo >> (k - 1)) & 1u)), 0, 0));
                r1 = r1 * FP_B1 + c; r2 = r2 * FP_B2 + c;
            }
            for (; k >= 4; k -= 4) {
                const uint32_t ix = (((hi >> (k - 4)) & 15u) << 4) | ((lo >> (k - 4)) & 15u);
                r1 = r1 * B1_4 + T.r1[ix]; r2 = r2 * B2_4 + T.r2[ix];
            }
        } else
            for (; k > 0; --k) {
                const unsigned long long c = fp_comp(fp_of_code((int)(((hi >> (k - 1)) & 1u) << 1 | ((lo >> (k - 1)) & 1u)), (int)((m >> (k - 1)) & 1u), (int)((lo >> (k - 1)) & 1u)));
                r1 = r1 * FP_B1 + c; r2 = r2 * FP_B2 + c;
            }
    }
    f1 += (unsigned long long)len * FP_LEN; r1 += (unsigned long long)len * FP_LEN;
    FpKey k;
    if (f1 < r1 || (f1 == r1 && f2 <= r2)) { k.a = f1; k.b = f2; } else { k.a = r1; k.b = r2; }
    k.idx = (uint32_t)r; k.pad = 0;
    keys[r] = k;
}
// Streamed -d: reads arrive in several pushes (batches of a large file), and a read is a duplicate of any KEPT read of an
// earlier push as well (mc.py:345 keeps one set for the whole run).  The context therefore keeps the fingerprints of the
// reads it has kept so far (`store`, 16 bytes per read); they enter the sort next to the reads of the push -- entries with
// bit 31 of the index set -- and a fingerprint group that holds one has its keeper already: every read of the push in it
// is a duplicate.  mcx_dedup_reset empties the store (start of a run).
struct FpStore { const unsigned long long *a, *b; };
constexpr uint32_t FP_STORED = 0x80000000u;
__device__ __forceinline__ void fp_of_entry(uint32_t v, const FpKey *__restrict__ fp, const FpStore &S, unsigned long long &a, unsigned long long &b) {
    if (v & FP_STORED) { a = S.a[v & ~FP_STORED]; b = S.b[v & ~FP_STORED]; }
    else { a = fp[v].a; b = fp[v].b; }
}
// sort input of the duplicate test: (a, read index) of every read, in read order, then the stored fingerprints
__global__ void k_fp_keys(const FpKey *__restrict__ fp, int64_t n, FpStore S, int64_t n_store, unsigned long long *__restrict__ ka, uint32_t *__restrict__ vi) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) { ka[r] = fp[r].a; vi[r] = (uint32_t)r; }
    else if (r < n + n_store) { ka[r] = S.a[r - n]; vi[r] = FP_STORED | (uint32_t)(r - n); }
}
// One thread per run of equal sort key (the upper FP_SORT_BITS of `a`) in the sorted list.  Inside a run the reads are
// grouped by their full fingerprint (runs of more than one fingerprint are a once-in-a-billion event, handled all the
// same): the first QC-passing read of a group -- smallest index -- stays, every other long-enough read of the group
// behind it is a duplicate; if the group holds a stored fingerprint, every long-enough read of it is.  Too-short reads
// are decided before the duplicate test (mc.py:342) and skipped.
constexpr int FP_SORT_BITS = 48;
__global__ void k_mark_dups(const unsigned long long *__restrict__ ka, const uint32_t *__restrict__ vi,
                            const FpKey *__restrict__ fp, FpStore S, int64_t n, uint8_t *__restrict__ code) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    const unsigned long long key = ka[p] >> (64 - FP_SORT_BITS);
    if (p > 0 && (ka[p - 1] >> (64 - FP_SORT_BITS)) == key) return;      // not the first of its run
    int64_t e = p + 1;
    while (e < n && (ka[e] >> (64 - FP_SORT_BITS)) == key) ++e;
    if (e == p + 1) return;
    for (int64_t s = p; s < e; ++s) {
        unsigned long long sa, sb, qa, qb;
        fp_of_entry(vi[s], fp, S, sa, sb);
        bool first = true;
        for (int64_t q = p; q < s; ++q) { fp_of_entry(vi[q], fp, S, qa, qb); if (qa == sa && qb == sb) { first = false; break; } }
        if (!first) continue;
        bool stored = false;
        uint32_t keeper = 0xffffffffu;                        // smallest index among the group's reads that pass QC
        for (int64_t q = s; q < e; ++q) {
            const uint32_t i = vi[q];
            if (q > s) { fp_of_entry(i, fp, S, qa, qb); if (qa != sa || qb != sb) continue; }
            if (i & FP_STORED) stored = true;
            else if (code[i] == 0 && i < keeper) keeper = i;
        }
        if (!stored && keeper == 0xffffffffu) continue;
        for (int64_t q = s; q < e; ++q) {
            const uint32_t i = vi[q];
            if (i & FP_STORED) continue;
            if (q > s) { fp_of_entry(i, fp, S, qa, qb); if (qa != sa || qb != sb) continue; }
            if ((stored || i > keeper) && code[i] != 1) code[i] = 3;
        }
    }
}
// the kept reads of a push join the store (reads [0, upto): the reads examined by the search)
__global__ void k_store_append(const FpKey *__restrict__ fp, const uint8_t *__restrict__ code, int64_t upto,
                               unsigned long long *__restrict__ sa, unsigned long long *__restrict__ sb, unsigned long long *n_store) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool take = r < upto && code[r] == 0;
    const uint32_t bm = __ballot_sync(0xffffffffu, take);
    if (!bm) return;
    const int lane = threadIdx.x & 31;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(n_store, (unsigned long long)__popc(bm));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (take) { const unsigned long long o = base + __popc(bm & ((1u << lane) - 1)); sa[o] = fp[r].a; sb[o] = fp[r].b; }
}

// counts of codes 0..3 among reads [0, upto)
__global__ void k_count_codes(const uint8_t *__restrict__ code, int64_t upto, unsigned long long *__restrict__ cnt) {
    __shared__ unsigned int s[4];
    if (threadIdx.x < 4) s[threadIdx.x] = 0;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < upto; i += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&s[code[i] & 3], 1u);
    __syncthreads();
    if (threadIdx.x < 4 && s[threadIdx.x]) atomicAdd(&cnt[threadIdx.x], (unsigned long long)s[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------
// K2: seeds + ungapped extension.  One thread per (kept read, frame).
// ------------------------------------------------------------------------------------------------
// K2a: one thread per (kept read, frame): translate, test every 12-window against the SEG cut-offs and write the
// frame to the global frame store (each warp copies its 32 rows as words).  Frames holding a low-entropy window
// (a few per cent) are queued for k_seg instead of running the irregular SEG code with one lane alive.
struct FrameArgs {
    ReadStore S;
    const int32_t *kept;
    int64_t first;                 // kept[first ...] are the reads of this launch
    const unsigned long long *n_search;   // how many (device counter: the launch is sized for the largest possible chunk)
    int L;
    uint8_t *frames;               // rows of fstride bytes, one per (read, frame)
    uint32_t *segq;                // frames that need the full SEG
    unsigned long long *n_segq;
    uint32_t *segm;                // per queued frame: nwr words "window start k is at or below locut", then nwr words for hicut
    int nwr;                       // words per mask = ceil(number of 12-windows of the longest frame / 32), <= 6
};

// Translation goes through a 2 x 125-entry table in shared memory indexed by three base codes (T C A G = 0..3,
// anything else 4 -> '.'), one half per strand: the reverse frames walk the read backwards and the table holds the
// codon of the complemented bases, so both strands share one code path and no lane tests for invalid bases.  The
// block first decodes the bases of its NT/6 reads into shared memory once (each base is used by all six frames).
__device__ uint8_t g_codon_lut[256];

template <int NT>
__global__ void __launch_bounds__(NT) k_frames(FrameArgs A, int fstride) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int RPB = NT / 6;                                  // reads per block
    SegTab *s_tab = reinterpret_cast<SegTab *>(smem);
    uint8_t *s_lut = smem + sizeof(SegTab);                      // 256 bytes
    uint8_t *s_aa = s_lut + 256;                                 // NT rows of fstride bytes
    uint8_t *s_code = s_aa + NT * fstride;                       // RPB reads of L base codes
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = A.L, nwr = A.nwr;
    uint32_t *wm = reinterpret_cast<uint32_t *>(s_code + ((RPB * L + 3) & ~3)) + tid;   // [2 * nwr][NT] window masks, this thread's column
    for (int k = tid; k < (int)(sizeof(SegTab) / 4); k += NT) reinterpret_cast<uint32_t *>(s_tab)[k] = reinterpret_cast<const uint32_t *>(&g_segtab)[k];
    for (int k = tid; k < 64; k += NT) reinterpret_cast<uint32_t *>(s_lut)[k] = reinterpret_cast<const uint32_t *>(g_codon_lut)[k];
    for (int k = tid; k < NT * fstride / 4; k += NT) reinterpret_cast<uint32_t *>(s_aa)[k] = 0x14141414u;  // AA_STOP
    const int64_t read0 = (int64_t)blockIdx.x * RPB;
    const int64_t n_search = (int64_t)*A.n_search;
    if (read0 >= n_search) return;
    for (int r = warp; r < RPB; r += NT / 32) {
        if (read0 + r >= n_search) break;
        const int64_t rd = A.kept[A.first + read0 + r];
        const int G = (int)((A.S.len[rd] + 31u) >> 5);
        const uint32_t *__restrict__ rec = A.S.pk + A.S.woff[rd];
        for (int k = lane; k < L; k += 32) {                   // the three plane words of a group are the same for the warp
            const int g = k >> 5;
            const uint32_t lo = __ldg(rec + g) >> lane, hi = __ldg(rec + G + g) >> lane, mk = __ldg(rec + 2 * G + g) >> lane;
            s_code[r * L + k] = (mk & 1u) ? (uint8_t)4 : (uint8_t)(((hi & 1u) << 1) | (lo & 1u));
        }
    }
    __syncthreads();
    const int64_t g = (int64_t)blockIdx.x * NT + tid;          // frame row within this launch
    const int r = tid / 6, frame = tid - r * 6;
    uint8_t *fr = s_aa + tid * fstride;
    bool trig = false;
    if (read0 + r < n_search) {
        const int o = frame % 3, m = (L - o) / 3;
        const bool rev = frame >= 3;
        const int step = rev ? -1 : 1;
        const uint8_t *cd = s_code + r * L + (rev ? L - 1 - o : o);
        const uint8_t *lut = s_lut + (rev ? 125 : 0);
        for (int k = 0; k < m; ++k, cd += 3 * step) fr[k] = lut[25 * cd[0] + 5 * cd[step] + cd[2 * step]];
        // does any 12-window have entropy <= locut?  (Seg::segseq only acts on frames that have one.)  The window
        // slides here at one letter out, one in per position, so the verdicts of every window against both cut-offs are
        // kept as bit masks and handed to k_seg with the queue entry (k_seg used to rebuild each window from scratch:
        // 28 % of its instructions)
        if (m >= SEG_WINDOW) {
            const SegTab &T = *s_tab;
            for (int k = 0; k < 2 * nwr; ++k) wm[k * NT] = 0;
            WinG w; w.clear();
            for (int k = 0; k < SEG_WINDOW; ++k) w.add(fr[k], T);
            uint32_t clo = 0, chi = 0;
            for (int st = 0;; ++st) {
                clo |= (uint32_t)w.low(T) << (st & 31); chi |= (uint32_t)w.high(T) << (st & 31);
                const bool last = st + SEG_WINDOW >= m;
                if ((st & 31) == 31 || last) { wm[(st >> 5) * NT] = clo; wm[(nwr + (st >> 5)) * NT] = chi; trig |= clo != 0; clo = chi = 0; }
                if (last) break;
                w.sub(fr[st], T); w.add(fr[st + SEG_WINDOW], T);
            }
        }
    }
    const uint32_t tm = __ballot_sync(0xffffffffu, trig);
    if (tm) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(A.n_segq, (unsigned long long)__popc(tm));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (trig) {
            const unsigned long long at = base + __popc(tm & ((1u << lane) - 1));
            A.segq[at] = (uint32_t)g;
            uint32_t *dm = A.segm + at * (unsigned long long)(2 * nwr);
            for (int k = 0; k < 2 * nwr; ++k) dm[k] = wm[k * NT];
        }
    }
    __syncwarp();
    const int64_t row0 = (int64_t)blockIdx.x * NT + (tid - lane);
    uint32_t *dst = reinterpret_cast<uint32_t *>(A.frames + row0 * fstride);
    const uint32_t *src = reinterpret_cast<const uint32_t *>(s_aa + (tid - lane) * fstride);
    for (int k = lane; k < 32 * fstride / 4; k += 32) dst[k] = src[k];
}

// K2a': full SEG for the queued frames, one WARP per frame; masked residues are overwritten in the frame store.
// The control flow of Seg::segseq is warp-uniform (every lane runs the same scalar code on masks held in shared
// memory); the expensive part, Seg::trim, evaluates the windows of one length in parallel, one lane per window
// start, from a prefix-count table of the segment, and takes the minimum with seg.c's scan order as tie-break
// (longer windows first, then leftmost).  First version: one thread per frame, 24 ms for 2M reads with 2 of 32
// lanes active on average (profiles/); this one keeps the warp busy.
__device__ __forceinline__ bool sbit(const uint32_t *m, int k) { return (m[k >> 5] >> (k & 31)) & 1; }
// smallest k in [from, to] whose bit is set (SET) or clear (!SET); -1 if none
template <bool SET>
__device__ __forceinline__ int next_bit(const uint32_t *m, int from, int to) {
    if (from > to) return -1;
    int w = from >> 5;
    const int wl = to >> 5;
    uint32_t x = (SET ? m[w] : ~m[w]) & (0xffffffffu << (from & 31));
    for (;;) {
        if (w == wl) x &= 0xffffffffu >> (31 - (to & 31));
        if (x) return (w << 5) + __ffs(x) - 1;
        if (w == wl) return -1;
        ++w;
        x = SET ? m[w] : ~m[w];
    }
}
// largest k in [down_to, from] whose bit is clear; -1 if none
__device__ __forceinline__ int prev_clear_bit(const uint32_t *m, int from, int down_to) {
    if (from < down_to) return -1;
    int w = from >> 5;
    const int wl = down_to >> 5;
    uint32_t x = ~m[w] & (0xffffffffu >> (31 - (from & 31)));
    for (;;) {
        if (w == wl) x &= 0xffffffffu << (down_to & 31);
        if (x) return (w << 5) + 31 - __clz(x);
        if (w == wl) return -1;
        --w;
        x = ~m[w];
    }
}

// doubles -> unsigned integers of the same order (no NaNs here)
__device__ __forceinline__ unsigned long long dkey(double x) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

__host__ __device__ inline int seg_warp_bytes(int fstride, int maxm) {   // shared memory of one warp of k_seg
    return 18 * 4 + fstride + (((maxm + 1) * 20 + 3) & ~3) + (maxm + 2) * 32;
}

constexpr int SEG_TRI = 1328;       // window numbers whose row is tabulated (segments of up to 51 residues: every frame of a 150 bp read)
__device__ void coop_trim(const uint8_t *fr, int off, int tl, uint8_t *P, uint8_t *nc, int lane, const double *lnfac,
                          const double *ln20, const uint32_t *zt, const uint8_t *tri, int &leftend, int &rightend) {
    __syncwarp();
    if (lane < 20) {                       // P[k][a] = occurrences of letter a among the first k residues
        int acc = 0;
        P[lane] = 0;
        for (int k = 0; k < tl; ++k) { acc += (fr[off + k] == lane); P[(k + 1) * 20 + lane] = (uint8_t)acc; }
    }
    __syncwarp();
    int lend = 0, rend = tl - 1, minlen = 1;
    if (tl - SEG_MAXTRIM > minlen) minlen = tl - SEG_MAXTRIM;
    unsigned long long minkey = dkey(1.0);             // seg.c: minprob = 1.0, strict <
    // windows in seg.c's scan order: length tl, tl-1, ... minlen+1, starts left to right; row d = tl - len holds
    // d + 1 windows, so window number w sits in row d with d(d+1)/2 <= w < (d+1)(d+2)/2.  32 windows per round.
    const int D = tl - minlen, NW = D * (D + 1) / 2;
    for (int base = 0; base < NW; base += 32) {
        const int w = base + lane;
        double prob = 1.0e300;
        int st = 0, len = tl;
        if (w < NW) {
            int d;
            if (w < SEG_TRI) d = tri[w];
            else {
                d = (int)((sqrtf(8.0f * (float)w + 1.0f) - 1.0f) * 0.5f);
                while (d * (d + 1) / 2 > w) --d;
                while ((d + 1) * (d + 2) / 2 <= w) ++d;
            }
            len = tl - d; st = w - d * (d + 1) / 2;
            // composition of the window = difference of two rows of the prefix table, four letters per word
            const uint32_t *w0 = reinterpret_cast<const uint32_t *>(P + st * 20), *w1 = reinterpret_cast<const uint32_t *>(P + (st + len) * 20);
            uint32_t cw[5];
#pragma unroll
            for (int q = 0; q < 5; ++q) cw[q] = w1[q] - w0[q];      // no borrow: every byte of w1 >= that of w0
            if (len <= SEGP_MAXLEN) {
                uint32_t sig = 0;
#pragma unroll
                for (int q = 0; q < 5; ++q) {
                    const uint32_t x = cw[q];
                    if (x) sig += zt[x & 0xffu] + zt[(x >> 8) & 0xffu] + zt[(x >> 16) & 0xffu] + zt[x >> 24];
                }
                prob = seg_prob_lookup(sig, len);
            } else {
                int maxc = 0;
#pragma unroll
                for (int a = 0; a < 20; ++a) {
                    const int c = (int)((cw[a >> 2] >> (8 * (a & 3))) & 0xffu);
                    if (c) { nc[c * 32]++; maxc = c > maxc ? c : maxc; }
                }
                prob = seg_getprob(nc, maxc, len, lnfac, ln20);
            }
        }
        // warp argmin with seg.c's tie-break (first window in scan order = lowest lane): the doubles are mapped to
        // integers of the same order and reduced with three redux / ballot steps instead of five shuffle rounds
        const unsigned long long key = dkey(prob);
        const uint32_t khi = (uint32_t)(key >> 32), klo = (uint32_t)key;
        const uint32_t mh = __reduce_min_sync(0xffffffffu, khi);
        const uint32_t ml = __reduce_min_sync(0xffffffffu, khi == mh ? klo : 0xffffffffu);
        const int bl = __ffs(__ballot_sync(0xffffffffu, khi == mh && klo == ml)) - 1;
        const unsigned long long best = ((unsigned long long)mh << 32) | ml;
        if (best < minkey) {
            minkey = best;
            lend = __shfl_sync(0xffffffffu, st, bl);
            rend = __shfl_sync(0xffffffffu, len, bl) + lend - 1;
        }
    }
    rightend -= (tl - rend - 1);
    leftend += lend;
}

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) k_seg(uint8_t *frames, int fstride, int L, const uint32_t *__restrict__ segq,
                                                    const uint32_t *__restrict__ segm, int nwr,
                                                    const unsigned long long *n_queued, int maxm, unsigned int *work) {
    const int64_t n = (int64_t)*n_queued;      // device-side count: no host round trip between k_frames and this launch
    if ((int64_t)blockIdx.x * WARPS >= n) return;
    extern __shared__ __align__(16) uint8_t smem[];
    double *s_lnfac = reinterpret_cast<double *>(smem);        // [SEG_TAB] ln(i!)
    double *s_ln20 = s_lnfac + SEG_TAB;                         // [SEG_TAB] i ln 20
    SegTab *s_tab = reinterpret_cast<SegTab *>(s_ln20 + SEG_TAB);
    uint32_t *s_z = reinterpret_cast<uint32_t *>(s_tab + 1);   // [32] signature words
    uint8_t *s_tri = reinterpret_cast<uint8_t *>(s_z + 32);    // [SEG_TRI] row of window number w in the triangular scan order of Seg::trim
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *wbase = smem + 2 * SEG_TAB * sizeof(double) + sizeof(SegTab) + 128 + SEG_TRI + (size_t)warp * seg_warp_bytes(fstride, maxm);
    if (threadIdx.x < 32) s_z[threadIdx.x] = g_segz[threadIdx.x];
    for (int d = threadIdx.x; d * (d + 1) / 2 < SEG_TRI; d += WARPS * 32)
        for (int w = d * (d + 1) / 2; w < (d + 1) * (d + 2) / 2 && w < SEG_TRI; ++w) s_tri[w] = (uint8_t)d;
    uint32_t *s_m = reinterpret_cast<uint32_t *>(wbase);       // [0..5] lo, [6..11] hi, [12..17] result mask
    uint8_t *fr = wbase + 18 * 4;
    uint8_t *P = fr + fstride;                                 // [maxm + 1][20] prefix counts of the segment being trimmed
    uint8_t *nc = P + (((maxm + 1) * 20 + 3) & ~3) + lane;     // [maxm + 2][32 lanes] letters-per-count histogram, kept zero
    for (int k = threadIdx.x; k < SEG_TAB; k += WARPS * 32) { s_lnfac[k] = g_lnfac[k]; s_ln20[k] = g_ln20[k]; }
    for (int k = threadIdx.x; k < (int)(sizeof(SegTab) / 4); k += WARPS * 32) reinterpret_cast<uint32_t *>(s_tab)[k] = reinterpret_cast<const uint32_t *>(&g_segtab)[k];
    __syncthreads();
    for (int k = 0; k < maxm + 2; ++k) nc[k * 32] = 0;
    const uint32_t *lom = s_m, *him = s_m + 6;
    uint32_t *mask = s_m + 12;
    // resident blocks (the tables above are staged once per block) whose warps draw frames from the queue through a
    // shared counter: the cost of a frame varies with the number and length of its low-complexity segments, and a
    // fixed stride left the slowest warp running long after the others.  The next frame's row is fetched into
    // registers while the current one is processed (up to two words per lane)
    const int64_t gfirst = (int64_t)gridDim.x * WARPS;        // entries below it are the warps' first frames
    const int fw = fstride / 4;
    uint32_t nrow = 0, nw0 = 0, nw1 = 0, nmw = 0;
    // lanes 0..5 / 6..11 carry the locut / hicut mask words of the frame (k_frames computed them), lanes 12..17 clear the result
    const int mword = lane < 6 ? lane : lane - 6;
    const bool mlane = lane < 12 && mword < nwr;
    const int msrc = lane < 6 ? mword : nwr + mword;
    int64_t g = (int64_t)blockIdx.x * WARPS + warp;
    if (g < n) {
        nrow = segq[g];
        const uint32_t *src = reinterpret_cast<const uint32_t *>(frames + (int64_t)nrow * fstride);
        if (lane < fw) nw0 = src[lane];
        if (lane + 32 < fw) nw1 = src[lane + 32];
        if (mlane) nmw = segm[g * (2 * nwr) + msrc];
    }
    for (int64_t gn; g < n; g = gn) {
        const uint32_t row = nrow;
        uint8_t *gfr = frames + (int64_t)row * fstride;
        const int m = (L - (int)(row % 6u) % 3) / 3;
        __syncwarp();
        if (lane < fw) reinterpret_cast<uint32_t *>(fr)[lane] = nw0;
        if (lane + 32 < fw) reinterpret_cast<uint32_t *>(fr)[lane + 32] = nw1;
        if (lane < 18) s_m[lane] = nmw;
        {
            unsigned int t = 0;
            if (lane == 0) t = atomicAdd(work, 1u);
            gn = gfirst + __shfl_sync(0xffffffffu, t, 0);
        }
        if (gn < n) {
            nrow = segq[gn];
            const uint32_t *src = reinterpret_cast<const uint32_t *>(frames + (int64_t)nrow * fstride);
            if (lane < fw) nw0 = src[lane];
            if (lane + 32 < fw) nw1 = src[lane + 32];
            if (mlane) nmw = segm[gn * (2 * nwr) + msrc];
        }
        __syncwarp();
        // Seg::segseq (downset 0, upset 1); the recursion of seg.c only adds segments, so the left parts are queued.
        // Position i of a sub-sequence [off, off + slen) looks at the frame's window off + min(i, wmax); the scans
        // over positions are searches for the next set / clear bit of the two window masks.
        int wl_off[12], wl_len[12], nwl = 1;
        wl_off[0] = 0; wl_len[0] = m;
        while (nwl > 0) {
            --nwl;
            const int off = wl_off[nwl], slen = wl_len[nwl];
            if (SEG_WINDOW > slen) continue;
            const int last = slen - 1, wmax = slen - SEG_WINDOW;
            int lowlim = 0;
            for (int i = 0; i <= last; ++i) {
                if (i <= wmax) {
                    const int k = next_bit<true>(lom, off + i, off + wmax);
                    if (k < 0) break;              // the positions past wmax repeat window wmax, which is clear
                    i = k - off;
                } else if (!sbit(lom, off + wmax)) break;
                // a window at or below locut is at or below hicut: position i itself is set in `him`
                int loi = lowlim, hii = last;
                if (lowlim <= wmax) {
                    const int k = prev_clear_bit(him, off + (i < wmax ? i : wmax), off + lowlim);
                    if (k >= 0) loi = k - off + 1;
                }
                if (i <= wmax) {
                    const int k = next_bit<false>(him, off + i, off + wmax);
                    if (k >= 0) hii = k - off - 1;
                }
                int leftend = loi, rightend = hii;
                coop_trim(fr, off + leftend, rightend - leftend + 1, P, nc, lane, s_lnfac, s_ln20, s_z, s_tri, leftend, rightend);
                if (i < leftend && nwl < 12) { wl_off[nwl] = off + loi; wl_len[nwl] = leftend - loi; ++nwl; }
                if (lane < 6) {                    // mask[off + leftend .. off + rightend], one word per lane
                    const int b0 = max(off + leftend, lane * 32), b1 = min(off + rightend, lane * 32 + 31);
                    if (b0 <= b1) mask[lane] |= (0xffffffffu >> (31 - (b1 - b0))) << (b0 & 31);
                }
                __syncwarp();
                i = hii < rightend ? hii : rightend;
                lowlim = i + 1;
            }
        }
        __syncwarp();
        for (int k = lane; k < m; k += 32)
            if (sbit(mask, k)) gfr[k] = AA_STOP;
    }
}

// K2b: one thread per frame of the store: slide the 10-letter murphy10 window, probe the five word tables and
// queue every posting of every word hit as a candidate (gframe, subject, subject position, query position,
// pattern).  Space for a whole posting list is reserved with one atomic.
struct Cand {                      // 12 bytes
    uint32_t gframe;               // row of the frame store
    uint32_t sj;                   // subject << 11 | subject position
    uint32_t ip;                   // query position << 8 | pattern
};

// Queue space is taken in runs: a warp keeps [cur, end) of a queue and only goes to the queue's counter (an atomic
// whose round trip to L2 the whole warp waits for, serialised per address) when the run is used up.  A batch of `total`
// records that does not fit fills the rest of the run and continues in a new one: record e of the batch goes to
// run_pos().  Only what a warp has left when it finishes is wasted; it is marked empty by the caller.
struct QueueRun {
    uint32_t cur = 0, end = 0;     // warp-uniform
    uint32_t room = 0, base = 0, next = 0;   // of the last batch: the first `room` records start at base, record e of the rest is at next + e
};
__device__ __forceinline__ void run_take(QueueRun &r, uint32_t total, unsigned long long *counter, uint32_t chunk, int lane) {
    r.room = r.end - r.cur;
    if (total > r.room) {
        const uint32_t want = max(total - r.room, chunk);
        uint32_t nb = 0;
        if (lane == 0) nb = (uint32_t)min(atomicAdd(counter, (unsigned long long)want), 0xf0000000ull);   // fills stay far below 2^32
        nb = __shfl_sync(0xffffffffu, nb, 0);
        r.next = nb - r.room;                       // record e >= room goes to nb + (e - room)
        r.base = r.cur;
        r.cur = nb + (total - r.room); r.end = nb + want;
    } else {
        r.room = total; r.base = r.cur; r.next = 0;
        r.cur += total;
    }
}
__device__ __forceinline__ uint32_t run_pos(const QueueRun &r, uint32_t e) { return e < r.room ? r.base + e : r.next + e; }

struct ProbeArgs {
    const unsigned long long *n_reads;   // reads of this chunk (device counter); frames = 6 per read
    int L;
    DevDB db;
    const uint8_t *frames;
    Cand *passq;                   // NQ sub-queues of cap_pass entries: words that passed the filter (gframe, letters 0..7, ip | letters 8, 9 << 16 | letter before the window << 24)
    unsigned long long *n_pass;    // NQ counters
    unsigned long long cap_pass;   // per sub-queue
    Cand *cand;                    // NQ sub-queues of cap_cand entries each (spreads the append atomics)
    unsigned long long *n_cand;    // NQ counters
    unsigned long long cap_cand;   // per sub-queue
};
constexpr int NQ = 64;

__device__ __forceinline__ int warp_scan_add(int v, int lane) {
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) v += t; }
    return v;
}

// word code (base 10, the key of the slot tables) of pattern p in the window (lo = letters 0..7 as nibbles, hi = 8, 9):
// the nine letters that are not the wildcard, first letter most significant.  Only words that passed the filter get here.
__device__ __forceinline__ uint32_t word_code(uint32_t lo, uint32_t hi, int p) {
    const int skip = p == 0 ? 9 : p + 2;
    uint32_t c = 0;
#pragma unroll
    for (int k = 0; k < 10; ++k) {
        const uint32_t d = k < 8 ? (lo >> (4 * k)) & 15u : (hi >> (4 * (k - 8))) & 15u;
        if (k != skip) c = c * 10u + d;
    }
    return c;
}

#ifndef MCX_PROBE_POS
#define MCX_PROBE_POS 2
#endif
#ifndef MCX_PROBE_NT
#define MCX_PROBE_NT 64               /* threads per block of k_probe: small blocks retire early (measured 64 / 96 / 128 / 160 / 192 / 256: 5.17 / 5.19 / 5.30 / 5.41 / 5.71 / 6.18 ms at 100 bp) */
#endif
#ifndef MCX_RESOLVE_NT
#define MCX_RESOLVE_NT 128
#endif
constexpr int PROBE_POS = MCX_PROBE_POS;   // window positions per loop iteration (2: four filter blocks in flight)
#ifndef MCX_PASS_CHUNK
#define MCX_PASS_CHUNK 256
#endif
constexpr int PASS_CHUNK = MCX_PASS_CHUNK;  // records a warp of k_probe reserves at a time (a warp queues ~170 at 150 bp)
constexpr uint32_t PASS_EMPTY = 0xffffffffu; // ip of a reserved record that was not used

// K2b, filter half: one thread per frame of the store slides the 10-letter murphy10 window and tests its five words
// against the presence filter (two block loads per window).  Nothing else happens here: the ~4 % of the words that pass
// are appended to a queue (one reservation per warp and iteration, positions from ballots) and resolved by k_resolve,
// one LANE per word.  (Before: the warp resolved its own passes inside this loop -- table slot, posting list, copy --
// with 3 of 32 lanes in the slot lookup and every lane of the warp waiting on two dependent DRAM round trips per
// iteration; 43 % of the stall samples of the kernel sat on those lines.  An earlier attempt to batch the passes in a
// per-warp shared-memory ring inside this kernel lost to MIO stalls; a global queue and a second kernel does not touch
// the MIO pipe here at all.)
#ifndef MCX_PROBE_MINB
#define MCX_PROBE_MINB 16             /* caps k_probe at 64 registers (56 used): probe + resolve 3.54 ms at 1M x 150 bp against 3.67 ms uncapped (72 registers) and 3.69 ms at 46 registers */
#endif
template <int NT>
__global__ void __launch_bounds__(NT, MCX_PROBE_MINB) k_probe(ProbeArgs A, int fstride) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int64_t n_frames = 6 * (int64_t)*A.n_reads;
    uint8_t *s_aa = smem;
    __shared__ uint8_t s_red[32];                  // residue -> murphy10 letter (one LDS instead of a 64-bit shift-and-mask per residue)
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid < 32) s_red[tid] = (uint8_t)(tid < 21 ? red_of(tid) : 15);
    __syncthreads();
    const int sq = blockIdx.x & (NQ - 1);
    const uint32_t lt = (1u << lane) - 1u;
    QueueRun run;                                  // this warp's space in the pass queue
    Cand *const qbase = A.passq + (unsigned long long)sq * A.cap_pass;
    // resident blocks stride over the frame rows, 32 per warp and step
    for (int64_t blk = blockIdx.x; blk * NT < n_frames; blk += gridDim.x) {
    __syncwarp();
    {   // each warp stages its 32 rows
        const int64_t row0 = blk * NT + (tid - lane);
        const uint32_t *src = reinterpret_cast<const uint32_t *>(A.frames + row0 * fstride);
        uint32_t *dst = reinterpret_cast<uint32_t *>(s_aa + (tid - lane) * fstride);
        for (int k = lane; k < 32 * fstride / 4; k += 32) dst[k] = src[k];
    }
    __syncwarp();
    const int64_t g = blk * NT + tid;
    const uint8_t *fr = s_aa + tid * fstride;
    const int m = g < n_frames ? (A.L - (int)(g % 6) % 3) / 3 : 0;
    // reduced letters of the 10-window [i, i+10) as nibbles (letter k at bits 4k); 15 past the end
    unsigned long long win = 0;
    for (int k = 0; k < 10; ++k) win |= (unsigned long long)(k < m ? s_red[fr[k]] : 15) << (4 * k);
    const int mmax = A.L / 3;
    uint32_t before = 15;                          // reduced letter left of the window (15: none)
    for (int i = 0; i + 9 <= mmax; i += PROBE_POS) {
        uint32_t lo[PROBE_POS], hi[PROBE_POS], left[PROBE_POS];
        bool ok9[PROBE_POS], ok10[PROBE_POS];
#pragma unroll
        for (int h = 0; h < PROBE_POS; ++h) {
            lo[h] = (uint32_t)win; hi[h] = (uint32_t)(win >> 32);
            left[h] = before; before = lo[h] & 15u;
            // letters >= 10 (stop, masked, past the end) as one bit per nibble: bit 3 and (bit 2 or bit 1)
            const uint32_t blo = (lo[h] >> 3) & ((lo[h] >> 2) | (lo[h] >> 1)) & 0x11111111u;
            const uint32_t bhi = (hi[h] >> 3) & ((hi[h] >> 2) | (hi[h] >> 1)) & 0x11u;
            ok9[h] = (blo | (bhi & 1u)) == 0u; ok10[h] = (blo | bhi) == 0u;
            if (i + h + 9 > mmax) { ok9[h] = false; ok10[h] = false; }      // past the last window of the longest frame
            const int nx = i + h + 10;
            win = (win >> 4) | ((unsigned long long)(nx < m ? s_red[fr[nx]] : 15) << 36);
        }
        // the two filter blocks of every window of the iteration in flight together
        uint32_t ha[PROBE_POS], hb[PROBE_POS];
        uint4 fa[PROBE_POS];
        uint2 fb[PROBE_POS];
#pragma unroll
        for (int h = 0; h < PROBE_POS; ++h) {
            ha[h] = filt_hash_a(lo[h], hi[h]); hb[h] = filt_hash_b(lo[h], hi[h]);
            fa[h] = ok9[h] ? __ldg(A.db.filt_a + filt_block(ha[h])) : make_uint4(0u, 0u, 0u, 0u);
            fb[h] = ok10[h] ? __ldg(A.db.filt_b + filt_block(hb[h])) : make_uint2(0u, 0u);
        }
        bool pass[N_PAT * PROBE_POS];
        uint32_t bal[N_PAT * PROBE_POS];
        int total = 0;
#pragma unroll
        for (int h = 0; h < PROBE_POS; ++h) {
            uint32_t b1, b2;
            filt_bits(0, lo[h], hi[h], ha[h], b1, b2); pass[N_PAT * h + 0] = (fa[h].x & b1) && (fa[h].w & b2);
            filt_bits(1, lo[h], hi[h], ha[h], b1, b2); pass[N_PAT * h + 1] = ok10[h] && (fa[h].y & (b1 | b2)) == (b1 | b2);
            filt_bits(2, lo[h], hi[h], ha[h], b1, b2); pass[N_PAT * h + 2] = ok10[h] && (fa[h].z & (b1 | b2)) == (b1 | b2);
            filt_bits(3, lo[h], hi[h], hb[h], b1, b2); pass[N_PAT * h + 3] = (fb[h].x & (b1 | b2)) == (b1 | b2);
            filt_bits(4, lo[h], hi[h], hb[h], b1, b2); pass[N_PAT * h + 4] = (fb[h].y & (b1 | b2)) == (b1 | b2);
#pragma unroll
            for (int p = 0; p < N_PAT; ++p) { bal[N_PAT * h + p] = __ballot_sync(0xffffffffu, pass[N_PAT * h + p]); total += __popc(bal[N_PAT * h + p]); }
        }
        if (total > 0) {
            run_take(run, (uint32_t)total, A.n_pass + sq, PASS_CHUNK, lane);
            if ((unsigned long long)run.end <= A.cap_pass) {
                int o = 0;
#pragma unroll
                for (int q = 0; q < N_PAT * PROBE_POS; ++q) {
                    if (pass[q]) {
                        Cand r; r.gframe = (uint32_t)g; r.sj = lo[q / N_PAT];
                        r.ip = ((uint32_t)(i + q / N_PAT) << 8) | (uint32_t)(q % N_PAT) | (hi[q / N_PAT] << 16) | (left[q / N_PAT] << 24);
                        qbase[run_pos(run, (uint32_t)(o + __popc(bal[q] & lt)))] = r;
                    }
                    o += __popc(bal[q]);
                }
            }
        }
    }
    }
    for (uint32_t e = run.cur + lane; e < run.end; e += 32)          // whole records: the readers load all three words
        if (e < A.cap_pass) { Cand z; z.gframe = 0u; z.sj = 0u; z.ip = PASS_EMPTY; qbase[e] = z; }
}

// K2b, table half: one lane per word that passed the filter: slot of its pattern's table (key and value share 8
// bytes: one load), then a cooperative, coalesced copy of all postings of the warp's 32 words into the candidate queue
// (gframe, subject, subject position, query position, pattern).  Resident warps walk their sub-queue in steps of 32
// words and take queue space CAND_CHUNK candidates at a time (unused records are marked empty), so the reservation --
// a round trip to L2 on which the whole warp waited, a third of the stall samples -- is paid once per several steps.
#ifndef MCX_CAND_CHUNK
#define MCX_CAND_CHUNK 512
#endif
constexpr int CAND_CHUNK = MCX_CAND_CHUNK;
constexpr uint32_t CAND_EMPTY = 0xffffffffu;    // ip of a reserved candidate record that was not used
template <int NT>
__global__ void __launch_bounds__(NT) k_resolve(ProbeArgs A) {
    __shared__ uint32_t s_x[NT / 32][128];          // per warp: inclusive prefix of posting counts, posting start, gframe, ip
    const int sq = blockIdx.y, lane = threadIdx.x & 31;
    const unsigned long long fill = min(A.n_pass[sq], A.cap_pass);
    uint32_t *xs = s_x[threadIdx.x >> 5];
    Cand *const qbase = A.cand + (unsigned long long)sq * A.cap_cand;
    QueueRun run;                                   // this warp's space in the candidate queue
    for (unsigned long long k = (unsigned long long)blockIdx.x * NT + threadIdx.x; k - lane < fill; k += (unsigned long long)gridDim.x * NT) {
        uint32_t cnt = 0, pi = 0, gframe = 0, ip = 0;
        Cand r; r.ip = PASS_EMPTY;
        if (k < fill) r = A.passq[(unsigned long long)sq * A.cap_pass + k];
        if (r.ip != PASS_EMPTY) {
            const int p = (int)(r.ip & 0xffu);
            const uint32_t c = word_code(r.sj, (r.ip >> 16) & 0xffu, p);
            // the query letter of the first rejection test (ExtendSeq2Set 0x4140c0-0x414113): the letter left of an exact
            // word (a word whose left neighbours also agree is found again one position to the left: left-maximal only), the
            // letter under the wildcard of a one-substitution word (if it agrees, the exact word finds the stretch)
            const uint32_t ql = p == 0 ? (r.ip >> 24) & 15u : (r.sj >> (4 * (p + 2))) & 15u;
            gframe = r.gframe; ip = (r.ip & 0xffffu) | (ql << 16);
            const uint2 *__restrict__ tb = A.db.htab + ((size_t)p << A.db.hbits);
            const uint32_t hmask = (1u << A.db.hbits) - 1u;
            uint32_t sl = (c * 2654435761u) >> (32 - A.db.hbits);
            uint2 kv = __ldg(tb + sl);
            while (kv.x != 0xffffffffu && kv.x != c) { sl = (sl + 1) & hmask; kv = __ldg(tb + sl); }
            if (kv.x == c) {
                const uint32_t v = kv.y;
                pi = v & 0x1ffffffu;                              // 25-bit start, 7-bit (count - 1)
                cnt = (v >> 25) + 1;
                if ((v >> 25) == 127) { cnt = __ldg(A.db.post + pi); ++pi; }   // longer lists start with their length
            }
        }
        const int inc2 = warp_scan_add((int)cnt, lane);
        const int tot2 = __shfl_sync(0xffffffffu, inc2, 31);
        if (tot2 == 0) continue;
        __syncwarp();
        xs[lane] = (uint32_t)inc2; xs[32 + lane] = pi; xs[64 + lane] = gframe; xs[96 + lane] = ip;
        __syncwarp();
        for (int e0 = 0; e0 < tot2; e0 += 32) {
            const int e = e0 + lane;
            bool keep = false;
            Cand c; c.gframe = c.sj = c.ip = 0;
            if (e < tot2) {
                int lo = 0;                                   // first owner whose inclusive prefix exceeds e
#pragma unroll
                for (int step = 16; step; step >>= 1) if (xs[lo + step - 1] <= (uint32_t)e) lo += step;
                const uint32_t q = (uint32_t)e - (lo ? xs[lo - 1] : 0u);
                const uint32_t post = __ldg(A.db.post + xs[32 + lo] + q), meta = xs[96 + lo];
                const uint32_t ql = meta >> 16, tl = (post >> 26) & 15u;
                keep = !(ql == tl && ql < 10u);               // equal valid letters: rejected (three candidates in five)
                c.gframe = xs[64 + lo]; c.sj = post & 0x3ffffffu; c.ip = meta & 0xffffu;
            }
            const uint32_t km = __ballot_sync(0xffffffffu, keep);
            if (km == 0u) continue;
            run_take(run, (uint32_t)__popc(km), A.n_cand + sq, CAND_CHUNK, lane);
            if ((unsigned long long)run.end > A.cap_cand) continue;
            if (keep) qbase[run_pos(run, (uint32_t)__popc(km & ((1u << lane) - 1u)))] = c;
        }
    }
    for (uint32_t e = run.cur + lane; e < run.end; e += 32)
        if (e < A.cap_cand) { Cand z; z.gframe = 0u; z.sj = 0u; z.ip = CAND_EMPTY; qbase[e] = z; }
}

// K2b: one thread per candidate: grow the word to the maximal murphy10-identical stretch, apply the seed
// acceptance test and walk the ungapped X-drop extension both ways (ExtendSeq2Set 0x413fc4-0x414073, AlignFwd /
// AlignBwd).  HSPs reaching the report floor are appended to the survivor list.
struct ExtArgs {
    const int32_t *kept;
    int64_t first;
    int L, fstride;
    int thr_report;                // ungapped HSPs at or above this raw score survive
    DevDB db;
    const uint8_t *frames;
    const Cand *cand;
    const unsigned long long *qfill;     // NQ sub-queue fills (device counters)
    unsigned long long cap_cand;   // per sub-queue
    uint4 *surv;
    unsigned long long *n_surv;
    unsigned long long cap_surv;
    uint4 *seedq;                  // accepted seeds (k_seed -> k_walk)
    unsigned long long *n_seedq;
    unsigned long long cap_seedq;
    unsigned long long *seen;      // open-addressing set of the HSP keys appended in this launch, ~0 = empty
    unsigned long long seen_mask;
    int seen_shift;
};

// (Tried and measured slower -- 5.1 -> 5.4 ms at 100 bp, 9.4 -> 19.3 ms at 150 bp: copying the frame row and the subject
// residues on the candidate's diagonal into shared memory up front, with all word loads in flight together.  Three in
// four candidates are rejected after looking at a dozen residues; staging whole rows for all of them costs more
// than the dependent byte loads of the few that walk far.)
// Two kernels with a compacted queue between them: three in four candidates are rejected by k_seed, and the walks of
// the rest are the long part -- in one kernel they ran with 8 of 32 lanes active.
// accepted seed, 16 bytes: x frame row | y subject(15) sb(11) | z qb(8) len(8) score0(16) | w id0
__device__ __forceinline__ uint4 seed_pack(uint32_t gframe, int s, int sb, int qb, int len, int score0, int id0) {
    return make_uint4(gframe, (uint32_t)s | ((uint32_t)sb << 15), (uint32_t)qb | ((uint32_t)len << 8) | ((uint32_t)score0 << 16), (uint32_t)id0);
}

// (No duplicate filter here: the left-maximal rule for exact words and the one-window-per-position rule for the
// substitution words already make every accepted stretch unique -- 74,491,397 of 74,491,397 at 2M x 150 bp.)
#ifndef MCX_SEED_NT
#define MCX_SEED_NT 128
#endif
#ifndef MCX_GAP_NT
#define MCX_GAP_NT 128
#endif
#ifndef MCX_WALK_NT
#define MCX_WALK_NT MCX_SEED_NT
#endif
#ifndef MCX_SEG_W
#define MCX_SEG_W 4
#endif
#ifndef MCX_FRAMES_NT
#define MCX_FRAMES_NT 192
#endif
constexpr int SEED_NT = MCX_SEED_NT;   // threads per block of k_seed
constexpr int WALK_NT = MCX_WALK_NT;   // threads per block of k_walk
constexpr int GAP_NT = MCX_GAP_NT;     // threads per block of k_gap_dir
#define SAME(a, b) ((s_same[(a)] >> (b)) & 1u)   /* red_eq() from the shared-memory masks */
__device__ uint32_t g_same[32];                  // bit b of g_same[a]: residues a and b share a murphy10 letter (upload_tables)
#ifndef MCX_SEED_CHUNK
#define MCX_SEED_CHUNK 256
#endif
constexpr int SEED_CHUNK = MCX_SEED_CHUNK;
constexpr uint32_t SEED_EMPTY = 0xffffffffu;     // x (frame row) of a reserved seed record that was not used
// K2c: one thread per candidate: the cheap rejections, growth of the word to the maximal murphy10-identical stretch
// and the seed acceptance test (ExtendSeq2Set 0x413fc4-0x414073); accepted seeds are queued for k_walk.
template <int NT>
__global__ void __launch_bounds__(NT) k_seed(ExtArgs A) {
    __shared__ __align__(4) int8_t s_bl[21 * 32];
    __shared__ uint32_t s_same[32];                 // bit b of s_same[a]: residues a and b share a murphy10 letter
    for (int k = threadIdx.x; k < 21 * 32 / 4; k += NT) reinterpret_cast<uint32_t *>(s_bl)[k] = reinterpret_cast<const uint32_t *>(g_blosum)[k];
    if (threadIdx.x < 32) s_same[threadIdx.x] = g_same[threadIdx.x];
    __syncthreads();
    // grid.y = candidate sub-queue, whose fill is read on the device; the blocks of a row are resident and stride over
    // it (the tables above are staged once per block, not once per 128 candidates), and every warp takes space in the
    // seed queue SEED_CHUNK records at a time, unused records marked empty: one counter, ~3 M additions per million
    // reads when every warp added for itself, which the L2 serialises
    const int sq = blockIdx.y, lane = threadIdx.x & 31;
    const unsigned long long fill = min(A.qfill[sq], A.cap_cand);
    QueueRun run;                                   // this warp's space in the seed queue
    for (unsigned long long k = (unsigned long long)blockIdx.x * NT + threadIdx.x; k - lane < fill; k += (unsigned long long)gridDim.x * NT) {
    uint4 rec;
    const bool accepted = k < fill && [&]() -> bool {
    const Cand c = A.cand[(unsigned long long)sq * A.cap_cand + k];
    if (c.ip == CAND_EMPTY) return false;
    const int frame = (int)(c.gframe % 6u);
    const int m = (A.L - frame % 3) / 3;
    const uint8_t *__restrict__ fr = A.frames + (int64_t)c.gframe * A.fstride;
    const int s = (int)(c.sj >> 11), j = (int)(c.sj & 0x7ff), i = (int)(c.ip >> 8), p = (int)(c.ip & 0xff);
    const int32_t o = __ldg(A.db.off + s);
    const int n = __ldg(A.db.off + s + 1) - o;
    const uint8_t *__restrict__ t = A.db.res + o;
    // The sixteen residues around the word on both sequences (positions i-3 .. i+12 and j-3 .. j+12) are fetched as
    // five aligned words each, all in flight together, and every test below reads them from registers.  (Before: each
    // test waited for its own pair of byte loads -- up to a dozen dependent round trips per candidate.)  Only a stretch
    // that grows past the fetched window on either side takes the byte-wise path.
    uint32_t Q[4], T[4];
    {
        const uint8_t *pq = fr + i - 3, *pt = t + j - 3;         // the frame store and the residues are padded on both sides
        const uint32_t *aq = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(pq) & ~(uintptr_t)3);
        const uint32_t *at = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(pt) & ~(uintptr_t)3);
        const int shq = 8 * (int)(reinterpret_cast<uintptr_t>(pq) & 3), sht = 8 * (int)(reinterpret_cast<uintptr_t>(pt) & 3);
        uint32_t wq[5], wt[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) { wq[k] = __ldg(aq + k); wt[k] = __ldg(at + k); }
#pragma unroll
        for (int k = 0; k < 4; ++k) { Q[k] = __funnelshift_r(wq[k], wq[k + 1], shq); T[k] = __funnelshift_r(wt[k], wt[k + 1], sht); }
    }
#define QB(d) ((int)((Q[((d) + 3) >> 2] >> (8 * (((d) + 3) & 3))) & 0xffu))
#define TB(d) ((int)((T[((d) + 3) >> 2] >> (8 * (((d) + 3) & 3))) & 0xffu))
    // (exact words whose left neighbours agree and one-substitution words whose replaced letter agrees never get here:
    // k_resolve drops them from the letter it finds in the posting)
    // one-substitution words: keep one window per substituted position (all windows give the same seed)
    if (p >= 2 && i + 10 < m && j + 10 < n && SAME(QB(10), TB(10))) return false;
    int qb, sb, len, score0 = 0, id0 = 0;
    {
        int r = p == 0 ? 9 : 10, l = 0;             // the stretch is [i - l, i + r)
        // (bitwise &, selects and unconditional table reads on purpose: with && / if the compiler turns these unrolled
        // steps into per-lane branches and the warp runs them at 9 of 32 lanes)
#pragma unroll
        for (int d = 9; d <= 12; ++d) r += (int)((uint32_t)(d == r) & (uint32_t)(i + d < m) & (uint32_t)(j + d < n) & SAME(QB(d), TB(d)));
#pragma unroll
        for (int d = 1; d <= 3; ++d) l += (int)((uint32_t)(d == l + 1) & (uint32_t)(i - d >= 0) & (uint32_t)(j - d >= 0) & SAME(QB(-d), TB(-d)));
        const bool beyond = (r == 13 && i + 13 < m && j + 13 < n) || (l == 3 && i - 4 >= 0 && j - 4 >= 0);
        if (!beyond) {
            qb = i - l; sb = j - l; len = r + l;
#pragma unroll
            for (int d = -3; d <= 12; ++d) {
                const int a = QB(d), b = TB(d);                      // residues or padding: always 0..20
                const int in = (int)((uint32_t)(d >= -l) & (uint32_t)(d < r));
                score0 += in * (int)s_bl[a * 32 + b];
                id0 += in & (int)((uint32_t)(a == b) & (uint32_t)(a < 20));
            }
        } else {
            qb = i; sb = j; len = p == 0 ? 9 : 10;
            while (qb + len < m && sb + len < n && SAME(fr[qb + len], t[sb + len])) ++len;
            while (qb > 0 && sb > 0 && SAME(fr[qb - 1], t[sb - 1])) { --qb; --sb; ++len; }
            for (int k = 0; k < len; ++k) {
                const int a = fr[qb + k], b = t[sb + k];
                score0 += s_bl[a * 32 + b];
                id0 += (a == b && a < 20);
            }
        }
    }
#undef QB
#undef TB
    if (score0 < SEED_MIN_SCORE || id0 < SEED_MIN_IDENT) return false;
    rec = seed_pack(c.gframe, s, sb, qb, len, score0, id0);
    return true;
    }();
    const uint32_t am = __ballot_sync(0xffffffffu, accepted);
    if (am == 0u) continue;
    run_take(run, (uint32_t)__popc(am), A.n_seedq, SEED_CHUNK, lane);
    const uint32_t at = run_pos(run, (uint32_t)__popc(am & ((1u << lane) - 1u)));
    if (accepted && at < A.cap_seedq) A.seedq[at] = rec;
    }
    for (uint32_t e = run.cur + lane; e < run.end; e += 32) if (e < A.cap_seedq) A.seedq[e] = make_uint4(SEED_EMPTY, 0u, 0u, 0u);
}

#undef SAME
// K2d: one thread per accepted seed: the ungapped X-drop walks both ways (AlignFwd / AlignBwd); HSPs reaching the
// report floor are appended to the survivor list.
// (Tried and measured slower, 1.61 -> 2.15 ms at 1M x 150 bp: loading the residues of four steps together, the next four
// while the current four are scored.  The walks are short -- most stop after a few residues -- so the batches mostly
// fetch what is never used, and the kernel went from 36 to 80 registers, 69 % to 35 % occupancy.
// Also slower, 1.69 -> 1.96 ms: one loop stepping the forward and the backward walk together, so that their byte loads
// are in flight at the same time -- 48 registers, and every iteration carries the bookkeeping of both directions although
// one of them has usually stopped.)
__device__ __forceinline__ void walk_one(const ExtArgs &A, const int8_t *s_bl, int64_t g) {
    const uint4 sd = A.seedq[g];
    const uint32_t gframe = sd.x;
    if (gframe == SEED_EMPTY) return;
    const int s = (int)(sd.y & 0x7fffu), sb = (int)(sd.y >> 15), qb = (int)(sd.z & 0xffu), len = (int)((sd.z >> 8) & 0xffu);
    const int score0 = (int)(sd.z >> 16), id0 = (int)sd.w;
    const int frame = (int)(gframe % 6u);
    const int m = (A.L - frame % 3) / 3;
    const uint8_t *__restrict__ fr = A.frames + (int64_t)gframe * A.fstride;
    const int32_t o = __ldg(A.db.off + s);
    const int n = __ldg(A.db.off + s + 1) - o;
    const uint8_t *__restrict__ t = A.db.res + o;
    // both walks start from the seed score; stop after a residue that leaves the running score below -20 or
    // at least 9 (> 8.94) under the best so far
    int fe = 0, fid = 0, gf = 0, be = 0, bid = 0, gb = 0;
    {
        const int nq = m - qb - len, nt = n - sb - len;
        if (nq > 0 && nt > 0) {
            int best = score0, cur = score0, k = 0, id = 0;
            for (;;) {
                const int a = fr[qb + len + k], b = t[sb + len + k];
                cur += s_bl[a * 32 + b];
                id += (a == b && a < 20);
                ++k;
                if (cur > best) { best = cur; fe = k; fid = id; }
                if (k >= nt || k >= nq) break;
                if (cur < UNGAP_FLOOR || cur <= best - 9) break;
            }
            gf = best - score0;
        }
    }
    {
        const int nq = qb, nt = sb;
        if (nq > 0 && nt > 0) {
            int best = score0, cur = score0, k = 0, id = 0;
            for (;;) {
                const int a = fr[qb - 1 - k], b = t[sb - 1 - k];
                cur += s_bl[a * 32 + b];
                id += (a == b && a < 20);
                ++k;
                if (cur > best) { best = cur; be = k; bid = id; }
                if (k >= nt || k >= nq) break;
                if (cur < UNGAP_FLOOR || cur <= best - 9) break;
            }
            gb = best - score0;
        }
    }
    const int total = score0 + gf + gb;
    if (total < A.thr_report) return;
    const int hq0 = qb - be, hq1 = qb + len + fe - 1, ht0 = sb - be;
    {   // An HSP is found once from every seed it contains; only its first copy goes on (the gapped extensions of
        // the copies would be identical).  64-bit key: frame row, subject, (q0, q1) as a triangular index, t0.
        const unsigned long long key = ((unsigned long long)gframe << 40) | ((unsigned long long)s << 25) |
                                       ((unsigned long long)(hq1 * (hq1 + 1) / 2 + hq0) << 11) | (unsigned long long)ht0;
        unsigned long long slot = (key * 0x9E3779B97F4A7C15ull) >> A.seen_shift;
        for (int probe = 0; probe < 4096; ++probe) {
            const unsigned long long old = atomicCAS(A.seen + slot, ~0ull, key);
            if (old == ~0ull) break;
            if (old == key) return;
            slot = (slot + 1) & A.seen_mask;
        }
    }
    const uint32_t mask = __activemask();
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(A.n_surv, (unsigned long long)__popc(mask));
    base = __shfl_sync(mask, base, leader);
    const unsigned long long idx = base + __popc(mask & ((1u << lane) - 1));
    if (idx >= A.cap_surv) return;
    Surv v;
    v.read = A.kept[A.first + gframe / 6u]; v.subject = s; v.frame = frame;
    v.q0 = hq0; v.q1 = hq1;
    v.ident = id0 + fid + bid; v.t0 = ht0;
    v.score = total;
    v.gframe = gframe;
    A.surv[idx] = surv_pack(v);
}
// grid-stride over the seed queue, whose length is read on the device (no host round trip after k_seed)
template <int NT>
__global__ void __launch_bounds__(NT) k_walk(ExtArgs A) {
    __shared__ __align__(4) int8_t s_bl[21 * 32];
    const int64_t n_seeds = (int64_t)min(*A.n_seedq, A.cap_seedq);
    if ((int64_t)blockIdx.x * NT >= n_seeds) return;          // the grid is sized for a full chunk: small batches leave most blocks without work
    for (int k = threadIdx.x; k < 21 * 32 / 4; k += NT) reinterpret_cast<uint32_t *>(s_bl)[k] = reinterpret_cast<const uint32_t *>(g_blosum)[k];
    __syncthreads();
    for (int64_t g = (int64_t)blockIdx.x * NT + threadIdx.x; g < n_seeds; g += (int64_t)gridDim.x * NT) walk_one(A, s_bl, g);
}

// ------------------------------------------------------------------------------------------------
// K3: gapped X-drop extension (AlignGapped 0x40a550) with the alignment statistics carried forward.
// The binary stores three trace matrices and walks back from the best cell; every choice it makes is
// local to a cell (diagonal unless E is strictly larger, then F only if strictly larger; a gap opens
// rather than extends on ties), so carrying (identities, columns, gap columns, gap runs) along the same
// choices gives the same numbers without storing a matrix.  The live column window [cs, ce] and its
// pruning follow the binary exactly because they decide which cells exist.
// stats word: ident bits 0-7, aln 8-16, gap columns 17-25, gap runs 26-31
// ------------------------------------------------------------------------------------------------
#define ST_ALN 0x100u
#define ST_GAPCOL 0x20000u
#define ST_GAPRUN 0x4000000u
struct __align__(16) GExtRec { int32_t gain; uint16_t eq, et; uint32_t st; uint32_t cells; };   // result of one direction

struct GapArgs {
    int L, fstride;
    DevDB db;
    const uint8_t *frames;         // frame store of the chunk the survivors came from
    const uint4 *surv;             // survivors [first, first + n_surv) of the global list
    int64_t first, n_surv;
    unsigned long long *items;     // work list: sort key << 32 | (survivor - first) << 1 | direction
    unsigned long long *n_items;
    unsigned long long *n_items_total;   // running total over the chunks of a search
    GExtRec *ext;                  // [2 * (survivor - first) + direction], zeroed before the launch
    mcx_hit *hsp;
    SortKey *keys;
    int32_t *idx;
    unsigned long long *counters;  // [0] gapped extensions, [1] cells
};

// K3a: which (survivor, direction) pairs get a gapped extension (AlignSeqs 0x4134c8-0x4135b4: ungapped total >= 48.17
// and more than two residues left on both sequences on that side).  Compaction again: the DP kernel only sees work.
__global__ void k_gap_list(GapArgs A) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool f = false, b = false;
    uint32_t kf = 0, kb = 0;
    if (g < A.n_surv) {
        const Surv v = surv_unpack(A.surv[A.first + g]);
        if (v.score >= 49) {
            const int m = (A.L - v.frame % 3) / 3;
            const int n = A.db.off[v.subject + 1] - A.db.off[v.subject];
            const int t1 = v.t0 + (v.q1 - v.q0);
            f = (m - (v.q1 + 1) > 2) && (n - (t1 + 1) > 2);
            b = (v.q0 > 2) && (v.t0 > 2);
            // sort key: longest remaining query stretch first (the rows the DP can run over); threads of a warp
            // then finish at similar times
            kf = 255u - (uint32_t)min(m - (v.q1 + 1), 255);
            kb = 255u - (uint32_t)min((int)v.q0, 255);
        }
    }
    const int lane = threadIdx.x & 31;
    const uint32_t mf = __ballot_sync(0xffffffffu, f), mb = __ballot_sync(0xffffffffu, b);
    const int tot = __popc(mf) + __popc(mb);
    if (tot == 0) return;
    unsigned long long base = 0;
    if (lane == 0) { base = atomicAdd(A.n_items, (unsigned long long)tot); atomicAdd(A.n_items_total, (unsigned long long)tot); }
    base = __shfl_sync(0xffffffffu, base, 0);
    const uint32_t lt = (1u << lane) - 1;
    if (f) A.items[base + __popc(mf & lt)] = ((unsigned long long)kf << 32) | (uint32_t)(g << 1);
    if (b) A.items[base + __popc(mf) + __popc(mb & lt)] = ((unsigned long long)kb << 32) | (uint32_t)(g << 1) | 1u;
}

// K3b, new layout (round 2): two kernels, no local memory.
//  * k_gap_screen: ALL extensions, one thread each, until the extension either dies without ever reaching a positive
//    score (72-85 % of them: nothing to add to the HSP) or produces its first positive cell (then it is queued for
//    k_gap_dp).  While the best score is still 0 the X-drop bookkeeping collapses: the threshold is the constant -27,
//    the best column is 0, so the window always starts at column 1, the left side is never pruned and the boundary
//    cell of row i is -11 - i in closed form.  The DP rows are one packed word per column (H and F as 16-bit halves)
//    in shared memory, column-major with the thread as the fastest index (bank = lane: conflict-free whatever column
//    each lane is at).  All lanes of a warp start row 1 together, so their windows have similar widths throughout.
//    The recurrences use the DPX forms: E and F are max(a + b, c) = viaddmax, H is a three-way max = vimax3.
//  * k_gap_dp + k_gap_trace: the extensions that gain.  k_gap_dp runs the complete X-drop DP (scores only) to its natural
//    end with the rows in a 64-column ring of packed H|F words in shared memory, and records for every cell which way it
//    came as a nibble in global memory (what the binary keeps in its three trace matrices); k_gap_trace walks back from
//    the best cell like the binary's CalRes and counts identities, columns, gap columns and gap runs.  (Carrying those
//    statistics through the DP, as round 1 did, needs two more words per column: 768 bytes of shared memory per
//    extension, 9 warps per SM, 32 % of the issue slots used.)  An extension whose live window [cs - 1, ce] reaches 56
//    columns is handed to the local-memory kernel k_gap_dir below, which stays as that fallback.  Measured on a B200
//    (mcx_search_counters [5] / [6]): on 200,000 reads of the bench stream at 150 bp, 71,088 extensions went to
//    k_gap_dp and none to k_gap_dir (widest window: 47 columns); on divergent homologs of the markers
//    (tests/homologs.py) 15 of 2,325,109 at 150 bp (100,000 reads) and 9 of 523,564 at 500 bp (3,000 reads).
// The first version of this stage (k_gap_dir for everything: rows of GROW ints in local memory, 6 LDL + 14 STL sites in
// the score pass, 1.09 GB of DRAM writes per 226 M cells) ran at 110 GCUPS at 100 bp and 85 at 150 bp.
#ifndef MCX_GAP_REFILL
#define MCX_GAP_REFILL 24
#endif
// (the hand-off limits the kernels test are arguments: these sizes by default, lower with MCX_GAP_SCREEN_ROWS / _COLS and
// MCX_GAP_DP_COLS, see gapped_stage)
constexpr int SCR_COLS = 48;                   // columns of the screening pass (an extension that needs more goes to k_gap_dp)
constexpr int RING = 64;                       // ring of k_gap_dp
#ifndef MCX_SCR_NT
#define MCX_SCR_NT 128
#endif
#ifndef MCX_FULL_NT
#define MCX_FULL_NT 128
#endif
__device__ __forceinline__ uint32_t pack_hf(int h, int f) { return ((uint32_t)h & 0xffffu) | ((uint32_t)f << 16); }
__device__ __forceinline__ int hf_h(uint32_t w) { return (int)(short)(w & 0xffffu); }
__device__ __forceinline__ int hf_f(uint32_t w) { return (int)w >> 16; }

constexpr int SCR_ROWS = 32;                   // rows of the screening pass (no extension without a gain came near: they die by row 28)
// residues p[0], p[step], p[2 step], ... (at most 4 W of them, `have` exist) -> W words of four in a column of shared
// memory with stride NT; aligned 32-bit loads, shifted into place (and byte-reversed for step = -1)
template <int W, int NT>
__device__ __forceinline__ void load_residues(const uint8_t *p, int step, int have, uint32_t *dst) {
    const int nw = min(W, (have + 3) >> 2);
    if (step > 0) {
        const uint32_t *a = reinterpret_cast<const uint32_t *>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
        const int sh = 8 * (int)(reinterpret_cast<uintptr_t>(p) & 3);
        uint32_t lo = __ldg(a);
        for (int k = 0; k < nw; ++k) { const uint32_t hi = __ldg(a + k + 1); dst[k * NT] = __funnelshift_r(lo, hi, sh); lo = hi; }
    } else {
        // bytes p[0], p[-1], ...: the word holding p[0] is the highest one
        const uintptr_t top = reinterpret_cast<uintptr_t>(p) + 1;            // one past p[0]
        const uint32_t *a = reinterpret_cast<const uint32_t *>((top + 3) & ~(uintptr_t)3);   // first aligned word boundary at or above top
        const int sh = 8 * (int)((reinterpret_cast<uintptr_t>(a) - top) & 3);               // bytes of a[-1] above p[0]
        uint32_t hi = __ldg(a - 1);
        for (int k = 0; k < nw; ++k) {
            const uint32_t lo = __ldg(a - 2 - k);
            // four bytes ending at p[-4k]: (lo:hi) shifted left by sh bytes, upper word, then reversed
            dst[k * NT] = __byte_perm(__funnelshift_l(lo, hi, sh), 0, 0x0123);
            hi = lo;
        }
    }
}
struct ExtSetup { const uint8_t *qp, *t; int step, nQ, nD; };
__device__ __forceinline__ ExtSetup ext_setup(const GapArgs &A, uint32_t item) {
    const int64_t g = item >> 1;
    const Surv v = surv_unpack(A.surv[A.first + g]);
    const uint8_t *fr = A.frames + (int64_t)v.gframe * A.fstride;
    const int m = (A.L - v.frame % 3) / 3;
    const int32_t o = A.db.off[v.subject];
    const int n = A.db.off[v.subject + 1] - o;
    const int q0 = v.q0, q1 = v.q1, t0 = v.t0, t1 = v.t0 + (v.q1 - v.q0);
    ExtSetup S;
    int ql, tl;
    if ((item & 1) == 0) { ql = m - (q1 + 1); tl = n - (t1 + 1); S.qp = fr + q1 + 1; S.t = A.db.res + o + t1 + 1; S.step = 1; }
    else { ql = q0; tl = t0; S.qp = fr + q0 - 1; S.t = A.db.res + o + t0 - 1; S.step = -1; }
    if (tl > ql + GAP_SLACK) tl = ql + GAP_SLACK;
    S.nQ = ql; S.nD = tl;
    return S;
}

template <int NT>
__global__ void __launch_bounds__(NT) k_gap_screen(GapArgs A, const unsigned long long *__restrict__ items,
                                                   unsigned long long *__restrict__ gainers, unsigned long long *n_gainers,
                                                   int scr_rows, int scr_cols) {
    __shared__ __align__(16) int8_t s_bl[21 * 32];
    __shared__ uint32_t s_hf[SCR_COLS * NT];
    __shared__ uint32_t s_tq[(SCR_COLS / 4 + SCR_ROWS / 4) * NT];    // subject residues of columns 1 .. 48 and query residues of rows 1 .. 32, four per word
    for (int k = threadIdx.x; k < 21 * 32 / 4; k += NT) reinterpret_cast<uint32_t *>(s_bl)[k] = reinterpret_cast<const uint32_t *>(g_blosum)[k];
    __syncthreads();
    const int64_t n_items = (int64_t)*A.n_items;
    uint32_t *tw = s_tq + threadIdx.x, *qw = tw + (SCR_COLS / 4) * NT;
    const int lane = threadIdx.x & 31;
    const int GI = GAP_OPEN, GE = GAP_EXT, GIE = GAP_OPEN + GAP_EXT;
    constexpr int LIMIT = 15, DROP = 27;       // (int)((26.98 - 11) / 1); h < best - 26.98 <=> h <= best - 27
    uint32_t *hf = s_hf + threadIdx.x;
#define HF(j) hf[(j) * NT]
    for (int64_t w = (int64_t)blockIdx.x * NT + threadIdx.x; w - lane < n_items; w += (int64_t)gridDim.x * NT) {
        bool gain = false, busy = false;
        uint32_t item = 0;
        int nQ = 0, nD = 0, step = 1, ce = LIMIT, cells = 0, i = 1;
        const uint8_t *__restrict__ qp = nullptr, *__restrict__ t = nullptr;
        if (w < n_items) {
            item = (uint32_t)items[w];
            const ExtSetup S = ext_setup(A, item);
            nQ = S.nQ; nD = S.nD; step = S.step; qp = S.qp; t = S.t;
            // the residues this pass can touch go to shared memory once (with 25-34 KB of shared memory per block the L1
            // left over does not hold the rows of a thousand threads: the per-cell byte loads missed it 97 % of the time)
            load_residues<SCR_COLS / 4, NT>(t, step, nD, tw);
            load_residues<SCR_ROWS / 4, NT>(qp, step, nQ, qw);
            // row 0: H = -11 - j, F = H - 11 for j = 1 .. 15 (the cells past nD are never read)
#pragma unroll
            for (int j = 1; j <= LIMIT; ++j) HF(j) = pack_hf(-GI - j * GE, -GI - j * GE - GI);
            busy = nQ >= 1;
        }
        // one row per trip for every lane that still runs: the vote at the top brings the warp back together each row
        // (left to themselves the lanes drift apart and the warp issues their loops one after the other: 2 of 32 lanes
        // per instruction in the first version of this kernel)
        for (;;) {
            const uint32_t bm = __ballot_sync(0xffffffffu, busy);
            if (!bm) break;
            if (busy) {
                // boundary cell, column 0: H = F = -11 - i; the diagonal of column 1 is the boundary of the row before
                const int v = -GI - i * GE;
                int diag = i == 1 ? 0 : v + GE;
                int E = v - GI, hl = v, j = 1;
                bool skip_tail = false;
                const int8_t *brow_q = s_bl + ((qw[((i - 1) >> 2) * NT] >> (8 * ((i - 1) & 3))) & 0xffu) * 32;
                const int jend = min(ce, nD);
                // four columns per word of subject residues; one test covers both ways a row can end early: h outside
                // [-26, 0] (a positive cell = gain; h <= -27 = dead, and with the best column at 0 every column is right of
                // it).  An exit leaves j = first column not computed.  (One copy of the cell code on purpose: a variant with
                // a check-free copy for whole groups ran at 10.8 instead of 17.2 lanes per instruction -- lanes in different
                // copies cannot issue together.)
                int hx = 0;
                bool stop = false, ended = false;
                for (int jb = 0; jb < jend && !ended; jb += 4) {
                    const uint32_t tword = tw[(jb >> 2) * NT];
                    uint32_t *hp = hf + (jb + 1) * NT;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (jb + k + 1 > jend) { ended = true; break; }
                        const uint32_t old = hp[k * NT];
                        const int Ho = hf_h(old), Fo = hf_f(old);
                        E = __viaddmax_s32(hl, -GIE, E - GE);
                        const int Fv = __viaddmax_s32(Ho, -GIE, Fo - GE);
                        const int h = __vimax3_s32(diag + brow_q[(tword >> (8 * k)) & 0xffu], E, Fv);
                        diag = Ho;
                        hp[k * NT] = pack_hf(h, Fv);
                        hl = h;
                        if ((unsigned)(h + (DROP - 1)) >= (unsigned)DROP) { j = jb + k + 2; hx = h; stop = true; ended = true; break; }
                    }
                }
                if (!stop) j = jend + 1;
                else if (hx > 0) gain = true;
                else { skip_tail = j - 1 < ce; ce = j - 1; }
                if (gain) busy = false;
                else {
                    cells += j - 1;
                    if (!skip_tail) {                            // run on along the row by horizontal gaps
                        for (int jj = ce + 1; jj <= nD; ++jj) {
                            if (jj >= scr_cols) { gain = true; busy = false; break; }   // needs more columns than this pass has: the full pass takes it
                            ++cells;
                            E = __viaddmax_s32(hl, -GIE, E - GE);
                            HF(jj) = pack_hf(E, E - GI);
                            hl = E;
                            if (E <= -DROP) { ce = jj; break; }
                        }
                    }
                    if (!(1 < ce) || i >= nQ) busy = false;
                    else if (i >= scr_rows) { gain = true; busy = false; }   // more rows than this pass holds residues for
                    ++i;
                }
            }
        }
        if (w < n_items && !gain) {
            GExtRec r;
            r.gain = 0; r.eq = 0; r.et = 0; r.st = 0; r.cells = (uint32_t)cells;
            A.ext[item] = r;
        }
        const uint32_t mg = __ballot_sync(0xffffffffu, gain);
        if (mg) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(n_gainers, (unsigned long long)__popc(mg));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (gain) gainers[base + __popc(mg & ((1u << lane) - 1))] = item;
        }
    }
#undef HF
}

// complete score-only DP for the extensions that gain, recording per cell which way it came (for k_gap_trace); lanes draw
// extensions from the list as they finish.  Directions: 9 words per row of an extension -- the row's cs, then a nibble
// per column (ring-indexed like the DP row): bits 0-1 = 0 diagonal / 1 from E / 2 from F, bit 2 = E was opened from H
// (rather than extended), bit 3 = F was opened.
constexpr int DIR_ROW_WORDS = 1 + RING / 8;
template <int NT>
__global__ void __launch_bounds__(NT) k_gap_dp(GapArgs A, const unsigned long long *__restrict__ items, int64_t first, int64_t n_items,
                                               uint32_t *__restrict__ dirs, int rows_per_ext,
                                               unsigned long long *__restrict__ wide, unsigned long long *n_wide, unsigned int *work,
                                               int dp_cols) {
    __shared__ __align__(16) int8_t s_bl[21 * 32];
    __shared__ uint32_t s_ring[RING * NT];
    __shared__ uint32_t s_tr[(RING / 4) * NT];       // subject residues of the columns around the window, ring-indexed like the row
    for (int k = threadIdx.x; k < 21 * 32 / 4; k += NT) reinterpret_cast<uint32_t *>(s_bl)[k] = reinterpret_cast<const uint32_t *>(g_blosum)[k];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1;
    const int GI = GAP_OPEN, GE = GAP_EXT, GIE = GAP_OPEN + GAP_EXT;
    constexpr int LIMIT = 15, DROP = 27;
    uint32_t *hf = s_ring + threadIdx.x, *tr = s_tr + threadIdx.x;
#define RI(j) (((j) & (RING - 1)) * NT)
    bool busy = false, dry = false;
    uint32_t item = 0;
    const uint8_t *qp = nullptr, *t = nullptr;
    uint32_t *drow = nullptr;                  // directions of the current row
    int step = 1, nQ = 0, nD = 0;
    int i = 1, cs = 1, ce = LIMIT, best = 0, bcol = 0, brow = 0, cells = 0;
    int t_hi = 0, qa_next = 0;                 // columns 0 .. t_hi - 1 are (or were) in the residue ring; query residue of the next row
    for (;;) {
        const uint32_t idle = __ballot_sync(0xffffffffu, !busy && !dry);
        const uint32_t live = __ballot_sync(0xffffffffu, busy);
        if (idle && (live == 0 || __popc(idle) >= MCX_GAP_REFILL)) {
            unsigned int base = 0;
            if (lane == 0) base = atomicAdd(work, (unsigned int)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (!busy && !dry) {
                const int64_t w = (int64_t)base + __popc(idle & lt);
                if (w >= n_items) dry = true;
                else {
                    item = (uint32_t)items[first + w];
                    const ExtSetup S = ext_setup(A, item);
                    qp = S.qp; t = S.t; step = S.step; nQ = S.nQ; nD = S.nD;
                    drow = dirs + (size_t)w * (size_t)rows_per_ext * DIR_ROW_WORDS;
                    hf[0] = pack_hf(0, -GI);
#pragma unroll
                    for (int j = 1; j <= LIMIT; ++j) hf[j * NT] = pack_hf(-GI - j * GE, -GI - j * GE - GI);
                    i = 1; cs = 1; ce = LIMIT; best = 0; bcol = 0; brow = 0; cells = 0;
                    // the residue of column j sits in byte j & 63 of the ring (column 0 has none: whatever precedes the
                    // extension is loaded in its place and never used)
                    load_residues<RING / 4, NT>(t - step, step, nD + 1, tr);
                    t_hi = RING;
                    qa_next = qp[0];
                    busy = true;
                }
            }
        }
        if (__all_sync(0xffffffffu, !busy && dry)) break;
        if (busy) {
            bool fin = true, over = false;
            if (i <= nQ) {
                // every column this row can touch must fit the ring next to column cs - 1 (8 columns to spare: a word of
                // direction nibbles is written once per row)
                if (min(ce, nD) - (cs - 1) >= dp_cols) over = true;
                else {
                    const int r0 = RI(cs - 1);
                    const uint32_t w0 = hf[r0];
                    int diag = hf_h(w0);
                    const int v = __viaddmax_s32(hf_h(w0), -GIE, hf_f(w0) - GE);
                    hf[r0] = pack_hf(v, v);
                    int E = v - GI, hl = v;
                    const int8_t *brow_q = s_bl + qa_next * 32;
                    if (i < nQ) qa_next = qp[i * step];                   // a row ahead: its latency hides behind this row
                    // residues of the columns this row can reach (the tail stops 55 columns right of cs - 1 at the latest)
                    for (const int need = min(nD, cs + RING - 9); t_hi <= need; t_hi += 4) {
                        const uint8_t *tp = t + (t_hi - 1) * step;
                        tr[((t_hi & (RING - 1)) >> 2) * NT] = (uint32_t)tp[0] | ((uint32_t)tp[step] << 8) | ((uint32_t)tp[2 * step] << 16) | ((uint32_t)tp[3 * step] << 24);
                    }
                    uint32_t *dw = drow + (size_t)(i - 1) * DIR_ROW_WORDS;
                    dw[0] = (uint32_t)cs;
                    uint32_t acc = 0;
                    int cur = (cs & (RING - 1)) >> 3;
                    // main loop over columns cs .. min(ce, nD) in aligned groups of four (one word of residues, half a word of
                    // direction nibbles).  dead = the row ended at a dead cell right of the best column (then `jx` is that
                    // column); cand = rightmost dead cell at or left of the best column seen on the way (the left prune
                    // below starts from it instead of walking back over the whole row); moved = the best cell moved in
                    // this row.
                    const int jend = min(ce, nD);
                    int jx = 0, cand = cs - 1;
                    bool dead = false, moved = false;
                    if (cs <= jend) {
                        int j = cs, ro = cs & (RING - 1);
                        uint32_t tword = tr[(ro >> 2) * NT] >> (8 * (ro & 3));       // residue of the current column in the low byte
                        for (;;) {
                            const uint32_t old = hf[ro * NT];
                            const int Ho = hf_h(old), Fo = hf_f(old);
                            const int a = hl - GIE, b = E - GE;
                            uint32_t nib = a >= b ? 4u : 0u;
                            E = max(a, b);
                            const int c = Ho - GIE, d = Fo - GE;
                            nib |= c >= d ? 8u : 0u;
                            const int Fv = max(c, d);
                            int h = diag + brow_q[tword & 0xffu];
                            if (E > h) { h = E; nib |= 1u; }
                            if (h < Fv) { h = Fv; nib = (nib & 12u) | 2u; }
                            diag = Ho;
                            hf[ro * NT] = pack_hf(h, Fv);
                            hl = h;
                            const int wi = ro >> 3;
                            if (wi != cur) { dw[1 + cur] = acc; acc = 0; cur = wi; }
                            acc |= nib << (4 * (ro & 7));
                            if (h > best) { best = h; bcol = j; brow = i; moved = true; }
                            else if (h <= best - DROP) {
                                if (j > bcol) { jx = j; dead = true; break; }
                                cand = j;
                            }
                            ++j;
                            if (j > jend) break;
                            ro = (ro + 1) & (RING - 1);
                            tword >>= 8;
                            if ((ro & 3) == 0) tword = tr[(ro >> 2) * NT];
                        }
                    }
                    bool skip_tail = false;
                    if (dead) { cells += jx - cs + 1; skip_tail = jx < ce; ce = jx; }
                    else if (cs <= jend) cells += jend - cs + 1;
                    if (!skip_tail) {
                        for (int jj = ce + 1; jj <= nD; ++jj) {          // run on along the row by horizontal gaps
                            if (jj - (cs - 1) >= dp_cols) { over = true; break; }
                            ++cells;
                            const int a = hl - GIE, b = E - GE;
                            const uint32_t nib = (a > b ? 4u : 0u) | 8u | 1u;
                            E = max(a, b);
                            hf[RI(jj)] = pack_hf(E, E - GI);
                            hl = E;
                            const int wi = (jj & (RING - 1)) >> 3;
                            if (wi != cur) { dw[1 + cur] = acc; acc = 0; cur = wi; }
                            acc |= nib << (4 * (jj & 7));
                            if (E > best) { best = E; bcol = jj; brow = i; moved = true; }
                            else if (E <= best - DROP) { ce = jj; break; }
                        }
                        if (!over && cs <= bcol) {                       // drop dead cells on the left: cs = rightmost dead column <= bcol
                            // cells recorded in `cand` are dead under the final threshold as well (it only rises within a
                            // row); cells between cand and a best cell that moved may have died with the higher threshold
                            const int thr = best - DROP;
                            int nc = cand;
                            if (moved) for (int c = bcol - 1; c > cand; --c) if (hf_h(hf[RI(c)]) <= thr) { nc = c; break; }
                            if (nc >= cs) cs = nc;
                        }
                    }
                    dw[1 + cur] = acc;
                    fin = !(cs < ce) || i >= nQ;
                    ++i;
                }
            }
            if (over) {                                                  // hand the extension to the wide-row fallback
                const uint32_t am = __activemask();
                unsigned long long base = 0;
                const int leader = __ffs(am) - 1;
                if (lane == leader) base = atomicAdd(n_wide, (unsigned long long)__popc(am));
                base = __shfl_sync(am, base, leader);
                wide[base + __popc(am & lt)] = item;
                GExtRec r;
                r.gain = 0; r.eq = 0; r.et = 0; r.st = 0; r.cells = 0;
                A.ext[item] = r;
                busy = false;
            } else if (fin) {
                GExtRec r;
                r.gain = 0; r.eq = 0; r.et = 0; r.st = 0; r.cells = (uint32_t)cells;
                if (best > 0) { r.gain = best; r.eq = (uint16_t)brow; r.et = (uint16_t)bcol; }
                A.ext[item] = r;
                busy = false;
            }
        }
    }
#undef RI
}

// K3b'': walk back from the best cell of every extension k_gap_dp finished with a gain (AlignGapped's traceback, CalRes):
// identities, alignment columns, gap columns and gap runs.  One thread per extension; the steps are dependent loads
// of the direction words (L2), a few dozen per extension.
__global__ void k_gap_trace(GapArgs A, const unsigned long long *__restrict__ items, int64_t first, int64_t n_items,
                            const uint32_t *__restrict__ dirs, int rows_per_ext) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_items) return;
    const uint32_t item = (uint32_t)items[first + w];
    const GExtRec r = A.ext[item];
    if (r.gain <= 0) return;
    const ExtSetup S = ext_setup(A, item);
    const uint32_t *drow = dirs + (size_t)w * (size_t)rows_per_ext * DIR_ROW_WORDS;
    enum { C_S = 0, C_E_OPEN, C_E_EXT, C_D_OPEN, C_D_EXT, C_ORIGIN };
    // what the three trace matrices hold at (i, j): m = M, e = EM, f = FM of the oracle
    auto cell = [&](int i, int j, int &m, int &e, int &f) {
        if (i == 0) {
            if (j == 0) { m = C_ORIGIN; e = C_ORIGIN; f = C_ORIGIN; return; }
            m = e = (j == 1) ? C_E_OPEN : C_E_EXT; f = C_D_OPEN;
            return;
        }
        const uint32_t *dw = drow + (size_t)(i - 1) * DIR_ROW_WORDS;
        const int cs = (int)dw[0];
        if (j == cs - 1) { m = f = (i == 1) ? C_D_OPEN : C_D_EXT; e = (i == 1) ? C_E_OPEN : C_E_EXT; return; }
        const uint32_t nib = (dw[1 + ((j & (RING - 1)) >> 3)] >> (4 * (j & 7))) & 15u;
        e = (nib & 4u) ? C_E_OPEN : C_E_EXT;
        f = (nib & 8u) ? C_D_OPEN : C_D_EXT;
        m = (nib & 3u) == 0 ? C_S : (nib & 3u) == 1 ? e : f;
    };
    int i = r.eq, j = r.et, c = C_S, prev = -1;
    int ident = 0, aln = 0, gapcols = 0, gapruns = 0;
    while (c != C_ORIGIN && aln < 1023) {
        ++aln;
        int m, e, f;
        if (c == C_S) {
            const int qa = S.qp[(i - 1) * S.step], tb = S.t[(j - 1) * S.step];
            ident += (qa == tb && qa < 20);
            --i; --j; prev = 0;
            cell(i, j, m, e, f);
            c = m;
        } else if (c == C_D_OPEN || c == C_D_EXT) {
            ++gapcols; gapruns += (prev != 1); prev = 1;
            --i;
            cell(i, j, m, e, f);
            c = (c == C_D_OPEN) ? m : f;
        } else {
            ++gapcols; gapruns += (prev != 2); prev = 2;
            --j;
            cell(i, j, m, e, f);
            c = (c == C_E_OPEN) ? m : e;
        }
    }
    A.ext[item].st = (uint32_t)ident | ((uint32_t)aln << 8) | ((uint32_t)gapcols << 17) | ((uint32_t)gapruns << 26);
}

// K3b (fallback for extensions whose live window outgrows the ring of k_gap_dp; the first version of the stage): the DP
// itself, one LANE per gapped extension (one direction of one survivor), rows in local memory; a lane that
// finishes its extension draws the next one from the work list instead of idling until the longest extension of its
// warp is done -- the X-drop decides the size of an extension and nothing known beforehand predicts it (the first
// version, one thread per list entry, ran at 9-10 of 32 lanes: 2.72 -> 2.08 ms at 100 bp, 6.12 -> 4.80 at 150 bp).
// Resident blocks; every trip of the warp loop advances each busy lane by ONE row of its own extension; idle lanes are
// refilled together once MCX_GAP_REFILL of them wait (a refill is three dependent loads plus row 0, issued for the whole
// warp whatever the number of lanes that need it; measured 1 / 4 / 8 / 16 / 24 / 28: 5.69 / 5.50 / 5.28 / 5.19 / 4.80 /
// 4.80 ms at 150 bp, flat at 100 bp).
// First a score-only pass over all extensions (two DP rows); only the ~16 % that gain anything are queued for the
// second pass, which repeats the same DP carrying the alignment statistics and stops at the row of the best cell.
// (Tried and measured slower on 2M x 100 bp: rows in shared memory, column-major and conflict-free -- 6.8 ms instead
// of 4.9, the 53-80 KB per block leave too few warps to hide the serial dependency of the cells; packed (H, F) cells
// with the next cell prefetched -- no change; rows as a 64-column ring -- slower at every length.)
template <int NT, int GROW, bool STATS>
__global__ void __launch_bounds__(NT) k_gap_dir(GapArgs A, const unsigned long long *__restrict__ items, const unsigned long long *n_items_dev,
                                                unsigned long long *__restrict__ items2, unsigned long long *n_items2,
                                                unsigned int *work) {
    const int64_t n_items = (int64_t)*n_items_dev;
    if (n_items == 0) return;
    __shared__ __align__(16) int8_t s_bl[21 * 32];
    for (int k = threadIdx.x; k < 21 * 32 / 4; k += NT) reinterpret_cast<uint32_t *>(s_bl)[k] = reinterpret_cast<const uint32_t *>(g_blosum)[k];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1;
    const int GI = GAP_OPEN, GE = GAP_EXT, GIE = GAP_OPEN + GAP_EXT;
    const int limit = 15;                      // (int)((26.98 - 11) / 1)
    int H[GROW], F[GROW];
    uint32_t HS[STATS ? GROW : 1], FS[STATS ? GROW : 1];
    bool busy = false, dry = false;            // dry: the work list has nothing left for this lane
    uint32_t item = 0;
    const uint8_t *qp = nullptr, *t = nullptr; // residue of row i is qp[(i - 1) * step], of column j is t[(j - 1) * step]
    int step = 1, nQ = 0, nD = 0;
    int i = 1, cs = 1, ce = limit, best = 0, bcol = 0, brow = 0, cells = 0;
    uint32_t bst = 0;
    for (;;) {
        const uint32_t idle = __ballot_sync(0xffffffffu, !busy && !dry);
        const uint32_t live = __ballot_sync(0xffffffffu, busy);
        if (idle && (live == 0 || __popc(idle) >= MCX_GAP_REFILL)) {
            unsigned int base = 0;
            if (lane == 0) base = atomicAdd(work, (unsigned int)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (!busy && !dry) {
                const int64_t w = (int64_t)base + __popc(idle & lt);
                if (w >= n_items) dry = true;
                else {
                    item = (uint32_t)items[w];
                    const int64_t g = item >> 1;
                    const Surv v = surv_unpack(A.surv[A.first + g]);
                    const uint8_t *fr = A.frames + (int64_t)v.gframe * A.fstride;
                    const int m = (A.L - v.frame % 3) / 3;
                    const int32_t o = A.db.off[v.subject];
                    const int n = A.db.off[v.subject + 1] - o;
                    const int q0 = v.q0, q1 = v.q1, t0 = v.t0, t1 = v.t0 + (v.q1 - v.q0);
                    // the statistics pass stops with the row of the best cell found by the score pass
                    int row_limit = 1 << 30;
                    if (STATS) row_limit = A.ext[item].eq;
                    int ql, tl;
                    if ((item & 1) == 0) { ql = m - (q1 + 1); tl = n - (t1 + 1); qp = fr + q1 + 1; t = A.db.res + o + t1 + 1; step = 1; }
                    else { ql = q0; tl = t0; qp = fr + q0 - 1; t = A.db.res + o + t0 - 1; step = -1; }
                    if (tl > ql + GAP_SLACK) tl = ql + GAP_SLACK;
                    nQ = min(ql, row_limit); nD = tl;
                    H[0] = 0; F[0] = -GI;
                    if (STATS) { HS[0] = 0; FS[0] = 0; }
                    // row 0: the binary fills min(limit, nD) cells of it; the ones past nD are never read
#pragma unroll
                    for (int j = 1; j <= limit; ++j) {
                        H[j] = -GI - j * GE; F[j] = -GI - j * GE - GI;
                        if (STATS) { HS[j] = (uint32_t)j * (ST_ALN + ST_GAPCOL) + ST_GAPRUN; FS[j] = HS[j]; }
                    }
                    i = 1; cs = 1; ce = limit; best = 0; bcol = 0; brow = 0; cells = 0; bst = 0;
                    busy = true;
                }
            }
        }
        if (__all_sync(0xffffffffu, !busy && dry)) break;
        bool again = false;
        if (busy) {
            bool fin = true;
            if (i <= nQ) {
                int diag = H[cs - 1];
                uint32_t dst = 0, bs = 0;
                if (STATS) {
                    dst = HS[cs - 1];
                    bs = (i == 1 ? HS[cs - 1] + ST_GAPRUN : FS[cs - 1]) + ST_ALN + ST_GAPCOL;
                }
                int v = H[cs - 1] - GIE, f1 = F[cs - 1] - GE;
                if (v < f1) v = f1;
                F[cs - 1] = v; H[cs - 1] = v;
                if (STATS) { HS[cs - 1] = bs; FS[cs - 1] = bs; }
                int E = v - GI, hl = v, j = cs;
                uint32_t ES = bs, hls = bs;
                bool skip_tail = false;
                const int qa = qp[(i - 1) * step];
                const int8_t *brow_q = s_bl + qa * 32;
                if (!(cs > ce || cs > nD)) {
                    for (;;) {
                        ++cells;
                        int a = hl - GIE, b = E - GE;
                        if (a >= b) { E = a; if (STATS) ES = hls + ST_ALN + ST_GAPCOL + ST_GAPRUN; } else { E = b; if (STATS) ES += ST_ALN + ST_GAPCOL; }
                        int c = H[j] - GIE, d = F[j] - GE, Fv;
                        uint32_t FSv = 0;
                        if (c >= d) { Fv = c; if (STATS) FSv = HS[j] + ST_ALN + ST_GAPCOL + ST_GAPRUN; } else { Fv = d; if (STATS) FSv = FS[j] + ST_ALN + ST_GAPCOL; }
                        const int tb = t[(j - 1) * step];
                        int h = diag + brow_q[tb];
                        uint32_t hs = 0;
                        if (STATS) hs = dst + ST_ALN + (uint32_t)(qa == tb && qa < 20);
                        if (E > h) { h = E; hs = ES; }
                        if (h < Fv) { h = Fv; hs = FSv; }
                        diag = H[j];
                        if (STATS) dst = HS[j];
                        H[j] = h; F[j] = Fv; hl = h;
                        if (STATS) { HS[j] = hs; FS[j] = FSv; hls = hs; }
                        if (h > best) { best = h; bcol = j; brow = i; bst = hs; }
                        else if (h <= best - 27 && j > bcol) {       // h < best - 26.98
                            if (j >= ce) { ce = j; break; }
                            ce = j; skip_tail = true; break;
                        }
                        ++j;
                        if (j > nD || j > ce) break;
                    }
                }
                if (!skip_tail) {
                    for (int jj = ce + 1; jj <= nD; ++jj) {          // run on along the row by horizontal gaps
                        ++cells;
                        int a = hl - GIE, b = E - GE;
                        if (a > b) { E = a; if (STATS) ES = hls + ST_ALN + ST_GAPCOL + ST_GAPRUN; } else { E = b; if (STATS) ES += ST_ALN + ST_GAPCOL; }
                        H[jj] = E; F[jj] = E - GI; hl = E;
                        if (STATS) { HS[jj] = ES; FS[jj] = ES; hls = ES; }
                        if (E > best) { best = E; bcol = jj; brow = i; bst = ES; }
                        else if (E <= best - 27) { ce = jj; break; }
                    }
                    if (cs <= bcol) {                                // drop dead cells on the left
                        int thr = best - 27;
                        if (H[bcol] <= thr) cs = bcol;
                        else for (int c = bcol - 1; c >= cs; --c) if (H[c] <= thr) { cs = c; break; }
                    }
                }
                fin = !(cs < ce) || i >= nQ;
                ++i;
            }
            if (fin) {
                if (STATS) {
                    A.ext[item].st = best > 0 ? bst : 0u;
                } else {
                    GExtRec r;
                    r.gain = 0; r.eq = 0; r.et = 0; r.st = 0; r.cells = (uint32_t)cells;
                    if (best > 0) { r.gain = best; r.eq = (uint16_t)brow; r.et = (uint16_t)bcol; }
                    A.ext[item] = r;
                    again = best > 0;
                }
                busy = false;
            }
        }
        if (!STATS) {
            const uint32_t ma = __ballot_sync(0xffffffffu, again);
            if (ma) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(n_items2, (unsigned long long)__popc(ma));
                base = __shfl_sync(0xffffffffu, base, 0);
                // the statistics pass repeats this DP: most cells first
                if (again) items2[base + __popc(ma & lt)] = ((unsigned long long)(65535u - (uint32_t)min(cells, 65535)) << 32) | item;
            }
        }
    }
}

// K3c: one thread per survivor: add the two extensions to the ungapped HSP, write the HSP record and its sort key
__global__ void k_gap_finish(GapArgs A) {
    int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= A.n_surv) return;
    const GExtRec ef = A.ext[2 * g], eb = A.ext[2 * g + 1];
    g += A.first;
    const Surv v = surv_unpack(A.surv[g]);
    int q0 = v.q0, q1 = v.q1, t0 = v.t0, t1 = v.t0 + (v.q1 - v.q0);
    int score = v.score, ident = v.ident, aln = q1 - q0 + 1, gapcols = 0, gapo = 0;
    if (ef.gain > 0) {
        score += ef.gain; q1 += ef.eq; t1 += ef.et;
        ident += ef.st & 0xff; aln += (ef.st >> 8) & 0x1ff; gapcols += (ef.st >> 17) & 0x1ff; gapo += ef.st >> 26;
    }
    if (eb.gain > 0) {
        score += eb.gain; q0 -= eb.eq; t0 -= eb.et;
        ident += eb.st & 0xff; aln += (eb.st >> 8) & 0x1ff; gapcols += (eb.st >> 17) & 0x1ff; gapo += eb.st >> 26;
    }
    {   // counters: one atomic per warp, not per survivor (2M atomics on one address were half of this kernel)
        const uint32_t am = __activemask();
        const unsigned nc = __reduce_add_sync(am, ef.cells + eb.cells);
        const unsigned ng = __reduce_add_sync(am, (unsigned)((ef.gain > 0) + (eb.gain > 0)));
        if ((threadIdx.x & 31) == __ffs(am) - 1) {
            if (nc) atomicAdd(&A.counters[1], (unsigned long long)nc);
            if (ng) atomicAdd(&A.counters[0], (unsigned long long)ng);
        }
    }
    mcx_hit h;
    h.read = v.read; h.subject = v.subject; h.frame = v.frame; h.score = score;
    h.aln = aln; h.ident = ident; h.mism = aln - ident - gapcols; h.gapo = gapo;
    h.q0 = q0; h.q1 = q1; h.t0 = t0; h.t1 = t1;
    {   // 48-byte record as three 128-bit stores
        uint4 *dst = reinterpret_cast<uint4 *>(A.hsp + g);
        dst[0] = make_uint4((uint32_t)h.read, (uint32_t)h.subject, (uint32_t)h.frame, (uint32_t)h.score);
        dst[1] = make_uint4((uint32_t)h.aln, (uint32_t)h.ident, (uint32_t)h.mism, (uint32_t)h.gapo);
        dst[2] = make_uint4((uint32_t)h.q0, (uint32_t)h.q1, (uint32_t)h.t0, (uint32_t)h.t1);
    }
    // Sort key = every field the classifier needs, in the order that decides which of several overlapping HSPs of a
    // (read, subject) pair is printed: score, then -- for alignments of equal score grown from different seeds --
    // the longest, then the one from the leftmost ungapped HSP (RAPsearch2's choice, tools/blackbox/tie_rule.py).
    SortKey k;
    k.k1 = ((unsigned long long)(uint32_t)v.read << 37) | ((unsigned long long)v.subject << 22) |
           ((unsigned long long)(2047 - score) << 11) | ((unsigned long long)(511 - aln) << 2);
    k.k2 = ((unsigned long long)v.q0 << 56) | ((unsigned long long)v.frame << 53) | ((unsigned long long)q0 << 45) |
           ((unsigned long long)q1 << 37) | ((unsigned long long)t0 << 26) | ((unsigned long long)t1 << 15) |
           ((unsigned long long)ident << 6);
    A.keys[g] = k;
    A.idx[g] = (int32_t)g;
}

// ------------------------------------------------------------------------------------------------
// K4: per read -- HSP de-duplication, cutoffs, best hit, per-family sums.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void dna_coords(int L, int frame, int q0, int q1, int &qs, int &qe) {
    int a0 = q0 + 1, a1 = q1 + 1;
    if (frame < 3) { qs = 3 * (a0 - 1) + frame + 1; qe = 3 * a1 + frame; }
    else { int o = frame - 3; qs = L - o - 3 * (a0 - 1); qe = L - o - 3 * a1 + 1; }
}

// mc.py:400-418 operation for operation in IEEE double (compiled with -fmad=false)
__device__ double alignment_coverage(int L, int qs_, int qe_, int t0, int t1, int aln_, int tlen) {
    double query_len = (double)L / 3;
    double qs = (double)(qs_ < qe_ ? qs_ : qe_), qe = (double)(qs_ < qe_ ? qe_ : qs_);
    int fmi = (qs_ < qe_ ? qs_ : qe_) % 3;
    double frame = (fmi == 1 || fmi == 2) ? (double)fmi : 3.0;
    double query_start = (qs + 3 - frame) / 3;
    double query_stop = (qe + 1 - frame) / 3;
    double a = (double)t0 + 1, b = (double)t1 + 1;
    double target_start = a < b ? a : b, target_stop = a < b ? b : a;
    double x = (query_start - 1 < target_start - 1) ? query_start - 1 : target_start - 1;
    double y = (double)aln_;
    double tl = (double)tlen;
    double z = (query_len - query_stop < tl - target_stop) ? query_len - query_stop : tl - target_stop;
    double maxaln = x + y + z;
    return (double)aln_ / maxaln;
}

// The sorted key of an HSP (k_gap_finish) holds every field the classifier needs, so K4 streams the 16-byte keys in
// sorted order and never gathers the 48-byte records.
struct KeyHit { int read, subject, score, frame, q0, q1, t0, t1, aln, ident; };
__device__ __forceinline__ KeyHit key_decode(const SortKey &k) {
    KeyHit h;
    h.read = (int)(k.k1 >> 37); h.subject = (int)(k.k1 >> 22) & 0x7fff; h.score = 2047 - ((int)(k.k1 >> 11) & 0x7ff);
    h.aln = 511 - ((int)(k.k1 >> 2) & 0x1ff);
    h.frame = (int)(k.k2 >> 53) & 7; h.q0 = (int)(k.k2 >> 45) & 0xff; h.q1 = (int)(k.k2 >> 37) & 0xff;
    h.t0 = (int)(k.k2 >> 26) & 0x7ff; h.t1 = (int)(k.k2 >> 15) & 0x7ff; h.ident = (int)(k.k2 >> 6) & 0x1ff;
    return h;
}

struct ClsArgs {
    const SortKey *keys;           // sorted: (read, subject, score desc, ...)
    int64_t n;
    int L;
    int min_report;
    DevDB db;
    uint8_t *keep;                 // per sorted position: 1 = reported line
    int32_t *caplist;              // sorted positions of the first HSP of reads with more than 500 reported lines
    unsigned long long *n_cap;
    int32_t *nrep;                 // per pushed read: reported lines (before the 500-line cap), zeroed
    unsigned long long *bestkey;   // per pushed read: (score + 1) << 32 | ~position of the best passing line, zeroed
    int32_t *best_subject;         // per pushed read
    unsigned long long *acc;       // [0] reads_with_hits [1] classified [2] n_hsp, then fam_hits[30], fam_aln[30]
    unsigned long long *aln_by_len;
};

// K4a: one thread per (read, subject) group of the sorted list (1-2 HSPs almost always): which HSPs are printed -- at
// or above the floor and, in score order, disjoint in query and subject range from every HSP already kept for that
// subject.
__global__ void k_cls_groups(ClsArgs A) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= A.n) return;
    const unsigned long long grp = A.keys[p].k1 >> 22;
    if (p > 0 && (A.keys[p - 1].k1 >> 22) == grp) return;
    int nk = 0, nrep = 0;
    int kqs[8], kqe[8], kt0[8], kt1[8];
    for (int64_t e = p; e < A.n; ++e) {
        const SortKey k = A.keys[e];
        if ((k.k1 >> 22) != grp) break;
        const KeyHit h = key_decode(k);
        int qs, qe;
        dna_coords(A.L, h.frame, h.q0, h.q1, qs, qe);
        const int lo = qs < qe ? qs : qe, hi = qs < qe ? qe : qs;
        bool keep = h.score >= A.min_report;
        for (int j = 0; j < nk && keep; ++j)
            if (!(hi < kqs[j] || kqe[j] < lo) || !(h.t1 < kt0[j] || kt1[j] < h.t0)) keep = false;
        A.keep[e] = keep;
        if (!keep) continue;
        if (nk < 8) { kqs[nk] = lo; kqe[nk] = hi; kt0[nk] = h.t0; kt1[nk] = h.t1; ++nk; }
        ++nrep;
    }
    if (nrep) atomicAdd(&A.nrep[(int)(grp >> 15)], nrep);
}

// K4b: one thread per read of the sorted list: count it; reads with more than 500 reported lines go on a list.
__global__ void k_cls_cap(ClsArgs A) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int nrep = 0;
    if (p < A.n) {
        const int read = (int)(A.keys[p].k1 >> 37);
        if (p == 0 || (int)(A.keys[p - 1].k1 >> 37) != read) nrep = A.nrep[read];
        if (nrep > MAX_LINES) {
            A.caplist[atomicAdd(A.n_cap, 1ull)] = (int32_t)p;
            nrep = MAX_LINES;
        }
    }
    const uint32_t any = __ballot_sync(0xffffffffu, nrep > 0);
    if (!any) return;
    const int lines = __reduce_add_sync(0xffffffffu, nrep);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&A.acc[0], (unsigned long long)__popc(any)); atomicAdd(&A.acc[2], (unsigned long long)lines); }
}

// K4b': RAPsearch2 prints at most 500 lines per query (-v default), best first: keep the 500 highest scores, ties
// at the cut score in (subject, ...) order.  One warp per listed read: score histogram in shared memory, cut score
// from its suffix sums, then the ties in sorted order.  (First version: one thread per read bisecting the cut score
// with 11 passes over its HSPs -- 1 ms for a few hundred reads.)
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) k_cls_cap_apply(ClsArgs A) {
    __shared__ int s_hist[WARPS][2048];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int *hist = s_hist[warp];
    const unsigned long long ncap = *A.n_cap;
    for (unsigned long long q = (unsigned long long)blockIdx.x * WARPS + warp; q < ncap; q += (unsigned long long)gridDim.x * WARPS) {
        const int64_t p = A.caplist[q];
        const int read = (int)(A.keys[p].k1 >> 37);
        for (int k = lane; k < 2048; k += 32) hist[k] = 0;
        __syncwarp();
        int64_t end = p;
        for (;; end += 32) {                                 // histogram of the kept scores; finds the end of the read
            const int64_t e = end + lane;
            const bool mine = e < A.n && (int)(A.keys[e].k1 >> 37) == read;
            if (mine && A.keep[e]) atomicAdd(&hist[key_decode(A.keys[e]).score], 1);
            const uint32_t bm = __ballot_sync(0xffffffffu, mine);
            if (bm != 0xffffffffu) { end += __popc(bm); break; }
        }
        __syncwarp();
        int T = 0, above = 0, run = 0;                       // largest T with count(score >= T) >= 500
        for (int top = 2047; top >= 0; top -= 32) {
            const int c = hist[top - lane];
            int inc = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
            const uint32_t hit = __ballot_sync(0xffffffffu, run + inc >= MAX_LINES);
            if (hit) {
                const int l = __ffs(hit) - 1;
                T = top - l;
                above = run + __shfl_sync(0xffffffffu, inc - c, l);
                break;
            }
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
        const int allow = MAX_LINES - above;
        int taken = 0;
        for (int64_t base = p; base < end; base += 32) {     // ties at T in sorted order
            const int64_t e = base + lane;
            bool tie = false;
            if (e < end && A.keep[e]) {
                const int sc = key_decode(A.keys[e]).score;
                if (sc < T) A.keep[e] = 0;
                tie = sc == T;
            }
            const uint32_t tm = __ballot_sync(0xffffffffu, tie);
            if (tie && taken + __popc(tm & ((1u << lane) - 1)) >= allow) A.keep[e] = 0;
            taken += __popc(tm);
        }
        __syncwarp();
    }
}

// K4c: one thread per HSP: the three cutoffs of its subject's family (mc.py:420-430); the best passing line of a
// read is the highest score, first in sorted order on ties (mc.py:450-453) -- one atomicMax per passing line.
__global__ void k_cls_filter(ClsArgs A) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= A.n || !A.keep[p]) return;
    const KeyHit h = key_decode(A.keys[p]);
    int qs, qe;
    dna_coords(A.L, h.frame, h.q0, h.q1, qs, qe);
    const int fam = A.db.fam[h.subject];
    const int slen = A.db.off[h.subject + 1] - A.db.off[h.subject];
    const mcx_cutoff c = c_cut[fam];
    if (alignment_coverage(A.L, qs, qe, h.t0, h.t1, h.aln, slen) < c.min_cov) return;
    if (h.score < c.min_raw) return;
    if ((double)(100 * h.ident) > c.max_aaid * (double)h.aln) return;
    atomicMax(&A.bestkey[h.read], ((unsigned long long)(h.score + 1) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)p));
}

// K4d: one thread per read of the sorted list: per-family sums of the classified reads (mc.py:462-472)
__global__ void k_cls_sum(ClsArgs A) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= A.n) return;
    const int read = (int)(A.keys[p].k1 >> 37);
    if (p > 0 && (int)(A.keys[p - 1].k1 >> 37) == read) return;
    const unsigned long long b = A.bestkey[read];
    if (!b) return;
    const KeyHit h = key_decode(A.keys[0xffffffffu - (uint32_t)b]);
    const int fam = A.db.fam[h.subject];
    const int slen = A.db.off[h.subject + 1] - A.db.off[h.subject];
    atomicAdd(&A.acc[1], 1ull);
    atomicAdd(&A.acc[3 + fam], 1ull);
    atomicAdd(&A.acc[3 + MCX_N_FAM + fam], (unsigned long long)h.aln);
    atomicAdd(&A.aln_by_len[fam * MCX_LEN_BINS + slen], (unsigned long long)h.aln);
    A.best_subject[read] = h.subject;
}

__global__ void k_fill_i32(int32_t *p, int64_t n, int32_t v) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void k_gather_hits(const mcx_hit *__restrict__ hsp, const int32_t *__restrict__ idx,
                              const uint8_t *__restrict__ keep, const int32_t *__restrict__ pos, int64_t n,
                              mcx_hit *__restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && keep[i]) out[pos[i]] = hsp[idx[i]];
}
__global__ void k_keep_sorted(const uint8_t *__restrict__ keep, int64_t n, int32_t *__restrict__ flag) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = keep[i];
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
constexpr int MAX_COPY_STEPS = 64;             // host->device copies of a push are cut into at most this many steps
struct mcx_ctx;
static int fail(mcx_ctx *ctx, int code, const std::string &msg);
#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(ctx, MCX_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));       \
    } while (0)
#define TRY(call)                                                                                  \
    do { const int rc_ = (call); if (rc_ != MCX_OK) return rc_; } while (0)

template <typename T>
static cudaError_t dev_alloc(T **p, size_t n) { return cudaMalloc((void **)p, n * sizeof(T) ? n * sizeof(T) : 1); }

// a device buffer with its capacity in entries; a borrowed one (caller's storage, mcx_push_reads*_dev) has capacity 0,
// is never freed here, and the next ensure() replaces it with storage of the context's own
template <typename T>
struct DevBuf {
    T *p = nullptr;
    int64_t cap = 0;
    bool owned = true;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { if (owned && p) cudaFree(p); }
    operator T *() const { return p; }
    int release(mcx_ctx *ctx) {
        if (owned && p) CK(cudaFree(p));
        p = nullptr; cap = 0; owned = true;
        return MCX_OK;
    }
    // room for `need` entries, contents not kept: free, then allocate need + need/8 + slack; *grew: it reallocated
    int ensure(mcx_ctx *ctx, int64_t need, bool *grew = nullptr, int64_t slack = 16) {
        if (grew) *grew = false;
        if (cap >= need && p) return MCX_OK;
        TRY(release(ctx));
        CK(dev_alloc(&p, (size_t)(need + need / 8 + slack)));
        cap = need + need / 8 + slack;
        if (grew) *grew = true;
        return MCX_OK;
    }
    // exactly `cap` entries, the first `keep` copied over (on the context's stream, waited for before the old one is freed)
    int grow_keep(mcx_ctx *ctx, int64_t keep, int64_t cap);
    int borrow(mcx_ctx *ctx, T *q) {
        TRY(release(ctx));
        p = q; owned = false;
        return MCX_OK;
    }
};

// events of the context's streams, named by the point they mark (0: start of a span, 1: end)
enum Ev { EV_QC0, EV_QC1, EV_KQC0, EV_KQC1, EV_DEDUP0, EV_DEDUP1, EV_H2D0, EV_LENS, EV_H2D1, EV_FRAMES0, EV_SEG0, EV_PROBE0, EV_KPROBE1,
          EV_SEED0, EV_KSEED1, EV_GAP0, EV_GAP1, EV_SORT0, EV_CLS0, EV_D2H0, EV_D2H1, EV_BENCH0, EV_BENCH1 /* microbenchmarks */, EV_N };
// slots of mcx_timings (include/mcx.h) and of mcx_timings_detail
enum Ms { MS_H2D, MS_QC, MS_PROBE, MS_GAPPED, MS_SORT, MS_CLASSIFY, MS_D2H, MS_EXTEND, MS_FRAMES, MS_SEG, MS_KQC, MS_DEDUP, MS_N };
enum MsDetail { MSD_KPROBE, MSD_KRESOLVE, MSD_KSEED, MSD_KWALK, MSD_N };
static_assert(MS_N == 12 && MSD_N == 4, "mcx_timings fills 12 slots, mcx_timings_detail 4");

struct mcx_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;             // kernels
    cudaStream_t copy_stream = nullptr;        // host -> device copies of pushed reads (overlap the search of earlier chunks)
    bool own_stream = true;
    std::string err;
    mcx_params par{};
    bool have_par = false;
    // database
    DevDB db{};
    std::vector<void *> db_allocs;
    // read store (see ReadStore)
    int64_t n_reads = 0, n_words = 0, n_bases = 0;
    DevBuf<uint32_t> d_pk, d_len;
    DevBuf<int64_t> d_woff, d_qoff;
    DevBuf<uint8_t> d_quals;
    bool have_quals = false;
    // ASCII staging of mcx_push_reads / mcx_push_reads_dev
    DevBuf<uint8_t> d_ascii;
    DevBuf<int64_t> d_aoffs;
    // progress of the host -> device copies: step k covers packed words [k * step_words, ...) and quality bytes
    // [k * step_qbytes, ...); ev_copy[k] is recorded behind it on the copy stream
    int n_steps = 0;                           // 0: nothing to wait for (device-resident push, or everything already waited on)
    int steps_waited = 0;
    int64_t step_words = 0, step_qbytes = 0;
    cudaEvent_t ev_copy[MAX_COPY_STEPS] = {nullptr};
    // QC state
    DevBuf<uint8_t> d_code;
    DevBuf<FpKey> d_fp;
    DevBuf<unsigned long long> d_fpa, d_fpa2;
    DevBuf<uint32_t> d_fpi, d_fpi2;
    DevBuf<int32_t> d_kept;
    // fingerprints of the reads kept by earlier pushes of the run (streamed -d)
    DevBuf<unsigned long long> d_store_a, d_store_b;
    int64_t n_store = 0;
    // cross-GPU -d exchange
    DevBuf<long long> d_xsend;
    DevBuf<uint8_t> d_xmarks;
    DevBuf<unsigned long long> d_xkg;
    DevBuf<uint32_t> d_xvi;
    int64_t x_nsend = 0;
    int64_t qc_upto = 0;                       // reads [0, qc_upto) have their verdict
    bool dedup_done = false, fp_done = false, counts_valid = false, kqc_pending = false;
    bool h2d_timed = false;                    // the last push recorded its copy events (host pushes only)
    mcx_qc qc{};
    bool pushed = false, searched = false;
    // search buffers
    DevBuf<uint4> d_surv;
    DevBuf<uint8_t> d_frames;
    DevBuf<uint32_t> d_segq, d_segm;
    DevBuf<unsigned long long> d_seen;         // k_walk's duplicate filter
    DevBuf<uint4> d_seedq;                     // accepted seeds between k_seed and k_walk
    DevBuf<unsigned long long> d_gitems;       // gapped work lists: three regions of 2 * survivors entries
    DevBuf<GExtRec> d_gext;
    DevBuf<uint32_t> d_dirs;                   // direction nibbles of k_gap_dp for k_gap_trace
    DevBuf<Cand> d_cand, d_passq;
    DevBuf<mcx_hit> d_hsp, d_hits_out;
    DevBuf<SortKey> d_keys;
    DevBuf<int32_t> d_idx, d_best, d_hflag, d_hpos;
    DevBuf<uint8_t> d_keep;
    DevBuf<int32_t> d_nrep;
    DevBuf<unsigned long long> d_bestkey;
    DevBuf<unsigned long long> d_cnt;          // 64 scalar counters (layout: enum Cnt)
    int n_sm = 148;                            // multiprocessors of the device (sizes the resident grids)
    DevBuf<unsigned long long> d_qcnt;         // NQ candidate sub-queue fills, then NQ filter-pass sub-queue fills
    DevBuf<unsigned long long> d_acc;          // 3 + 60
    DevBuf<unsigned long long> d_abl;          // 30 * 1280
    unsigned long long *h_cnt = nullptr;       // pinned mirror for counter read-backs (64 + NQ)
    DevBuf<uint8_t> d_temp;                    // CUB's temporary storage (cub_run)
    mcx_result res{};
    float ms[MS_N] = {0};
    float ms_detail[MSD_N] = {0};
    int64_t work[8] = {0};                     // mcx_search_counters of the last search
    int64_t launches = 0, host_syncs = 0;
    cudaEvent_t ev[EV_N] = {nullptr};
};
// slots of d_cnt
enum Cnt { C_QC0 = 0 /* ..3: verdict counts of the search */, C_QCALL = 4 /* ..7: verdict counts over all pushed reads */,
           C_SURV = 8, C_SEEDQ = 9, C_GAPPED = 10, C_CELLS = 11, C_SEGQ = 12, C_WORK = 13, C_ITEMS2 = 14, C_NCAP = 15,
           C_WORK1 = 16, C_WORK2 = 17, C_ITEMS = 18, C_NKEPT = 20, C_NWIDE = 24 /* ..26 */, C_NGAPTOT = 27, C_NFP = 21, C_TOTW = 22, C_TOTQ = 23,
           C_NSTORE = 28, C_XCNT = 64 /* ..191: owner counts and cursors of the -d exchange */, C_N = 192 };

static thread_local std::string g_err;

// elapsed time between two events, 0 when either was never recorded; never leaves an error behind (CUB aborts its next
// dispatch when cudaPeekAtLastError() still holds the "invalid resource handle" of such a call: a scan that silently did
// not run once left stale record offsets for the next push)
static float elapsed_ms(cudaEvent_t a, cudaEvent_t b) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, a, b) != cudaSuccess) { (void)cudaGetLastError(); return 0.f; }
    return t;
}

static int fail(mcx_ctx *ctx, int code, const std::string &msg) {
    if (ctx) ctx->err = msg;
    g_err = msg;
    return code;
}

template <typename T>
int DevBuf<T>::grow_keep(mcx_ctx *ctx, int64_t keep, int64_t c) {
    T *q = nullptr;
    CK(dev_alloc(&q, (size_t)c));
    if (p && keep > 0) CK(cudaMemcpyAsync(q, p, (size_t)keep * sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    TRY(release(ctx));
    p = q; cap = c;
    return MCX_OK;
}

// survivor-sized buffers: keep the first `keep` entries of the ones that carry state across chunks
static int grow_survivors(mcx_ctx *ctx, int64_t keep, int64_t cap) {
    TRY(ctx->d_surv.grow_keep(ctx, keep, cap));
    TRY(ctx->d_hsp.grow_keep(ctx, keep, cap));
    TRY(ctx->d_keys.grow_keep(ctx, keep, cap));
    TRY(ctx->d_idx.grow_keep(ctx, keep, cap));
    TRY(ctx->d_hits_out.grow_keep(ctx, 0, cap));
    TRY(ctx->d_hflag.grow_keep(ctx, 0, cap + 1));
    TRY(ctx->d_hpos.grow_keep(ctx, 0, cap + 1));
    TRY(ctx->d_keep.grow_keep(ctx, 0, cap));
    return MCX_OK;
}

// a CUB call in its two phases: the temporary storage it asks for, then the call itself on ctx->d_temp
template <typename F>
static int cub_run(mcx_ctx *ctx, const char *what, F call) {
    size_t tb = 0;
    cudaError_t e = call(nullptr, tb);
    if (e == cudaSuccess) {
        TRY(ctx->d_temp.ensure(ctx, (int64_t)tb, nullptr, 256));
        e = call(ctx->d_temp.p, tb);
    }
    if (e != cudaSuccess) return fail(ctx, MCX_ECUDA, std::string(what) + ": " + cudaGetErrorString(e));
    return MCX_OK;
}

// blocks of `kernel` that are resident on the device at once (at least one per multiprocessor)
template <typename K>
static int resident_blocks(mcx_ctx *ctx, K kernel, int nt, size_t smem, unsigned &blocks) {
    int per_sm = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, nt, smem));
    blocks = (unsigned)(std::max(per_sm, 1) * ctx->n_sm);
    return MCX_OK;
}

extern "C" const char *mcx_version(void) { return "mcx 0.1 (sm_100a)"; }
extern "C" const char *mcx_last_error(mcx_ctx *ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

#ifndef MCX_SLOT_ROOM_X10
#define MCX_SLOT_ROOM_X10 20               /* slots per distinct word x 10, rounded up to a power of two: 2^22 slots for 1.21 M words */
#endif
// seed index: one open-addressing table per word pattern over the murphy10 letters of the database
static int build_index(mcx_ctx *ctx, const mcx_db *db) {
    const int ns = db->n_subj;
    const int64_t nres = db->off[ns];
    std::vector<uint8_t> red((size_t)nres);
    for (int64_t g = 0; g < nres; ++g) red[(size_t)g] = db->res[g] < 20 ? MURPHY10[db->res[g]] : 10;
    for (int s = 0; s < ns; ++s)
        if (db->off[s + 1] - db->off[s] >= 2048) return fail(ctx, MCX_EINVAL, "subject longer than 2047 residues");
    // the five patterns are independent: one host thread each (entries + sort, then table fill into its own region)
    std::vector<uint32_t> filt_a((size_t)4 << FILT_BITS, 0u), filt_b((size_t)2 << FILT_BITS, 0u);
    std::vector<unsigned long long> ent[N_PAT];
    size_t distinct[N_PAT] = {0}, long_lists[N_PAT] = {0};
    auto collect = [&](int p) {
        std::vector<unsigned long long> &en = ent[p];
        en.reserve((size_t)nres);
        for (int s = 0; s < ns; ++s) {
            const int n = db->off[s + 1] - db->off[s];
            const uint8_t *r = red.data() + db->off[s];
            for (int j = 0; j + PAT_LEN[p] <= n; ++j) {
                uint32_t c = 0; bool ok = true;
                for (int k = 0; k < PAT_LEN[p]; ++k) {
                    if (k == PAT_WILD[p]) continue;
                    if (r[j + k] >= 10) { ok = false; break; }
                    c = c * 10 + r[j + k];
                }
                if (ok) en.push_back(((unsigned long long)c << 32) | ((uint32_t)s << 11) | (uint32_t)j);
            }
        }
        std::sort(en.begin(), en.end());
        for (size_t k = 0; k < en.size();) {
            size_t e = k;
            while (e + 1 < en.size() && (en[e + 1] >> 32) == (en[k] >> 32)) ++e;
            ++distinct[p];
            long_lists[p] += (e - k + 1 > 127);
            k = e + 1;
        }
    };
    {
        std::vector<std::thread> th;
        for (int p = 0; p < N_PAT; ++p) th.emplace_back(collect, p);
        for (auto &t : th) t.join();
    }
    size_t max_distinct = 0, post_base[N_PAT + 1] = {0};
    for (int p = 0; p < N_PAT; ++p) {
        max_distinct = std::max(max_distinct, distinct[p]);
        post_base[p + 1] = post_base[p] + ent[p].size() + long_lists[p];
    }
    if (post_base[N_PAT] >= (1u << 25)) return fail(ctx, MCX_EINVAL, "seed index too large for 25-bit posting offsets");
    // one table size for all patterns (load factor <= 0.5 for the fullest), slots of (key, value)
    uint32_t size = 1024; int bits = 10;
    while ((double)size < (double)max_distinct * (MCX_SLOT_ROOM_X10 / 10.0)) { size <<= 1; ++bits; }
    std::vector<uint2> tab((size_t)N_PAT << bits);
    std::vector<uint32_t> post_all(post_base[N_PAT]);
    auto fill = [&](int p) {
        uint2 *ht = tab.data() + ((size_t)p << bits);
        for (size_t k = 0; k < size; ++k) ht[k] = make_uint2(0xffffffffu, 0u);
        const std::vector<unsigned long long> &en = ent[p];
        size_t w = post_base[p];
        for (size_t k = 0; k < en.size();) {
            const uint32_t code = (uint32_t)(en[k] >> 32);
            size_t e = k;
            while (e + 1 < en.size() && (en[e + 1] >> 32) == code) ++e;
            const uint32_t cnt = (uint32_t)(e - k + 1);
            {   // the word as a nibble window (wildcard letter 0: no pattern looks at its own wildcard) -> its filter bits
                uint32_t d[10] = {0}, cc = code;
                for (int k = PAT_LEN[p] - 1; k >= 0; --k) if (k != PAT_WILD[p]) { d[k] = cc % 10u; cc /= 10u; }
                uint32_t lo = 0, hi = d[8] | (d[9] << 4), b1, b2;
                for (int k = 0; k < 8; ++k) lo |= d[k] << (4 * k);
                if (p <= 2) {
                    const uint32_t h = filt_hash_a(lo, hi);
                    uint32_t *blk = filt_a.data() + (size_t)4 * filt_block(h);
                    filt_bits(p, lo, hi, h, b1, b2);
                    if (p == 0) { __atomic_fetch_or(&blk[0], b1, __ATOMIC_RELAXED); __atomic_fetch_or(&blk[3], b2, __ATOMIC_RELAXED); }
                    else __atomic_fetch_or(&blk[p], b1 | b2, __ATOMIC_RELAXED);
                } else {
                    const uint32_t h = filt_hash_b(lo, hi);
                    filt_bits(p, lo, hi, h, b1, b2);
                    __atomic_fetch_or(&filt_b[(size_t)2 * filt_block(h) + (size_t)(p - 3)], b1 | b2, __ATOMIC_RELAXED);
                }
            }
            uint32_t slot = (code * 2654435761u) >> (32 - bits);
            while (ht[slot].x != 0xffffffffu) slot = (slot + 1) & (size - 1);
            ht[slot] = make_uint2(code, (uint32_t)w | ((cnt > 127 ? 127u : cnt - 1) << 25));
            if (cnt > 127) post_all[w++] = cnt;              // lists too long for the 7-bit field start with their length
            for (size_t q = k; q <= e; ++q) {
                // bits 26..29: the murphy10 letter of the subject that decides the first rejection test of a candidate --
                // the residue under the wildcard (one-substitution words), the residue left of the word (exact words;
                // 15 at the start of the subject) -- so that k_resolve applies the test without touching the residues
                const uint32_t sj = (uint32_t)(en[q] & 0x3ffffffu), subj = sj >> 11, jj = sj & 0x7ffu;
                const uint8_t *r = red.data() + db->off[subj];
                const uint32_t letter = p == 0 ? (jj > 0 ? r[jj - 1] : 15u) : r[jj + (uint32_t)PAT_WILD[p]];
                post_all[w++] = sj | (letter << 26) | (q == e ? 0x80000000u : 0u);
            }
            k = e + 1;
        }
        std::vector<unsigned long long>().swap(ent[p]);
    };
    {
        std::vector<std::thread> th;
        for (int p = 0; p < N_PAT; ++p) th.emplace_back(fill, p);
        for (auto &t : th) t.join();
    }
    {
        uint2 *dt = nullptr;
        CK(dev_alloc(&dt, tab.size())); ctx->db_allocs.push_back(dt);
        CK(cudaMemcpy(dt, tab.data(), tab.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        ctx->db.htab = dt; ctx->db.hbits = bits;
    }
    uint32_t *dp = nullptr;
    CK(dev_alloc(&dp, post_all.size())); ctx->db_allocs.push_back(dp);
    CK(cudaMemcpy(dp, post_all.data(), post_all.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    ctx->db.post = dp;
    uint32_t *dfa = nullptr, *dfb = nullptr;
    CK(dev_alloc(&dfa, filt_a.size())); ctx->db_allocs.push_back(dfa);
    CK(cudaMemcpy(dfa, filt_a.data(), filt_a.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CK(dev_alloc(&dfb, filt_b.size())); ctx->db_allocs.push_back(dfb);
    CK(cudaMemcpy(dfb, filt_b.data(), filt_b.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    ctx->db.filt_a = reinterpret_cast<const uint4 *>(dfa); ctx->db.filt_b = reinterpret_cast<const uint2 *>(dfb);
    return MCX_OK;
}

// every way of writing tot as at most 20 letter counts, largest first (the order seg.c sums them in): f(counts, n)
template <typename F>
static void for_each_partition(int tot, F f) {
    int part[20];
    auto rec = [&](auto &&self, int left, int maxpart, int np) -> void {
        if (left == 0) return f((const int *)part, np);
        if (np == 20) return;
        for (int k = std::min(left, maxpart); k >= 1; --k) { part[np] = k; self(self, left - k, k, np + 1); }
    };
    rec(rec, tot, tot, 0);
}

// the two SEG tables: the integer window test and getprob() of every window class
static int upload_seg_tables(mcx_ctx *ctx, const double *lnfac, const double *ln20, const double *ent) {
    // integer form of the SEG window test (see SegTab): thresholds taken from the reference's own double sums
    SegTab T;
    memset(&T, 0, sizeof T);
    long long gfix[13];
    gfix[0] = 0;
    for (int c = 1; c <= SEG_WINDOW; ++c) gfix[c] = llround((double)c * log2((double)c) * 16777216.0);
    for (int c = 0; c < SEG_WINDOW; ++c) T.dg[c] = (int)(gfix[c + 1] - gfix[c]);
    for (int tot = 0; tot <= SEG_WINDOW; ++tot) {
        long long min_yes[2] = {LLONG_MAX, LLONG_MAX}, max_no[2] = {LLONG_MIN, LLONG_MIN};
        for_each_partition(tot, [&](const int *part, int np) {
            double e = 0.0;
            long long G = 0;
            for (int k = 0; k < np; ++k) { e += ent[tot * 13 + part[k]]; G += gfix[part[k]]; }
            const double cut[2] = {SEG_LOCUT, SEG_HICUT};
            for (int q = 0; q < 2; ++q) {
                if (e <= cut[q]) min_yes[q] = std::min(min_yes[q], G);
                else max_no[q] = std::max(max_no[q], G);
            }
        });
        for (int q = 0; q < 2; ++q)
            if (max_no[q] >= min_yes[q]) return fail(ctx, MCX_EINVAL, "internal: integer SEG window test does not separate the entropy cut-offs");
        T.thr[tot].x = (int)std::min<long long>(min_yes[0], INT_MAX);
        T.thr[tot].y = (int)std::min<long long>(min_yes[1], INT_MAX);
    }
    CK(cudaMemcpyToSymbol(g_segtab, &T, sizeof T));
    // getprob() of every (window length <= 20, multiset of letter counts), see g_segprob
    uint32_t z[32] = {0};
    std::vector<SegProbSlot> tab;
    for (unsigned long long seed = 0x243F6A8885A308D3ull;; seed += 0x9E3779B97F4A7C15ull) {
        unsigned long long x = seed;
        z[0] = 0;
        for (int c = 1; c <= SEGP_MAXLEN; ++c) {         // splitmix64
            x += 0x9E3779B97F4A7C15ull;
            unsigned long long t = x;
            t = (t ^ (t >> 30)) * 0xBF58476D1CE4E5B9ull; t = (t ^ (t >> 27)) * 0x94D049BB133111EBull; t ^= t >> 31;
            z[c] = (uint32_t)t;
        }
        tab.assign(SEGP_SLOTS, SegProbSlot{~0ull, 0.0});
        bool unique = true;
        size_t classes = 0;
        for (int len = 1; len <= SEGP_MAXLEN && unique; ++len)
            for (int tot = 0; tot <= len && unique; ++tot)
                for_each_partition(tot, [&](const int *part, int np) {
                    if (!unique) return;
                    // seg.c getprob() on the counts, largest first (same operations as seg_getprob above)
                    double lnperm = lnfac[len], lnass = lnfac[20];
                    uint32_t sig = 0;
                    int nz = 0;
                    for (int k = 0; k < np;) {
                        int e = k;
                        while (e + 1 < np && part[e + 1] == part[k]) ++e;
                        const int c = part[k], n = e - k + 1;
                        if (c > 1) for (int r = 0; r < n; ++r) lnperm -= lnfac[c];
                        if (n > 1) lnass -= lnfac[n];
                        nz += n;
                        sig += (uint32_t)n * z[c];
                        k = e + 1;
                    }
                    if (nz > 0 && nz < 20) lnass -= lnfac[20 - nz];
                    const double prob = lnass + lnperm - ln20[len];
                    const unsigned long long key = ((unsigned long long)len << 32) | sig;
                    uint32_t sl = segp_slot(key);
                    while (tab[sl].key != ~0ull) {
                        if (tab[sl].key == key) { unique = false; return; }
                        sl = (sl + 1) & (SEGP_SLOTS - 1);
                    }
                    tab[sl] = SegProbSlot{key, prob};
                    ++classes;
                });
        if (unique && classes * 2 <= (size_t)SEGP_SLOTS) break;
        if (classes * 2 > (size_t)SEGP_SLOTS) return fail(ctx, MCX_EINVAL, "internal: SEG probability table too small");
    }
    CK(cudaMemcpyToSymbol(g_segz, z, sizeof z));
    CK(cudaMemcpyToSymbol(g_segprob, tab.data(), sizeof(SegProbSlot) * SEGP_SLOTS));
    return MCX_OK;
}

static int upload_tables(mcx_ctx *ctx) {
    double lnfac[256], ln20[256], ent[13 * 13];
    for (int i = 0; i < 256; ++i) { lnfac[i] = lgamma((double)i + 1.0); ln20[i] = (double)i * log(20.0); }
    lnfac[0] = 0.0; lnfac[1] = 0.0;
    for (int t = 0; t <= SEG_WINDOW; ++t)
        for (int c = 0; c <= SEG_WINDOW; ++c)
            ent[t * 13 + c] = (c == 0 || t == 0 || c > t) ? 0.0 : -((double)c / (double)t) * (log((double)c / (double)t) / log(2.0));
    int8_t bl[21 * 32];
    for (int a = 0; a < 21; ++a)
        for (int b = 0; b < 32; ++b) bl[a * 32 + b] = (a < 20 && b < 20) ? BLOSUM62[a][b] : (int8_t)-5;
    uint8_t codon[64];
    for (int i = 0; i < 64; ++i) {
        const char *p = strchr(AA_ORDER, CODON_AA[i]);
        codon[i] = (p && CODON_AA[i] != '.') ? (uint8_t)(p - AA_ORDER) : (uint8_t)AA_STOP;
    }
    TRY(upload_seg_tables(ctx, lnfac, ln20, ent));
    {
        uint8_t lut[256];
        memset(lut, AA_STOP, sizeof lut);
        for (int rev = 0; rev < 2; ++rev)
            for (int c0 = 0; c0 < 5; ++c0)
                for (int c1 = 0; c1 < 5; ++c1)
                    for (int c2 = 0; c2 < 5; ++c2) {
                        if (c0 == 4 || c1 == 4 || c2 == 4) continue;
                        const int f = rev ? 2 : 0;       // complement: T<->A, C<->G = code ^ 2
                        lut[125 * rev + 25 * c0 + 5 * c1 + c2] = codon[16 * (c0 ^ f) + 4 * (c1 ^ f) + (c2 ^ f)];
                    }
        CK(cudaMemcpyToSymbol(g_codon_lut, lut, sizeof lut));
    }
    {   // fingerprint contributions of four unmasked bases at a time (k_fingerprint)
        static FpTab T;
        for (int ix = 0; ix < 256; ++ix) {
            unsigned long long f1 = 0, f2 = 0, r1 = 0, r2 = 0, p1 = 1, p2 = 1;
            for (int k = 0; k < 4; ++k) {
                const unsigned long long c = fp_of_code((((ix >> 4) >> k) & 1) << 1 | ((ix >> k) & 1), 0, 0);
                f1 = f1 * FP_B1 + c; f2 = f2 * FP_B2 + c;
                r1 += fp_comp(c) * p1; r2 += fp_comp(c) * p2; p1 *= FP_B1; p2 *= FP_B2;
            }
            T.f1[ix] = f1; T.f2[ix] = f2; T.r1[ix] = r1; T.r2[ix] = r2;
        }
        CK(cudaMemcpyToSymbol(g_fptab, &T, sizeof T));
    }
    CK(cudaMemcpyToSymbol(g_blosum, bl, sizeof bl));
    {
        uint32_t same[32] = {0};
        for (int a = 0; a < 20; ++a) for (int b = 0; b < 20; ++b) same[a] |= (uint32_t)(MURPHY10[a] == MURPHY10[b]) << b;
        CK(cudaMemcpyToSymbol(g_same, same, sizeof same));
    }
    CK(cudaMemcpyToSymbol(g_lnfac, lnfac, sizeof lnfac));
    CK(cudaMemcpyToSymbol(g_ln20, ln20, sizeof ln20));
    return MCX_OK;
}

extern "C" int mcx_create(mcx_ctx **out, const mcx_db *db, int device) {
    if (!out || !db || !db->off || !db->res || !db->fam || db->n_subj <= 0 || db->n_subj >= 32768)
        return fail(nullptr, MCX_EINVAL, "mcx_create: bad database descriptor");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, MCX_ECUDA, std::string("mcx_create: no CUDA device (") + cudaGetErrorString(e) +
                                            "); libmcx has no CPU path");
    if (device < 0 || device >= ndev) return fail(nullptr, MCX_EINVAL, "mcx_create: device index out of range");
    mcx_ctx *ctx = new mcx_ctx();
    ctx->device = device;
    auto body = [&]() -> int {
        CK(cudaSetDevice(device));
        CK(cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, device));
        CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        for (auto &ev : ctx->ev) CK(cudaEventCreate(&ev));
        for (auto &ev : ctx->ev_copy) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        CK(cudaHostAlloc((void **)&ctx->h_cnt, (C_N + 2 * NQ) * sizeof(unsigned long long), cudaHostAllocDefault));
        const int ns = db->n_subj;
        const int64_t nres = db->off[ns];
        int32_t *doff = nullptr; uint8_t *dres = nullptr, *dfam = nullptr;
        CK(dev_alloc(&doff, (size_t)ns + 1)); ctx->db_allocs.push_back(doff);
        CK(dev_alloc(&dres, (size_t)nres + 64)); ctx->db_allocs.push_back(dres);
        CK(cudaMemset(dres, AA_STOP, (size_t)nres + 64));
        dres += 32;                                   // residues are also fetched as aligned words around a position (load_residues)
        CK(dev_alloc(&dfam, (size_t)ns)); ctx->db_allocs.push_back(dfam);
        CK(cudaMemcpy(doff, db->off, ((size_t)ns + 1) * sizeof(int32_t), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dres, db->res, (size_t)nres, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(dfam, db->fam, (size_t)ns, cudaMemcpyHostToDevice));
        ctx->db.n_subj = ns; ctx->db.off = doff; ctx->db.res = dres; ctx->db.fam = dfam;
        TRY(upload_tables(ctx));
        TRY(build_index(ctx, db));
        TRY(ctx->d_cnt.ensure(ctx, C_N));
        TRY(ctx->d_qcnt.ensure(ctx, 2 * NQ));
        TRY(ctx->d_acc.ensure(ctx, 3 + 2 * MCX_N_FAM));
        TRY(ctx->d_abl.ensure(ctx, (int64_t)MCX_N_FAM * MCX_LEN_BINS));
        return MCX_OK;
    };
    const int rc = body();
    if (rc != MCX_OK) { g_err = ctx->err; mcx_destroy(ctx); return rc; }
    *out = ctx;
    return MCX_OK;
}

extern "C" void mcx_destroy(mcx_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (void *p : ctx->db_allocs) cudaFree(p);
    if (ctx->h_cnt) cudaFreeHost(ctx->h_cnt);
    for (auto &ev : ctx->ev) if (ev) cudaEventDestroy(ev);
    for (auto &ev : ctx->ev_copy) if (ev) cudaEventDestroy(ev);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream && ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;                                   // the DevBuf members free their storage
}

extern "C" int mcx_set_stream(mcx_ctx *ctx, void *cuda_stream) {
    if (!ctx) return fail(ctx, MCX_EINVAL, "mcx_set_stream: null context");
    CK(cudaSetDevice(ctx->device));
    if (ctx->stream && ctx->own_stream) { CK(cudaStreamSynchronize(ctx->stream)); CK(cudaStreamDestroy(ctx->stream)); }
    ctx->stream = (cudaStream_t)cuda_stream;
    ctx->own_stream = false;
    return MCX_OK;
}

extern "C" int mcx_set_params(mcx_ctx *ctx, const mcx_params *p) {
    if (!ctx || !p) return fail(ctx, MCX_EINVAL, "mcx_set_params: null argument");
    if (p->read_length < 27 || p->read_length > 3 * MAX_FRAME)
        return fail(ctx, MCX_EINVAL, "mcx_set_params: read_length must be within 27..504");
    for (int f = 0; f < MCX_N_FAM; ++f)
        if (p->cut[f].stat < 0 || p->cut[f].stat > 2) return fail(ctx, MCX_EINVAL, "mcx_set_params: bad aln_stat");
    CK(cudaSetDevice(ctx->device));
    ctx->par = *p;
    ctx->have_par = true;
    ctx->n_store = 0;            // a new run: the duplicate filter starts empty
    CK(cudaMemcpyToSymbol(c_cut, p->cut, sizeof(mcx_cutoff) * MCX_N_FAM));
    return MCX_OK;
}

// ------------------------------------------------------------------------------------------------
// pushes: the four entry points end in the same read store (ReadStore); nothing here waits for the GPU
// ------------------------------------------------------------------------------------------------
static ReadStore read_store(const mcx_ctx *ctx) {
    ReadStore S;
    S.pk = ctx->d_pk; S.woff = ctx->d_woff; S.len = ctx->d_len;
    S.quals = (ctx->have_quals && ctx->par.has_quality) ? ctx->d_quals.p : nullptr;
    S.qoff = ctx->d_qoff; S.qbytes = ctx->n_bases;
    return S;
}

// offsets of the records and of the qualities from the lengths (two scans over n + 1 items: slot n receives the total)
static int scan_offsets(mcx_ctx *ctx, bool with_quals) {
    const int64_t n = ctx->n_reads;
    cudaStream_t st = ctx->stream;
    TRY(ctx->d_woff.ensure(ctx, n + 1));
    if (with_quals) TRY(ctx->d_qoff.ensure(ctx, n + 1));
    auto gw = thrust::make_transform_iterator(static_cast<const uint32_t *>(ctx->d_len.p), GroupsOf());
    auto gl = thrust::make_transform_iterator(static_cast<const uint32_t *>(ctx->d_len.p), LenOf());
    TRY(cub_run(ctx, "cub::DeviceScan::ExclusiveSum (record offsets)", [&](void *t, size_t &tb) {
        return cub::DeviceScan::ExclusiveSum(t, tb, gw, ctx->d_woff.p, (int)(n + 1), st); }));
    ctx->launches += 2;
    if (with_quals) {
        TRY(cub_run(ctx, "cub::DeviceScan::ExclusiveSum (quality offsets)", [&](void *t, size_t &tb) {
            return cub::DeviceScan::ExclusiveSum(t, tb, gl, ctx->d_qoff.p, (int)(n + 1), st); }));
        ctx->launches += 2;
    }
    return MCX_OK;
}

// n_words < 0: not known on the host (ASCII reads are packed on the device; nothing waits on copy steps then)
static int begin_push(mcx_ctx *ctx, const char *who, int64_t n, int64_t n_words, int64_t n_bases, const void *quals) {
    if (!ctx->have_par) return fail(ctx, MCX_ESTATE, std::string(who) + ": call mcx_set_params first");
    if (n >= (1ll << 27)) return fail(ctx, MCX_EINVAL, std::string(who) + ": at most 2^27 reads per call");
    if (ctx->par.has_quality && !quals && n > 0) return fail(ctx, MCX_EINVAL, std::string(who) + ": FASTQ parameters but no qualities");
    CK(cudaSetDevice(ctx->device));
    ctx->launches = 0; ctx->host_syncs = 0;
    memset(ctx->ms, 0, sizeof ctx->ms);
    (void)cudaGetLastError();                  // nothing an earlier call left behind may stop CUB's dispatches
    ctx->n_steps = 0; ctx->steps_waited = 0; ctx->h2d_timed = false;
    ctx->qc_upto = 0; ctx->dedup_done = false; ctx->fp_done = false; ctx->counts_valid = false;
    ctx->pushed = false; ctx->searched = false;
    ctx->n_reads = n; ctx->n_words = n_words; ctx->n_bases = n_bases; ctx->have_quals = quals != nullptr;
    return MCX_OK;
}

static int end_push(mcx_ctx *ctx) {
    const int64_t n = ctx->n_reads;
    TRY(ctx->d_code.ensure(ctx, n + 1));
    CK(cudaMemsetAsync(ctx->d_code, 4, (size_t)(n + 1), ctx->stream));       // 4 = not examined
    ctx->pushed = true;
    return MCX_OK;
}

// how many copy steps a push of this size is cut into (~32 MB each)
static int copy_steps(int64_t bytes) {
    int64_t k = (bytes + (32ll << 20) - 1) / (32ll << 20);
    if (const char *e = getenv("MCX_COPY_STEPS")) k = atoi(e);
    return (int)std::max<int64_t>(1, std::min<int64_t>(k, MAX_COPY_STEPS));
}

extern "C" int mcx_push_reads_packed(mcx_ctx *ctx, const uint32_t *packed, int64_t n_words, const uint32_t *lengths,
                                     const uint8_t *quals, int64_t n_bases, int64_t n) {
    if (!ctx || n < 0 || n_words < 0 || n_bases < 0 || (n > 0 && (!packed || !lengths)))
        return fail(ctx, MCX_EINVAL, "mcx_push_reads_packed: bad argument");
    TRY(begin_push(ctx, "mcx_push_reads_packed", n, n_words, n_bases, quals));
    TRY(ctx->d_pk.ensure(ctx, n_words + 4));
    TRY(ctx->d_len.ensure(ctx, n + 1));
    if (quals) TRY(ctx->d_quals.ensure(ctx, n_bases + 32));
    cudaStream_t cs = ctx->copy_stream;
    // the copies run on their own stream in steps, an event behind each; the search waits per chunk of reads for
    // the steps that hold it, so the copy of later reads overlaps the kernels of earlier ones
    CK(cudaEventRecord(ctx->ev[EV_H2D0], cs));
    if (n > 0) CK(cudaMemcpyAsync(ctx->d_len, lengths, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice, cs));
    CK(cudaMemsetAsync(ctx->d_len + n, 0, sizeof(uint32_t), cs));
    CK(cudaEventRecord(ctx->ev[EV_LENS], cs));
    const int K = copy_steps(n_words * 4 + (quals ? n_bases : 0));
    ctx->step_words = (n_words + K - 1) / K;
    ctx->step_qbytes = (((n_bases + K - 1) / K) + 15) & ~15ll;
    for (int k = 0; k < K; ++k) {
        const int64_t w0 = std::min(n_words, k * ctx->step_words), w1 = std::min(n_words, (k + 1) * ctx->step_words);
        if (w1 > w0) CK(cudaMemcpyAsync(ctx->d_pk + w0, packed + w0, (size_t)(w1 - w0) * 4, cudaMemcpyHostToDevice, cs));
        if (quals) {
            const int64_t q0 = std::min(n_bases, k * ctx->step_qbytes), q1 = std::min(n_bases, (k + 1) * ctx->step_qbytes);
            if (q1 > q0) CK(cudaMemcpyAsync(ctx->d_quals + q0, quals + q0, (size_t)(q1 - q0), cudaMemcpyHostToDevice, cs));
        }
        CK(cudaEventRecord(ctx->ev_copy[k], cs));
    }
    CK(cudaEventRecord(ctx->ev[EV_H2D1], cs));
    ctx->n_steps = K; ctx->h2d_timed = true;
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev[EV_LENS], 0));
    TRY(scan_offsets(ctx, quals != nullptr));
    return end_push(ctx);
}

extern "C" int mcx_push_reads_packed_dev(mcx_ctx *ctx, const uint32_t *d_packed, int64_t n_words, const uint32_t *d_lengths,
                                         const uint8_t *d_quals, int64_t n_bases, int64_t n) {
    if (!ctx || n < 0 || n_words < 0 || n_bases < 0 || (n > 0 && (!d_packed || !d_lengths)))
        return fail(ctx, MCX_EINVAL, "mcx_push_reads_packed_dev: bad argument");
    if (d_quals && ((uintptr_t)d_quals & 15)) return fail(ctx, MCX_EINVAL, "mcx_push_reads_packed_dev: qualities must be 16-byte aligned");
    TRY(begin_push(ctx, "mcx_push_reads_packed_dev", n, n_words, n_bases, d_quals));
    TRY(ctx->d_pk.borrow(ctx, const_cast<uint32_t *>(d_packed)));
    TRY(ctx->d_quals.borrow(ctx, const_cast<uint8_t *>(d_quals)));
    // the lengths are copied (n + 1 entries are scanned; the caller's array has n)
    TRY(ctx->d_len.ensure(ctx, n + 1));
    if (n > 0) CK(cudaMemcpyAsync(ctx->d_len, d_lengths, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx->stream));
    CK(cudaMemsetAsync(ctx->d_len + n, 0, sizeof(uint32_t), ctx->stream));
    TRY(scan_offsets(ctx, d_quals != nullptr));
    return end_push(ctx);
}

// ASCII reads (device-resident by now): lengths, offsets, bit-planes; the qualities take the offsets of the bases
static int pack_ascii(mcx_ctx *ctx, const uint8_t *d_bases, const int64_t *d_offsets, int64_t n, int64_t total) {
    cudaStream_t st = ctx->stream;
    TRY(ctx->d_len.ensure(ctx, n + 1));
    k_lens_from_offsets<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(d_offsets, n, ctx->d_len);
    TRY(scan_offsets(ctx, false));
    // every read of l bases takes 3 ceil(l / 32) words: at most 3 (total / 32 + n)
    const int64_t bound = 3 * (total / 32 + n) + 4;
    TRY(ctx->d_pk.ensure(ctx, bound));
    if (n > 0) k_pack_ascii<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(d_bases, d_offsets, n, ctx->d_woff, ctx->d_pk);
    ctx->launches += 2;
    if (ctx->have_quals) {
        TRY(ctx->d_qoff.ensure(ctx, n + 1));
        CK(cudaMemcpyAsync(ctx->d_qoff, d_offsets, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    }
    return MCX_OK;
}

extern "C" int mcx_push_reads(mcx_ctx *ctx, const uint8_t *bases, const uint8_t *quals, const int64_t *offsets,
                              int64_t n) {
    if (!ctx || !offsets || n < 0 || (n > 0 && !bases)) return fail(ctx, MCX_EINVAL, "mcx_push_reads: bad argument");
    const int64_t total = n > 0 ? offsets[n] : 0;
    TRY(begin_push(ctx, "mcx_push_reads", n, -1, total, quals));
    TRY(ctx->d_ascii.ensure(ctx, total + 16));
    TRY(ctx->d_aoffs.ensure(ctx, n + 1));
    if (quals) TRY(ctx->d_quals.ensure(ctx, total + 32));
    cudaStream_t st = ctx->stream;
    CK(cudaEventRecord(ctx->ev[EV_H2D0], st));
    if (total > 0) CK(cudaMemcpyAsync(ctx->d_ascii, bases, (size_t)total, cudaMemcpyHostToDevice, st));
    if (quals && total > 0) CK(cudaMemcpyAsync(ctx->d_quals, quals, (size_t)total, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_aoffs, offsets, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(ctx->ev[EV_H2D1], st));
    ctx->h2d_timed = true;
    TRY(pack_ascii(ctx, ctx->d_ascii, ctx->d_aoffs, n, total));
    return end_push(ctx);
}

extern "C" int mcx_push_reads_dev(mcx_ctx *ctx, const uint8_t *d_bases, const uint8_t *d_quals,
                                  const int64_t *d_offsets, int64_t n, int64_t total_bytes) {
    if (!ctx || !d_offsets || n < 0 || (n > 0 && !d_bases)) return fail(ctx, MCX_EINVAL, "mcx_push_reads_dev: bad argument");
    if (d_quals && ((uintptr_t)d_quals & 15)) return fail(ctx, MCX_EINVAL, "mcx_push_reads_dev: qualities must be 16-byte aligned");
    TRY(begin_push(ctx, "mcx_push_reads_dev", n, -1, total_bytes, d_quals));
    TRY(ctx->d_quals.borrow(ctx, const_cast<uint8_t *>(d_quals)));
    TRY(pack_ascii(ctx, d_bases, d_offsets, n, total_bytes));
    return end_push(ctx);
}

extern "C" int mcx_host_alloc(void **out, size_t bytes) {
    if (!out) return fail(nullptr, MCX_EINVAL, "mcx_host_alloc: null argument");
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) return fail(nullptr, MCX_ECUDA, std::string("mcx_host_alloc: ") + cudaGetErrorString(e));
    return MCX_OK;
}
extern "C" void mcx_host_free(void *p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------------
// QC
// ------------------------------------------------------------------------------------------------
// copy steps that hold packed words [0, words) and quality bytes [0, qbytes) (words < 0: all of them)
static int steps_holding(const mcx_ctx *ctx, int64_t words, int64_t qbytes) {
    if (words < 0) return ctx->n_steps;
    int need = 0;
    if (words > 0 && ctx->step_words > 0) need = (int)std::min<int64_t>(ctx->n_steps, (words + ctx->step_words - 1) / ctx->step_words);
    if (ctx->have_quals && qbytes > 0 && ctx->step_qbytes > 0)
        need = std::max(need, (int)std::min<int64_t>(ctx->n_steps, (qbytes + 15 + ctx->step_qbytes - 1) / ctx->step_qbytes));
    return need;
}
// make the compute stream wait for the copy steps that hold packed words [0, words) and quality bytes [0, qbytes)
static int wait_copies(mcx_ctx *ctx, int64_t words, int64_t qbytes) {
    if (ctx->steps_waited >= ctx->n_steps) return MCX_OK;
    const int need = steps_holding(ctx, words, qbytes);
    for (int k = ctx->steps_waited; k < need; ++k) CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy[k], 0));
    ctx->steps_waited = std::max(ctx->steps_waited, need);
    return MCX_OK;
}

static int pushed_on_device(mcx_ctx *ctx, const char *who) {
    if (!ctx->pushed) return fail(ctx, MCX_ESTATE, std::string(who) + ": no reads pushed");
    CK(cudaSetDevice(ctx->device));
    return MCX_OK;
}
// have the copy steps that hold packed words [0, words) and quality bytes [0, qbytes) finished? (does not wait)
static bool copies_arrived(mcx_ctx *ctx, int64_t words, int64_t qbytes) {
    const int need = steps_holding(ctx, words, qbytes);
    if (need <= ctx->steps_waited) return true;
    const cudaError_t q = cudaEventQuery(ctx->ev_copy[need - 1]);   // the steps complete in order
    if (q != cudaSuccess) (void)cudaGetLastError();                  // cudaErrorNotReady is not an error
    return q == cudaSuccess;
}

static void collect_kqc_time(mcx_ctx *ctx);
static int sync_stream(mcx_ctx *ctx) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    ++ctx->host_syncs;
    collect_kqc_time(ctx);
    return MCX_OK;
}

// verdicts of reads [qc_upto, upto) (the copies holding them must have been waited for)
static int qc_range(mcx_ctx *ctx, int64_t upto) {
    if (upto <= ctx->qc_upto) return MCX_OK;
    const mcx_params &P = ctx->par;
    const int64_t r0 = ctx->qc_upto, nr = upto - r0;
    CK(cudaEventRecord(ctx->ev[EV_KQC0], ctx->stream));
    k_qc<<<(unsigned)((nr * 8 + 255) / 256), 256, 0, ctx->stream>>>(read_store(ctx), r0, upto, P.read_length, P.quality_offset,
                                                                  P.min_quality, P.mean_quality, P.max_unknown, ctx->d_code);
    CK(cudaEventRecord(ctx->ev[EV_KQC1], ctx->stream));
    ctx->kqc_pending = true;
    ++ctx->launches;
    ctx->qc_upto = upto;
    return MCX_OK;
}

// after a synchronisation: add the time of the last k_qc launch to ms[MS_KQC]
static void collect_kqc_time(mcx_ctx *ctx) {
    if (!ctx->kqc_pending) return;
    ctx->ms[MS_KQC] += elapsed_ms(ctx->ev[EV_KQC0], ctx->ev[EV_KQC1]);
    ctx->kqc_pending = false;
}

// fingerprints of all pushed reads in d_fp (computed once per push)
static int ensure_fingerprints(mcx_ctx *ctx) {
    const int64_t n = ctx->n_reads;
    TRY(ctx->d_fp.ensure(ctx, std::max<int64_t>(n, 1)));
    if (n > 0 && !ctx->fp_done) {
        k_fingerprint<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(read_store(ctx), n, ctx->d_fp);
        ++ctx->launches; ctx->fp_done = true;
    }
    return MCX_OK;
}

// everything decided over all pushed reads: verdicts and, with -d, the duplicates
static int qc_all(mcx_ctx *ctx) {
    const int64_t n = ctx->n_reads;
    cudaStream_t st = ctx->stream;
    TRY(wait_copies(ctx, -1, -1));
    CK(cudaEventRecord(ctx->ev[EV_QC0], st));
    TRY(qc_range(ctx, n));
    if (ctx->par.filter_dups && !ctx->dedup_done && n > 0) {
        TRY(sync_stream(ctx));                             // (k_qc's events are read before they are reused)
        CK(cudaEventRecord(ctx->ev[EV_DEDUP0], st));
        const int64_t nt = n + ctx->n_store;               // reads of this push + fingerprints kept by earlier pushes
        if (nt >= (1ll << 31)) return fail(ctx, MCX_EINVAL, "mcx: more than 2^31 fingerprints in the duplicate filter");
        TRY(ctx->d_fpa.ensure(ctx, nt));
        TRY(ctx->d_fpa2.ensure(ctx, nt));
        TRY(ctx->d_fpi.ensure(ctx, nt));
        TRY(ctx->d_fpi2.ensure(ctx, nt));
        TRY(ensure_fingerprints(ctx));
        if (nt > 1) {
            // one radix sort on the upper 48 bits of the fingerprint brings equal fingerprints together; which read of a
            // group stays is decided by index inside k_mark_dups, so neither a stable sort nor a second key is needed
            const FpStore S{ctx->d_store_a, ctx->d_store_b};
            k_fp_keys<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(ctx->d_fp, n, S, ctx->n_store, ctx->d_fpa, ctx->d_fpi);
            TRY(cub_run(ctx, "cub::DeviceRadixSort::SortPairs (fingerprints)", [&](void *t, size_t &tb) {
                return cub::DeviceRadixSort::SortPairs(t, tb, ctx->d_fpa.p, ctx->d_fpa2.p, ctx->d_fpi.p, ctx->d_fpi2.p, (int)nt, 64 - FP_SORT_BITS, 64, st); }));
            k_mark_dups<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(ctx->d_fpa2, ctx->d_fpi2, ctx->d_fp, S, nt, ctx->d_code);
            ctx->launches += 9;
        }
        CK(cudaEventRecord(ctx->ev[EV_DEDUP1], st));
        TRY(sync_stream(ctx));
        ctx->ms[MS_DEDUP] += elapsed_ms(ctx->ev[EV_DEDUP0], ctx->ev[EV_DEDUP1]);
        ctx->dedup_done = true;
    }
    CK(cudaEventRecord(ctx->ev[EV_QC1], st));
    return MCX_OK;
}

static int qc_counts_all(mcx_ctx *ctx) {
    if (ctx->counts_valid) return MCX_OK;
    TRY(qc_all(ctx));
    const int64_t n = ctx->n_reads;
    cudaStream_t st = ctx->stream;
    CK(cudaMemsetAsync(ctx->d_cnt + C_QCALL, 0, 4 * sizeof(unsigned long long), st));
    if (n > 0) { k_count_codes<<<592, 256, 0, st>>>(ctx->d_code, n, ctx->d_cnt + C_QCALL); ++ctx->launches; }
    CK(cudaMemcpyAsync(ctx->h_cnt + C_QCALL, ctx->d_cnt + C_QCALL, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    TRY(sync_stream(ctx));
    const unsigned long long *c = ctx->h_cnt + C_QCALL;
    ctx->qc.n_reads = n; ctx->qc.kept = (int64_t)c[0]; ctx->qc.too_short = (int64_t)c[1];
    ctx->qc.low_qual = (int64_t)c[2]; ctx->qc.dups = (int64_t)c[3];
    ctx->counts_valid = true;
    return MCX_OK;
}

extern "C" int mcx_qc_export(mcx_ctx *ctx, uint8_t *code, uint64_t *fingerprints) {
    if (!ctx || !code) return fail(ctx, MCX_EINVAL, "mcx_qc_export: null argument");
    TRY(pushed_on_device(ctx, "mcx_qc_export"));
    const int64_t n = ctx->n_reads;
    cudaStream_t st = ctx->stream;
    if (n == 0) return MCX_OK;
    TRY(qc_all(ctx));
    CK(cudaMemcpyAsync(code, ctx->d_code, (size_t)n, cudaMemcpyDeviceToHost, st));
    if (fingerprints) {
        TRY(ensure_fingerprints(ctx));
        std::vector<FpKey> h((size_t)n);
        CK(cudaMemcpyAsync(h.data(), ctx->d_fp, (size_t)n * sizeof(FpKey), cudaMemcpyDeviceToHost, st));
        TRY(sync_stream(ctx));
        for (int64_t i = 0; i < n; ++i) { fingerprints[2 * i] = h[(size_t)i].a; fingerprints[2 * i + 1] = h[(size_t)i].b; }
    }
    return sync_stream(ctx);
}

extern "C" int mcx_qc_import(mcx_ctx *ctx, const uint8_t *code) {
    if (!ctx || !code) return fail(ctx, MCX_EINVAL, "mcx_qc_import: null argument");
    TRY(pushed_on_device(ctx, "mcx_qc_import"));
    TRY(qc_all(ctx));
    if (ctx->n_reads > 0)
        CK(cudaMemcpyAsync(ctx->d_code, code, (size_t)ctx->n_reads, cudaMemcpyHostToDevice, ctx->stream));
    ctx->counts_valid = false; ctx->searched = false;
    return qc_counts_all(ctx);
}

// Device-side access to the verdicts for the cross-GPU duplicate exchange (microbecensus_b200/distributed.py): the
// per-read codes and the fingerprint records (a, b, read index) stay in HBM, the caller's framework wraps the pointers,
// rewrites codes in place and calls mcx_qc_refresh.
extern "C" int mcx_qc_device(mcx_ctx *ctx, void **d_code, void **d_fingerprints, int64_t *n) {
    if (!ctx || !d_code || !n) return fail(ctx, MCX_EINVAL, "mcx_qc_device: null argument");
    TRY(pushed_on_device(ctx, "mcx_qc_device"));
    TRY(qc_all(ctx));
    *n = ctx->n_reads;
    *d_code = ctx->d_code;
    if (d_fingerprints) {
        TRY(ensure_fingerprints(ctx));
        *d_fingerprints = ctx->d_fp;
    }
    return sync_stream(ctx);
}

extern "C" int mcx_qc_refresh(mcx_ctx *ctx) {
    if (!ctx) return fail(ctx, MCX_EINVAL, "mcx_qc_refresh: null context");
    TRY(pushed_on_device(ctx, "mcx_qc_refresh"));
    ctx->counts_valid = false; ctx->searched = false;
    return qc_counts_all(ctx);
}

extern "C" int mcx_qc_counts(mcx_ctx *ctx, mcx_qc *out) {
    if (!ctx || !out) return fail(ctx, MCX_EINVAL, "mcx_qc_counts: null argument");
    TRY(pushed_on_device(ctx, "mcx_qc_counts"));
    TRY(qc_counts_all(ctx));
    *out = ctx->qc;
    return MCX_OK;
}

// ------------------------------------------------------------------------------------------------
// -d across GPUs (SURVEY 8e: the path's one real exchange step).  Every long-enough read sends (fingerprint a, b,
// global index << 1 | passed QC) to the rank that owns its fingerprint; the owner sorts what it received and marks every
// record behind the first QC-passing read of its fingerprint; the marks travel back.  The library does the three
// compute steps on the context's stream -- mcx_dedup_begin (partition by owner), mcx_dedup_owner (sort + mark),
// mcx_dedup_finish (apply) -- and the caller moves the two buffers between ranks (NCCL all-to-all through
// torch.distributed, microbecensus_b200/distributed.py).  (Round 1 did these steps with eager torch ops: three argsorts,
// bincount, scatter_reduce -- 17 ms of a 200 ms step, untimed.)
// ------------------------------------------------------------------------------------------------
struct XRec { unsigned long long a, b; long long gp; };
// room for `need` stored fingerprints, keeping the ones there are
static int reserve_store(mcx_ctx *ctx, int64_t need) {
    if (need <= ctx->d_store_a.cap) return MCX_OK;
    const int64_t cap = need + need / 2 + 1024;
    TRY(ctx->d_store_a.grow_keep(ctx, ctx->n_store, cap));
    TRY(ctx->d_store_b.grow_keep(ctx, ctx->n_store, cap));
    return MCX_OK;
}
extern "C" int mcx_dedup_reset(mcx_ctx *ctx) {
    if (!ctx) return fail(ctx, MCX_EINVAL, "mcx_dedup_reset: null context");
    ctx->n_store = 0;
    return MCX_OK;
}     // gp = global read index << 1 | passed QC
__device__ __forceinline__ int owner_of(unsigned long long a, int world) { return (int)((a & 0x7fffffffffffffffull) % (unsigned long long)world); }

__global__ void k_x_count(const FpKey *__restrict__ fp, const uint8_t *__restrict__ code, int64_t n, int world, unsigned long long *cnt) {
    __shared__ unsigned int s[64];
    if (threadIdx.x < 64) s[threadIdx.x] = 0;
    __syncthreads();
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
        if (code[r] != 1) atomicAdd(&s[owner_of(fp[r].a, world)], 1u);
    __syncthreads();
    if (threadIdx.x < world && s[threadIdx.x]) atomicAdd(&cnt[threadIdx.x], (unsigned long long)s[threadIdx.x]);
}
// cursor[o] starts at the first slot of owner o in the send buffer
__global__ void k_x_scatter(const FpKey *__restrict__ fp, const uint8_t *__restrict__ code, int64_t n, int world, long long first_index,
                            unsigned long long *cursor, XRec *__restrict__ send, uint32_t *__restrict__ send_read) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n || code[r] == 1) return;
    const FpKey k = fp[r];
    const unsigned long long at = atomicAdd(&cursor[owner_of(k.a, world)], 1ull);
    XRec x; x.a = k.a; x.b = k.b; x.gp = ((first_index + r) << 1) | (long long)(code[r] == 0);
    send[at] = x;
    send_read[at] = (uint32_t)r;
}
__global__ void k_x_keys(const XRec *__restrict__ recv, int64_t m, unsigned long long *__restrict__ kg, unsigned long long *__restrict__ ka, uint32_t *__restrict__ vi) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < m) { kg[p] = (unsigned long long)recv[p].gp; ka[p] = recv[p].a; vi[p] = (uint32_t)p; }
}
// one thread per run of equal sort key in the list sorted by the upper bits of `a`: marks[record] = 1 for every record
// of a fingerprint group behind (by global index) the group's first QC-passing read -- or for every record of the group
// if its fingerprint is already in the owner's store (kept in an earlier round of a streamed run); the fingerprint of a
// group that gets its keeper now joins the store
__device__ __forceinline__ void x_of_entry(uint32_t v, const XRec *__restrict__ recv, const FpStore &S, unsigned long long &a, unsigned long long &b) {
    if (v & FP_STORED) { a = S.a[v & ~FP_STORED]; b = S.b[v & ~FP_STORED]; }
    else { a = recv[v].a; b = recv[v].b; }
}
__global__ void k_x_keys_store(FpStore S, int64_t m, int64_t n_store, unsigned long long *__restrict__ ka, uint32_t *__restrict__ vi) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_store) { ka[m + p] = S.a[p]; vi[m + p] = FP_STORED | (uint32_t)p; }
}
__global__ void k_x_mark(const unsigned long long *__restrict__ ka, const uint32_t *__restrict__ vi, const XRec *__restrict__ recv, FpStore S,
                         int64_t m, uint8_t *__restrict__ marks, unsigned long long *__restrict__ new_a, unsigned long long *__restrict__ new_b,
                         unsigned long long *n_store) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    const unsigned long long key = ka[p] >> (64 - FP_SORT_BITS);
    if (p > 0 && (ka[p - 1] >> (64 - FP_SORT_BITS)) == key) return;
    int64_t e = p + 1;
    while (e < m && (ka[e] >> (64 - FP_SORT_BITS)) == key) ++e;
    for (int64_t s = p; s < e; ++s) {
        unsigned long long sa, sb, qa, qb;
        x_of_entry(vi[s], recv, S, sa, sb);
        bool first = true;
        for (int64_t q = p; q < s; ++q) { x_of_entry(vi[q], recv, S, qa, qb); if (qa == sa && qb == sb) { first = false; break; } }
        if (!first) continue;
        bool stored = false;
        long long keeper = LLONG_MAX;
        for (int64_t q = s; q < e; ++q) {
            const uint32_t v = vi[q];
            if (q > s) { x_of_entry(v, recv, S, qa, qb); if (qa != sa || qb != sb) continue; }
            if (v & FP_STORED) stored = true;
            else { const long long gp = recv[v].gp; if ((gp & 1) && (gp >> 1) < keeper) keeper = gp >> 1; }
        }
        if (!stored && keeper == LLONG_MAX) continue;
        if (!stored) { const unsigned long long o = atomicAdd(n_store, 1ull); new_a[o] = sa; new_b[o] = sb; }
        for (int64_t q = s; q < e; ++q) {
            const uint32_t v = vi[q];
            if (v & FP_STORED) continue;
            if (q > s) { x_of_entry(v, recv, S, qa, qb); if (qa != sa || qb != sb) continue; }
            if (stored || (recv[v].gp >> 1) > keeper) marks[v] = 1;
        }
    }
}
__global__ void k_x_apply(const uint8_t *__restrict__ marks, const uint32_t *__restrict__ send_read, int64_t ns, uint8_t *__restrict__ code) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < ns && marks[p]) code[send_read[p]] = 3;
}

extern "C" int mcx_dedup_begin(mcx_ctx *ctx, int world, int64_t first_index, void **d_send, int64_t *send_counts) {
    if (!ctx || !d_send || !send_counts || world < 1 || world > 64) return fail(ctx, MCX_EINVAL, "mcx_dedup_begin: bad argument (1 <= world <= 64)");
    TRY(pushed_on_device(ctx, "mcx_dedup_begin"));
    cudaStream_t st = ctx->stream;
    const int64_t n = ctx->n_reads;
    TRY(qc_all(ctx));
    TRY(sync_stream(ctx));
    CK(cudaEventRecord(ctx->ev[EV_DEDUP0], st));
    TRY(ensure_fingerprints(ctx));
    TRY(ctx->d_xsend.ensure(ctx, std::max<int64_t>(n, 1) * 3));
    TRY(ctx->d_fpi.ensure(ctx, std::max<int64_t>(n, 1)));
    unsigned long long *cnt = ctx->d_cnt + C_XCNT, *cur = ctx->d_cnt + C_XCNT + 64 + 0;   // counts, then cursors (exclusive prefix)
    CK(cudaMemsetAsync(cnt, 0, 128 * sizeof(unsigned long long), st));
    if (n > 0) k_x_count<<<592, 256, 0, st>>>(ctx->d_fp, ctx->d_code, n, world, cnt);
    CK(cudaMemcpyAsync(ctx->h_cnt, cnt, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    TRY(sync_stream(ctx));
    unsigned long long pre[64], acc = 0;
    for (int o = 0; o < 64; ++o) { pre[o] = acc; if (o < world) { send_counts[o] = (int64_t)ctx->h_cnt[o]; acc += ctx->h_cnt[o]; } }
    ctx->x_nsend = (int64_t)acc;
    CK(cudaMemcpyAsync(cur, pre, 64 * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
    if (n > 0) k_x_scatter<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ctx->d_fp, ctx->d_code, n, world, (long long)first_index, cur,
                                                                       reinterpret_cast<XRec *>(ctx->d_xsend.p), ctx->d_fpi);
    ctx->launches += 2;
    CK(cudaEventRecord(ctx->ev[EV_DEDUP1], st));
    TRY(sync_stream(ctx));
    ctx->ms[MS_DEDUP] += elapsed_ms(ctx->ev[EV_DEDUP0], ctx->ev[EV_DEDUP1]);
    *d_send = ctx->d_xsend;
    return MCX_OK;
}

extern "C" int mcx_dedup_owner(mcx_ctx *ctx, const void *d_recv, int64_t m, void **d_marks) {
    if (!ctx || !d_marks || m < 0 || (m > 0 && !d_recv)) return fail(ctx, MCX_EINVAL, "mcx_dedup_owner: bad argument");
    if (m >= (1ll << 31)) return fail(ctx, MCX_EINVAL, "mcx_dedup_owner: at most 2^31 records per rank");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int64_t mm = std::max<int64_t>(m, 1);
    const int64_t mt = m + ctx->n_store;                 // the records of this round + the fingerprints this rank has kept before
    if (mt >= (1ll << 31)) return fail(ctx, MCX_EINVAL, "mcx_dedup_owner: more than 2^31 fingerprints on one rank");
    TRY(ctx->d_xmarks.ensure(ctx, mm));
    TRY(ctx->d_fpa.ensure(ctx, m > 0 ? mt : 1));
    TRY(ctx->d_fpa2.ensure(ctx, m > 0 ? mt : 1));
    TRY(ctx->d_xkg.ensure(ctx, mm));
    TRY(ctx->d_xvi.ensure(ctx, m > 0 ? mt : 1));
    TRY(ctx->d_fpi2.ensure(ctx, m > 0 ? mt : 1));
    CK(cudaEventRecord(ctx->ev[EV_DEDUP0], st));
    CK(cudaMemsetAsync(ctx->d_xmarks, 0, (size_t)mm, st));
    if (m > 0) {
        TRY(reserve_store(ctx, ctx->n_store + m));
        const XRec *recv = reinterpret_cast<const XRec *>(d_recv);
        const FpStore S{ctx->d_store_a, ctx->d_store_b};
        k_x_keys<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(recv, m, ctx->d_xkg, ctx->d_fpa, ctx->d_xvi);
        if (ctx->n_store > 0) k_x_keys_store<<<(unsigned)((ctx->n_store + 255) / 256), 256, 0, st>>>(S, m, ctx->n_store, ctx->d_fpa, ctx->d_xvi);
        TRY(cub_run(ctx, "cub::DeviceRadixSort::SortPairs (owned fingerprints)", [&](void *t, size_t &tb) {
            return cub::DeviceRadixSort::SortPairs(t, tb, ctx->d_fpa.p, ctx->d_fpa2.p, ctx->d_xvi.p, ctx->d_fpi2.p, (int)mt, 64 - FP_SORT_BITS, 64, st); }));
        ctx->h_cnt[C_NSTORE] = (unsigned long long)ctx->n_store;
        CK(cudaMemcpyAsync(ctx->d_cnt + C_NSTORE, ctx->h_cnt + C_NSTORE, sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
        k_x_mark<<<(unsigned)((mt + 255) / 256), 256, 0, st>>>(ctx->d_fpa2, ctx->d_fpi2, recv, S, mt, ctx->d_xmarks, ctx->d_store_a, ctx->d_store_b, ctx->d_cnt + C_NSTORE);
        CK(cudaMemcpyAsync(ctx->h_cnt + C_NSTORE, ctx->d_cnt + C_NSTORE, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        ctx->launches += 10;
    }
    CK(cudaEventRecord(ctx->ev[EV_DEDUP1], st));
    TRY(sync_stream(ctx));
    if (m > 0) ctx->n_store = (int64_t)ctx->h_cnt[C_NSTORE];
    ctx->ms[MS_DEDUP] += elapsed_ms(ctx->ev[EV_DEDUP0], ctx->ev[EV_DEDUP1]);
    *d_marks = ctx->d_xmarks;
    return MCX_OK;
}

extern "C" int mcx_dedup_finish(mcx_ctx *ctx, const void *d_marks_back) {
    if (!ctx || (ctx->x_nsend > 0 && !d_marks_back)) return fail(ctx, MCX_EINVAL, "mcx_dedup_finish: bad argument");
    TRY(pushed_on_device(ctx, "mcx_dedup_finish"));
    if (ctx->x_nsend > 0) {
        k_x_apply<<<(unsigned)((ctx->x_nsend + 255) / 256), 256, 0, ctx->stream>>>(reinterpret_cast<const uint8_t *>(d_marks_back), ctx->d_fpi, ctx->x_nsend, ctx->d_code);
        ++ctx->launches;
    }
    ctx->dedup_done = true;
    ctx->counts_valid = false; ctx->searched = false;
    return qc_counts_all(ctx);
}

struct IsKept {
    const uint8_t *code;
    __device__ __forceinline__ bool operator()(const int32_t &i) const { return code[i] == 0; }
};

struct SearchPlan {
    int64_t quota, chunk;                      // quota < 0: all kept reads; chunk: reads the frame store and queues are sized for
    int maxm, fstride, nwr, thr;               // frame length, frame row stride, words of a 12-window mask, report floor
    uint8_t *frames;
    bool streaming;                            // rounds of pieces sized by what the host -> device copies have delivered
    std::vector<int64_t> bounds;               // piece c holds reads [bounds[c], bounds[c + 1])
    std::vector<long long> bw, bq;             // packed words / quality bytes before bounds[c] (-1: not read back)
    int pieces() const { return (int)bounds.size() - 1; }
};
// sums over the chunks of a search
struct SearchTally {
    int64_t sampled = 0, examined = 0;
    unsigned long long segq = 0, pass = 0, cand = 0, seeds = 0, surv = 0;   // surv: ungapped HSPs of all chunks so far
    unsigned long long gain = 0, wide = 0;                                   // extensions handed to k_gap_dp / to k_gap_dir
    float ms_qc = 0, ms_frames = 0, ms_seg = 0, ms_probe = 0, ms_kprobe = 0, ms_ext = 0, ms_kseed = 0, ms_gap = 0;
};

// buffer sizes from the chunk size and the MCX_* knobs
static int plan_search(mcx_ctx *ctx, int64_t quota, SearchPlan &S) {
    const mcx_params &P = ctx->par;
    const int64_t n = ctx->n_reads;
    int64_t per_read = 8;
    if (const char *e = getenv("MCX_SURV_PER_READ")) per_read = std::max(1, atoi(e));
    const int64_t want = std::max<int64_t>((quota >= 0 ? std::min(quota, n) : n) * per_read, 1 << 16);
    if (ctx->d_surv.cap < want) TRY(grow_survivors(ctx, 0, want));
    TRY(ctx->d_best.ensure(ctx, n + 1));
    TRY(ctx->d_nrep.ensure(ctx, n + 1));
    TRY(ctx->d_bestkey.ensure(ctx, n + 1));
    S.quota = quota;
    S.maxm = (P.read_length + 2) / 3;
    // an ungapped HSP of 49+ can still grow in the gapped stage, so it survives whatever the floor is
    S.thr = std::max(1, std::min(P.min_report_raw, 49));
    // the stages run per chunk of pushed reads so that the frame store and the queues stay bounded
    S.fstride = frame_stride(S.maxm);
    S.nwr = std::max(1, (S.maxm - SEG_WINDOW + 1 + 31) / 32);
    int64_t chunk = 2000000, cand_per_read = std::max<int64_t>(96, (int64_t)(0.8 * P.read_length));   // ~0.69 L word-hit postings per read on the marker set
    chunk = std::min<int64_t>(chunk, std::max<int64_t>(250000, 300000000 / P.read_length));   // queues scale with bases, not reads
    if (const char *e = getenv("MCX_CHUNK_READS")) chunk = std::min(2700000, std::max(1, atoi(e)));   // frame rows < 2^24
    if (const char *e = getenv("MCX_CAND_PER_READ")) cand_per_read = std::max(1, atoi(e));
    int64_t pass_per_read = std::max<int64_t>(32, (int64_t)(0.4 * P.read_length));    // ~0.23 L words per read pass the filter
    if (const char *e = getenv("MCX_PASS_PER_READ")) pass_per_read = std::max(1, atoi(e));
    chunk = std::min<int64_t>(chunk, std::max<int64_t>(n, 1));
    S.chunk = chunk;
    bool grew = false;
    TRY(ctx->d_frames.ensure(ctx, (chunk * 6 + 512) * S.fstride + 128, &grew));
    // k_seed reads 16-byte windows around a word without looking at the row ends: whatever lies there must be a residue code
    if (grew) CK(cudaMemsetAsync(ctx->d_frames, AA_STOP, (size_t)ctx->d_frames.cap, ctx->stream));
    TRY(ctx->d_cand.ensure(ctx, std::max<int64_t>(chunk * cand_per_read, 1 << 16)));
    TRY(ctx->d_passq.ensure(ctx, std::max<int64_t>(chunk * pass_per_read, 1 << 16)));
    TRY(ctx->d_seedq.ensure(ctx, std::max<int64_t>(ctx->d_cand.cap / 2, 1 << 16)));
    TRY(ctx->d_segq.ensure(ctx, chunk * 6 + 512));
    TRY(ctx->d_segm.ensure(ctx, (chunk * 6 + 512) * 2 * S.nwr));
    TRY(ctx->d_kept.ensure(ctx, chunk + 1));
    S.frames = ctx->d_frames + 64;             // rows are also read as aligned words around a position (load_residues)
    return MCX_OK;
}

// While host -> device copies are in flight the reads are cut into pieces of a sixteenth of a chunk, and every round of
// the chunk loop searches the pieces that have ARRIVED by then (at least two, at most a chunk): with one GPU on the link
// that is a small first round and then full chunks; with eight GPUs sharing the host's memory system (copies 2.3x
// slower) the rounds stay as large as the link allows and the search never waits for more than it needs (fixed rounds of
// 1/8, 1/4, 1/2, 1 chunk left the search idle 11 ms of an 80 ms step at 8 GPUs).
static int chunk_bounds(mcx_ctx *ctx, SearchPlan &S) {
    const int64_t n = ctx->n_reads;
    S.streaming = ctx->steps_waited < ctx->n_steps && ctx->n_steps > 1 && !ctx->par.filter_dups;
    const int64_t c = S.streaming ? std::min<int64_t>(S.chunk, std::max<int64_t>(S.chunk / 16, 65536)) : S.chunk;   // never more than the buffers hold
    S.bounds.assign(1, 0);
    while (S.bounds.back() < n) S.bounds.push_back(std::min(n, S.bounds.back() + c));
    const int nb = S.pieces();
    S.bw.assign((size_t)nb + 1, -1); S.bq.assign((size_t)nb + 1, -1);
    if (ctx->steps_waited < ctx->n_steps && !ctx->par.filter_dups) {
        // where the pieces end in the packed words / quality bytes (the offsets were scanned on the device)
        for (int k = 1; k <= nb; ++k) {
            CK(cudaMemcpyAsync(&S.bw[(size_t)k], ctx->d_woff + S.bounds[(size_t)k], sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
            if (ctx->have_quals) CK(cudaMemcpyAsync(&S.bq[(size_t)k], ctx->d_qoff + S.bounds[(size_t)k], sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
        }
        TRY(sync_stream(ctx));
        if (nb > 0 && (S.bw[(size_t)nb] != ctx->n_words || (ctx->have_quals && S.bq[(size_t)nb] != ctx->n_bases)))
            return fail(ctx, MCX_EINVAL, "mcx_search: the pushed lengths do not add up to the pushed words / bases");
    }
    return MCX_OK;
}

// K1 on the reads of pieces [c, c1): verdicts, the list of kept reads, the -n cut and the verdict counts up to the read
// that fills it (mc.py:356 leaves the loop there); nr = kept reads searched, -1: all of them, counted on the device
static int qc_chunk(mcx_ctx *ctx, const SearchPlan &S, int c, int c1, SearchTally &T, int64_t &nr) {
    cudaStream_t st = ctx->stream;
    unsigned long long *hc = ctx->h_cnt;
    const int64_t r0 = S.bounds[(size_t)c], r1 = S.bounds[(size_t)c1];
    TRY(wait_copies(ctx, S.bw[(size_t)c1], S.bq[(size_t)c1]));
    CK(cudaEventRecord(ctx->ev[EV_QC0], st));
    TRY(qc_range(ctx, r1));
    thrust::counting_iterator<int32_t> it((int32_t)r0);
    TRY(cub_run(ctx, "cub::DeviceSelect::If (kept reads)", [&](void *t, size_t &tb) {
        return cub::DeviceSelect::If(t, tb, it, ctx->d_kept.p, ctx->d_cnt + C_NKEPT, (int)(r1 - r0), IsKept{ctx->d_code}, st); }));
    ctx->launches += 2;
    int64_t upto = r1;                         // verdicts counted up to here
    nr = -1;
    if (S.quota >= 0) {
        CK(cudaMemcpyAsync(hc + C_NKEPT, ctx->d_cnt + C_NKEPT, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        TRY(sync_stream(ctx));
        const int64_t kept_c = (int64_t)hc[C_NKEPT], remaining = S.quota - T.sampled;
        nr = std::min(kept_c, remaining);
        if (nr == remaining && nr > 0) {     // the quota is filled inside this chunk: by its nr-th kept read
            int32_t cut = 0;
            CK(cudaMemcpyAsync(&cut, ctx->d_kept + (nr - 1), sizeof cut, cudaMemcpyDeviceToHost, st));
            TRY(sync_stream(ctx));
            upto = (int64_t)cut + 1;
        }
        if (nr < kept_c) { hc[C_NKEPT + 1] = (unsigned long long)nr; CK(cudaMemcpyAsync(ctx->d_cnt + C_NKEPT, hc + C_NKEPT + 1, sizeof(unsigned long long), cudaMemcpyHostToDevice, st)); }
    }
    if (upto > r0) { k_count_codes<<<592, 256, 0, st>>>(ctx->d_code + r0, upto - r0, ctx->d_cnt + C_QC0); ++ctx->launches; }
    T.examined = upto;
    return MCX_OK;
}

// six frames of every searched read, then the full SEG of the frames k_frames queued (resident blocks, queue length read
// on the device); nr_max bounds the launches
static int frames_and_seg(mcx_ctx *ctx, const SearchPlan &S, int64_t nr_max) {
    cudaStream_t st = ctx->stream;
    const int L = ctx->par.read_length;
    CK(cudaMemsetAsync(ctx->d_cnt + C_SEGQ, 0, 2 * sizeof(unsigned long long), st));   // SEG queue length, k_seg's work counter
    CK(cudaEventRecord(ctx->ev[EV_FRAMES0], st));
    constexpr int NTF = MCX_FRAMES_NT;         // a multiple of 6: whole reads per block
    FrameArgs F;
    F.S = read_store(ctx); F.kept = ctx->d_kept; F.first = 0; F.n_search = ctx->d_cnt + C_NKEPT;
    F.L = L; F.frames = S.frames; F.segq = ctx->d_segq; F.n_segq = ctx->d_cnt + C_SEGQ;
    F.segm = ctx->d_segm; F.nwr = S.nwr;
    const size_t fsmem = sizeof(SegTab) + 256 + (size_t)S.fstride * NTF + (size_t)((NTF / 6 * L + 3) & ~3) + (size_t)2 * S.nwr * NTF * 4;
    CK(cudaFuncSetAttribute(k_frames<NTF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fsmem));
    k_frames<NTF><<<(unsigned)((nr_max * 6 + NTF - 1) / NTF), NTF, fsmem, st>>>(F, S.fstride);
    ++ctx->launches;
    CK(cudaEventRecord(ctx->ev[EV_SEG0], st));
    constexpr int SW = MCX_SEG_W;
    const size_t smem = 2 * SEG_TAB * sizeof(double) + sizeof(SegTab) + 128 + SEG_TRI + (size_t)SW * seg_warp_bytes(S.fstride, S.maxm);
    CK(cudaFuncSetAttribute(k_seg<SW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned resident = 0;
    TRY(resident_blocks(ctx, k_seg<SW>, SW * 32, smem, resident));
    k_seg<SW><<<(unsigned)std::min<unsigned long long>((nr_max * 6 + SW - 1) / SW, resident), SW * 32, smem, st>>>(
        S.frames, S.fstride, L, ctx->d_segq, ctx->d_segm, S.nwr, ctx->d_cnt + C_SEGQ, S.maxm, reinterpret_cast<unsigned int *>(ctx->d_cnt + C_WORK));
    ++ctx->launches;
    CK(cudaEventRecord(ctx->ev[EV_PROBE0], st));
    return MCX_OK;
}

// K2: probe -> resolve -> seed -> walk, queue lengths read on the device, one read-back behind them; a queue that
// overflowed is sized for what was seen and the chunk's seed stage runs again
static int seed_stage(mcx_ctx *ctx, const SearchPlan &S, int64_t nr_max, SearchTally &T) {
    cudaStream_t st = ctx->stream;
    unsigned long long *hc = ctx->h_cnt;
    const unsigned long long surv_before = T.surv;
    unsigned long long n_cand = 0, n_seeds = 0, n_pass = 0;
    constexpr int NTP = MCX_PROBE_NT, NTR = MCX_RESOLVE_NT;
    const size_t psmem = (size_t)S.fstride * NTP;
    unsigned res_probe = 0, res_resolve = 0, res_seed = 0, res_walk = 0;
    CK(cudaFuncSetAttribute(k_probe<NTP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem));
    TRY(resident_blocks(ctx, k_probe<NTP>, NTP, psmem, res_probe));
    TRY(resident_blocks(ctx, k_resolve<NTR>, NTR, 0, res_resolve));
    TRY(resident_blocks(ctx, k_seed<SEED_NT>, SEED_NT, 0, res_seed));
    TRY(resident_blocks(ctx, k_walk<WALK_NT>, WALK_NT, 0, res_walk));
    auto row_blocks = [](unsigned resident, int nt, unsigned long long cap) -> unsigned {   // resident blocks per sub-queue row
        const unsigned long long want = ((unsigned long long)resident * 2 + NQ - 1) / NQ;
        return (unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>(want, (cap + nt - 1) / nt));
    };
    for (int attempt = 0;; ++attempt) {
        CK(cudaMemsetAsync(ctx->d_qcnt, 0, 2 * NQ * sizeof(unsigned long long), st));
        CK(cudaMemsetAsync(ctx->d_cnt + C_SEEDQ, 0, sizeof(unsigned long long), st));
        ProbeArgs A;
        A.n_reads = ctx->d_cnt + C_NKEPT; A.L = ctx->par.read_length; A.db = ctx->db; A.frames = S.frames; A.cand = ctx->d_cand;
        A.n_cand = ctx->d_qcnt; A.cap_cand = (unsigned long long)(ctx->d_cand.cap / NQ);
        A.passq = ctx->d_passq; A.n_pass = ctx->d_qcnt + NQ; A.cap_pass = (unsigned long long)(ctx->d_passq.cap / NQ);
        k_probe<NTP><<<(unsigned)std::min<unsigned long long>((nr_max * 6 + NTP - 1) / NTP, res_probe), NTP, psmem, st>>>(A, S.fstride);
        if (attempt == 0) CK(cudaEventRecord(ctx->ev[EV_KPROBE1], st));
        k_resolve<NTR><<<dim3(row_blocks(res_resolve, NTR, A.cap_pass), NQ), NTR, 0, st>>>(A);
        ++ctx->launches;
        if (attempt == 0) CK(cudaEventRecord(ctx->ev[EV_SEED0], st));
        ExtArgs E;
        E.kept = ctx->d_kept; E.first = 0; E.L = ctx->par.read_length; E.fstride = S.fstride; E.thr_report = S.thr; E.db = ctx->db;
        E.frames = S.frames; E.cand = ctx->d_cand; E.qfill = ctx->d_qcnt;
        E.cap_cand = (unsigned long long)(ctx->d_cand.cap / NQ);
        E.surv = ctx->d_surv; E.cap_surv = (unsigned long long)ctx->d_surv.cap;
        E.n_surv = ctx->d_cnt + C_SURV; E.n_seedq = ctx->d_cnt + C_SEEDQ;
        E.seedq = ctx->d_seedq; E.cap_seedq = (unsigned long long)ctx->d_seedq.cap;
        {   // duplicate filter: at least two slots per survivor the list can take
            int bits = 16;
            while ((1ll << bits) < 2 * ctx->d_surv.cap) ++bits;
            TRY(ctx->d_seen.ensure(ctx, 1ll << bits));
            CK(cudaMemsetAsync(ctx->d_seen, 0xff, (size_t)(1ll << bits) * sizeof(unsigned long long), st));
            E.seen = ctx->d_seen; E.seen_mask = (1ull << bits) - 1; E.seen_shift = 64 - bits;
        }
        k_seed<SEED_NT><<<dim3(row_blocks(res_seed, SEED_NT, E.cap_cand), NQ), SEED_NT, 0, st>>>(E);
        if (attempt == 0) CK(cudaEventRecord(ctx->ev[EV_KSEED1], st));
        k_walk<WALK_NT><<<res_walk * 8, WALK_NT, 0, st>>>(E);
        ctx->launches += 3;
        CK(cudaEventRecord(ctx->ev[EV_GAP0], st));
        CK(cudaMemcpyAsync(hc + C_N, ctx->d_qcnt, 2 * NQ * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(hc, ctx->d_cnt, C_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        TRY(sync_stream(ctx));
        unsigned long long worst = 0, worst_pass = 0;
        n_cand = 0;
        for (int q = 0; q < NQ; ++q) { n_cand += hc[C_N + q]; worst = std::max(worst, hc[C_N + q]); worst_pass = std::max(worst_pass, hc[C_N + NQ + q]); n_pass += hc[C_N + NQ + q]; }
        n_seeds = hc[C_SEEDQ];
        const bool over_pass = (int64_t)worst_pass > ctx->d_passq.cap / NQ;
        const bool over_cand = (int64_t)worst > ctx->d_cand.cap / NQ, over_seed = (int64_t)n_seeds > ctx->d_seedq.cap,
                   over_surv = (int64_t)hc[C_SURV] > ctx->d_surv.cap;
        if (!over_pass && !over_cand && !over_seed && !over_surv) { T.surv = hc[C_SURV]; break; }
        if (attempt >= 4) return fail(ctx, MCX_ENOMEM, "mcx_search: a queue (filter passes / candidates / seeds / survivors) overflowed after regrowth");
        // the fills are exact (of what the earlier queues let through): size the queue that overflowed for what was seen
        n_pass = 0;
        if (over_pass) TRY(ctx->d_passq.ensure(ctx, (int64_t)(worst_pass + worst_pass / 16 + 1024) * NQ));
        if (over_cand) TRY(ctx->d_cand.ensure(ctx, (int64_t)(worst + worst / 16 + 1024) * NQ));
        if (over_cand || over_seed) TRY(ctx->d_seedq.ensure(ctx, std::max<int64_t>((int64_t)(n_seeds + n_seeds / 8), ctx->d_cand.cap / 2)));
        if (over_surv) TRY(grow_survivors(ctx, (int64_t)surv_before, (int64_t)hc[C_SURV] + (int64_t)hc[C_SURV] / 4));
        hc[C_SURV] = surv_before;
        CK(cudaMemcpyAsync(ctx->d_cnt + C_SURV, hc + C_SURV, sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
    }
    T.cand += n_cand; T.seeds += n_seeds; T.pass += n_pass; T.segq += hc[C_SEGQ];
    return MCX_OK;
}

// gapped extension of the survivors [first, first + count): work list (padded with all-ones keys up to its bound, so that
// it can be sorted without knowing its length on the host) -> sorted by remaining query length -> screening pass ->
// complete DP + traceback for the extensions that gain -> (rare: wide-window fallback, see k_gap_dp) -> finish
static int gapped_stage(mcx_ctx *ctx, const SearchPlan &S, int64_t first, int64_t count, SearchTally &T) {
    cudaStream_t st = ctx->stream;
    GapArgs G;
    G.L = ctx->par.read_length; G.fstride = S.fstride; G.db = ctx->db; G.frames = S.frames; G.surv = ctx->d_surv;
    G.first = first; G.n_surv = count;
    G.hsp = ctx->d_hsp; G.keys = ctx->d_keys; G.idx = ctx->d_idx; G.counters = ctx->d_cnt + C_GAPPED;
    TRY(ctx->d_gitems.ensure(ctx, 6 * G.n_surv));
    TRY(ctx->d_gext.ensure(ctx, 2 * G.n_surv));
    G.items = ctx->d_gitems; G.ext = ctx->d_gext; G.n_items = ctx->d_cnt + C_ITEMS; G.n_items_total = ctx->d_cnt + C_NGAPTOT;
    CK(cudaMemsetAsync(ctx->d_gext, 0, (size_t)(2 * G.n_surv) * sizeof(GExtRec), st));
    CK(cudaMemsetAsync(ctx->d_cnt + C_ITEMS, 0, sizeof(unsigned long long), st));
    unsigned long long *list1 = ctx->d_gitems + G.n_surv * 2, *gainers = ctx->d_gitems + G.n_surv * 4, *wide = ctx->d_gitems;
    CK(cudaMemsetAsync(G.items, 0xff, (size_t)(2 * G.n_surv) * sizeof(unsigned long long), st));
    k_gap_list<<<(unsigned)((G.n_surv + 255) / 256), 256, 0, st>>>(G);
    TRY(cub_run(ctx, "cub::DeviceRadixSort::SortKeys (gapped work list)", [&](void *t, size_t &tb) {
        return cub::DeviceRadixSort::SortKeys(t, tb, G.items, list1, (int)(2 * G.n_surv), 32, 40, st); }));
    CK(cudaMemsetAsync(ctx->d_cnt + C_ITEMS2, 0, sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(ctx->d_cnt + C_WORK1, 0, 2 * sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(ctx->d_cnt + C_NWIDE, 0, 3 * sizeof(unsigned long long), st));
    constexpr int SNT = MCX_SCR_NT, FNT = MCX_FULL_NT, GW = MAX_FRAME + GAP_SLACK + 2;
    unsigned res_screen = 0, res_dp = 0, res_dir = 0, res_dir2 = 0;
    TRY(resident_blocks(ctx, k_gap_screen<SNT>, SNT, 0, res_screen));
    TRY(resident_blocks(ctx, k_gap_dp<FNT>, FNT, 0, res_dp));
    TRY(resident_blocks(ctx, k_gap_dir<GAP_NT, GW, false>, GAP_NT, 0, res_dir));
    TRY(resident_blocks(ctx, k_gap_dir<GAP_NT, GW, true>, GAP_NT, 0, res_dir2));
    auto grid = [](unsigned want, unsigned resident) { return std::max(1u, std::min(want, resident)); };
    // where the stage hands an extension on (screen -> k_gap_dp after this many rows or columns, k_gap_dp -> k_gap_dir once
    // the live window spans this many columns): the sizes of the kernels' shared-memory rows by default; smaller values
    // route work down the later paths (for tests: the results must not change)
    int scr_rows = SCR_ROWS, scr_cols = SCR_COLS, dp_cols = RING - 8;
    if (const char *e = getenv("MCX_GAP_SCREEN_ROWS")) scr_rows = std::min(SCR_ROWS, std::max(1, atoi(e)));
    if (const char *e = getenv("MCX_GAP_SCREEN_COLS")) scr_cols = std::min(SCR_COLS, std::max(1, atoi(e)));
    if (const char *e = getenv("MCX_GAP_DP_COLS")) dp_cols = std::min(RING - 8, std::max(1, atoi(e)));
    k_gap_screen<SNT><<<grid(((unsigned)(2 * G.n_surv) + SNT - 1) / SNT, res_screen), SNT, 0, st>>>(G, list1, gainers, ctx->d_cnt + C_ITEMS2,
                                                                                                   scr_rows, scr_cols);
    CK(cudaMemcpyAsync(ctx->h_cnt + C_ITEMS2, ctx->d_cnt + C_ITEMS2, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    TRY(sync_stream(ctx));
    const int64_t n_gain = (int64_t)ctx->h_cnt[C_ITEMS2];
    T.gain += (unsigned long long)n_gain;
    // complete DP + traceback of the extensions that gain, in batches that bound the direction scratch
    const int rows_per_ext = S.maxm;
    const int64_t per_ext = (int64_t)rows_per_ext * DIR_ROW_WORDS;
    int64_t batch = std::max<int64_t>(1, (int64_t)(2ll << 30) / (per_ext * 4));       // 2 GB of directions at most
    if (const char *e = getenv("MCX_GAP_BATCH")) batch = std::max(1, atoi(e));
    batch = std::min(batch, std::max<int64_t>(n_gain, 1));
    if (n_gain > 0) TRY(ctx->d_dirs.ensure(ctx, batch * per_ext));
    for (int64_t g0 = 0; g0 < n_gain; g0 += batch) {
        const int64_t ng = std::min(batch, n_gain - g0);
        CK(cudaMemsetAsync(ctx->d_cnt + C_WORK1, 0, sizeof(unsigned long long), st));
        k_gap_dp<FNT><<<grid((unsigned)((ng + FNT - 1) / FNT), res_dp), FNT, 0, st>>>(
            G, gainers, g0, ng, ctx->d_dirs, rows_per_ext, wide, ctx->d_cnt + C_NWIDE, reinterpret_cast<unsigned int *>(ctx->d_cnt + C_WORK1), dp_cols);
        k_gap_trace<<<(unsigned)((ng + 127) / 128), 128, 0, st>>>(G, gainers, g0, ng, ctx->d_dirs, rows_per_ext);
        ctx->launches += 2;
    }
    // fallback for extensions whose window outgrew the ring: score pass + statistics pass with rows in local memory.  The
    // list of the statistics pass takes the place of the sorted work list (read by the screen only): `wide` can hold up to
    // all 2 n_surv extensions, so no part of [0, 2 n_surv) is free while the score pass reads it.
    unsigned long long *wide2 = list1;
    unsigned int *work2 = reinterpret_cast<unsigned int *>(ctx->d_cnt + C_WORK2), *work3 = reinterpret_cast<unsigned int *>(ctx->d_cnt + C_NWIDE + 2);
    k_gap_dir<GAP_NT, GW, false><<<grid(64, res_dir), GAP_NT, 0, st>>>(G, wide, ctx->d_cnt + C_NWIDE, wide2, ctx->d_cnt + C_NWIDE + 1, work2);
    k_gap_dir<GAP_NT, GW, true><<<grid(64, res_dir2), GAP_NT, 0, st>>>(G, wide2, ctx->d_cnt + C_NWIDE + 1, nullptr, nullptr, work3);
    CK(cudaMemcpyAsync(ctx->h_cnt + C_NWIDE, ctx->d_cnt + C_NWIDE, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));   // read after the chunk's sync
    ctx->launches += 8;
    k_gap_finish<<<(unsigned)((G.n_surv + 255) / 256), 256, 0, st>>>(G);
    ctx->launches += 3;
    return MCX_OK;
}

// streamed -d: the reads kept by this push are what later pushes of the run must not repeat (mc.py:355)
static int append_kept_fingerprints(mcx_ctx *ctx, int64_t examined) {
    TRY(reserve_store(ctx, ctx->n_store + examined));
    ctx->h_cnt[C_NSTORE] = (unsigned long long)ctx->n_store;
    CK(cudaMemcpyAsync(ctx->d_cnt + C_NSTORE, ctx->h_cnt + C_NSTORE, sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->stream));
    k_store_append<<<(unsigned)((examined + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_fp, ctx->d_code, examined, ctx->d_store_a, ctx->d_store_b, ctx->d_cnt + C_NSTORE);
    ++ctx->launches;
    return MCX_OK;
}

// sort the ungapped HSPs of all chunks, classify, read the sums back and fill mcx_result, the counters and the timings
static int classify_and_collect(mcx_ctx *ctx, const SearchTally &T, bool stored) {
    cudaStream_t st = ctx->stream;
    unsigned long long *hc = ctx->h_cnt;
    mcx_result &R = ctx->res;
    R.sampled_reads = T.sampled;
    R.n_seed_hits = (int64_t)T.surv;
    ctx->work[0] = (int64_t)T.segq; ctx->work[1] = (int64_t)T.pass; ctx->work[2] = (int64_t)T.cand;
    ctx->work[3] = (int64_t)T.seeds; ctx->work[4] = (int64_t)T.surv;
    ctx->work[5] = (int64_t)T.gain; ctx->work[6] = (int64_t)T.wide;
    const int64_t ns = (int64_t)T.surv;
    CK(cudaEventRecord(ctx->ev[EV_SORT0], st));
    if (ns > 0) {
        TRY(cub_run(ctx, "cub::DeviceMergeSort::SortPairs (HSPs)", [&](void *t, size_t &tb) {
            return cub::DeviceMergeSort::SortPairs(t, tb, ctx->d_keys.p, ctx->d_idx.p, ns, SortKeyLess(), st); }));
        ctx->launches += 3;
    }
    CK(cudaEventRecord(ctx->ev[EV_CLS0], st));
    if (ns > 0) {
        ClsArgs C;
        C.keys = ctx->d_keys; C.n = ns; C.L = ctx->par.read_length; C.min_report = ctx->par.min_report_raw;
        C.db = ctx->db; C.keep = ctx->d_keep; C.nrep = ctx->d_nrep; C.bestkey = ctx->d_bestkey;
        C.best_subject = ctx->d_best; C.acc = ctx->d_acc; C.aln_by_len = ctx->d_abl;
        C.caplist = ctx->d_hflag; C.n_cap = ctx->d_cnt + C_NCAP;
        const unsigned cb = (unsigned)((ns + 255) / 256);
        k_cls_groups<<<cb, 256, 0, st>>>(C);
        k_cls_cap<<<cb, 256, 0, st>>>(C);
        k_cls_cap_apply<4><<<148, 128, 0, st>>>(C);
        k_cls_filter<<<cb, 256, 0, st>>>(C);
        k_cls_sum<<<cb, 256, 0, st>>>(C);
        ctx->launches += 5;
    }
    CK(cudaEventRecord(ctx->ev[EV_D2H0], st));
    std::vector<unsigned long long> acc(3 + 2 * MCX_N_FAM), abl((size_t)MCX_N_FAM * MCX_LEN_BINS);
    CK(cudaMemcpyAsync(acc.data(), ctx->d_acc, acc.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(abl.data(), ctx->d_abl, abl.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hc, ctx->d_cnt, C_N * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(ctx->ev[EV_D2H1], st));
    TRY(sync_stream(ctx));
    R.too_short = (int64_t)hc[C_QC0 + 1]; R.low_qual = (int64_t)hc[C_QC0 + 2]; R.dups = (int64_t)hc[C_QC0 + 3];
    if (stored) ctx->n_store = (int64_t)hc[C_NSTORE];
    R.reads_with_hits = (int64_t)acc[0]; R.reads_classified = (int64_t)acc[1]; R.n_hsp = (int64_t)acc[2];
    R.n_gapped = (int64_t)hc[C_NGAPTOT]; R.gapped_cells = (int64_t)hc[C_CELLS];
    R.n_capped_reads = (int64_t)hc[C_NCAP];
    if (getenv("MCX_DEBUG")) fprintf(stderr, "[mcx] filter passes %llu, candidates %llu, accepted seeds %llu, ungapped HSPs %llu; gapped extensions %llu, with gain > 0: %llu, cells %llu; host syncs %lld\n",
                                     T.pass, T.cand, T.seeds, T.surv, hc[C_NGAPTOT], hc[C_GAPPED], hc[C_CELLS], (long long)ctx->host_syncs);
    for (int f = 0; f < MCX_N_FAM; ++f) { R.fam_hits[f] = (int64_t)acc[3 + f]; R.fam_aln[f] = (int64_t)acc[3 + MCX_N_FAM + f]; }
    for (size_t k = 0; k < abl.size(); ++k) R.aln_by_len[k] = (int64_t)abl[k];
    ctx->ms_detail[MSD_KPROBE] = T.ms_kprobe; ctx->ms_detail[MSD_KRESOLVE] = T.ms_probe - T.ms_kprobe;
    ctx->ms_detail[MSD_KSEED] = T.ms_kseed; ctx->ms_detail[MSD_KWALK] = T.ms_ext - T.ms_kseed;
    ctx->ms[MS_QC] = T.ms_qc; ctx->ms[MS_PROBE] = T.ms_probe; ctx->ms[MS_EXTEND] = T.ms_ext; ctx->ms[MS_GAPPED] = T.ms_gap;
    ctx->ms[MS_FRAMES] = T.ms_frames; ctx->ms[MS_SEG] = T.ms_seg;
    ctx->ms[MS_SORT] = elapsed_ms(ctx->ev[EV_SORT0], ctx->ev[EV_CLS0]);
    ctx->ms[MS_CLASSIFY] = elapsed_ms(ctx->ev[EV_CLS0], ctx->ev[EV_D2H0]);
    ctx->ms[MS_D2H] = elapsed_ms(ctx->ev[EV_D2H0], ctx->ev[EV_D2H1]);
    if (ctx->h2d_timed && cudaEventQuery(ctx->ev[EV_H2D1]) == cudaSuccess) ctx->ms[MS_H2D] = elapsed_ms(ctx->ev[EV_H2D0], ctx->ev[EV_H2D1]);
    (void)cudaGetLastError();
    return MCX_OK;
}

extern "C" int mcx_search(mcx_ctx *ctx, int64_t quota) {
    if (!ctx) return fail(ctx, MCX_EINVAL, "mcx_search: null context");
    TRY(pushed_on_device(ctx, "mcx_search"));
    cudaStream_t st = ctx->stream;
    const int64_t n = ctx->n_reads;
    memset(&ctx->res, 0, sizeof ctx->res);
    SearchPlan S;
    TRY(plan_search(ctx, quota, S));
    TRY(chunk_bounds(ctx, S));
    CK(cudaMemsetAsync(ctx->d_nrep, 0, (size_t)(n + 1) * sizeof(int32_t), st));
    CK(cudaMemsetAsync(ctx->d_bestkey, 0, (size_t)(n + 1) * sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(ctx->d_cnt, 0, 4 * sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(ctx->d_cnt + C_SURV, 0, (C_N - C_SURV) * sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(ctx->d_acc, 0, (3 + 2 * MCX_N_FAM) * sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(ctx->d_abl, 0, (size_t)MCX_N_FAM * MCX_LEN_BINS * sizeof(unsigned long long), st));
    if (n > 0) { k_fill_i32<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ctx->d_best, n, -1); ++ctx->launches; }
    SearchTally T;
    if (ctx->par.filter_dups || ctx->counts_valid) {     // -d is decided over all reads before anything is searched
        TRY(qc_all(ctx));
        TRY(sync_stream(ctx));
        T.ms_qc += elapsed_ms(ctx->ev[EV_QC0], ctx->ev[EV_QC1]);
    }
    for (int c = 0, c1 = 0; c < S.pieces() && (quota < 0 || T.sampled < quota); c = c1) {
        c1 = c + 1;
        if (S.streaming)                       // a second piece whatever has arrived (if a chunk holds two), then what has arrived
            while (c1 < S.pieces() && S.bounds[(size_t)c1 + 1] - S.bounds[(size_t)c] <= S.chunk &&
                   (c1 - c < 2 || copies_arrived(ctx, S.bw[(size_t)c1 + 1], S.bq[(size_t)c1 + 1]))) ++c1;
        int64_t nr = 0;
        TRY(qc_chunk(ctx, S, c, c1, T, nr));
        if (nr == 0) continue;
        const int64_t nr_max = nr < 0 ? S.bounds[(size_t)c1] - S.bounds[(size_t)c] : nr;   // launch bound; the kernels read the count on the device
        TRY(frames_and_seg(ctx, S, nr_max));
        const unsigned long long surv_before = T.surv;
        TRY(seed_stage(ctx, S, nr_max, T));
        T.sampled += nr < 0 ? (int64_t)ctx->h_cnt[C_NKEPT] : nr;
        const bool gapped = T.surv > surv_before;
        if (gapped) TRY(gapped_stage(ctx, S, (int64_t)surv_before, (int64_t)(T.surv - surv_before), T));
        CK(cudaEventRecord(ctx->ev[EV_GAP1], st));
        TRY(sync_stream(ctx));
        if (gapped) T.wide += ctx->h_cnt[C_NWIDE];
        T.ms_qc += elapsed_ms(ctx->ev[EV_QC0], ctx->ev[EV_FRAMES0]);
        T.ms_frames += elapsed_ms(ctx->ev[EV_FRAMES0], ctx->ev[EV_SEG0]);
        T.ms_seg += elapsed_ms(ctx->ev[EV_SEG0], ctx->ev[EV_PROBE0]);
        T.ms_probe += elapsed_ms(ctx->ev[EV_PROBE0], ctx->ev[EV_SEED0]);
        T.ms_kprobe += elapsed_ms(ctx->ev[EV_PROBE0], ctx->ev[EV_KPROBE1]);
        T.ms_kseed += elapsed_ms(ctx->ev[EV_SEED0], ctx->ev[EV_KSEED1]);
        T.ms_ext += elapsed_ms(ctx->ev[EV_SEED0], ctx->ev[EV_GAP0]);
        T.ms_gap += elapsed_ms(ctx->ev[EV_GAP0], ctx->ev[EV_GAP1]);
    }
    const bool stored = ctx->par.filter_dups && ctx->fp_done && T.examined > 0;
    if (stored) TRY(append_kept_fingerprints(ctx, T.examined));
    TRY(classify_and_collect(ctx, T, stored));
    ctx->searched = true;
    return MCX_OK;
}

extern "C" int mcx_result_get(mcx_ctx *ctx, mcx_result *out) {
    if (!ctx || !out) return fail(ctx, MCX_EINVAL, "mcx_result_get: null argument");
    if (!ctx->searched) return fail(ctx, MCX_ESTATE, "mcx_result_get: no search has run");
    *out = ctx->res;
    return MCX_OK;
}

extern "C" int mcx_get_hits(mcx_ctx *ctx, mcx_hit *out, int64_t cap, int64_t *n) {
    if (!ctx || !n) return fail(ctx, MCX_EINVAL, "mcx_get_hits: null argument");
    if (!ctx->searched) return fail(ctx, MCX_ESTATE, "mcx_get_hits: no search has run");
    CK(cudaSetDevice(ctx->device));
    *n = ctx->res.n_hsp;
    const int64_t ns = ctx->res.n_seed_hits;              // the HSPs sorted by the search
    if (!out || cap <= 0 || ns == 0) return MCX_OK;
    cudaStream_t st = ctx->stream;
    k_keep_sorted<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(ctx->d_keep, ns, ctx->d_hflag);
    CK(cudaMemsetAsync(ctx->d_hflag + ns, 0, sizeof(int32_t), st));
    TRY(cub_run(ctx, "cub::DeviceScan::ExclusiveSum (reported HSPs)", [&](void *t, size_t &tb) {
        return cub::DeviceScan::ExclusiveSum(t, tb, ctx->d_hflag.p, ctx->d_hpos.p, (int)(ns + 1), st); }));
    k_gather_hits<<<(unsigned)((ns + 255) / 256), 256, 0, st>>>(ctx->d_hsp, ctx->d_idx, ctx->d_keep, ctx->d_hpos, ns, ctx->d_hits_out);
    const int64_t take = std::min<int64_t>(cap, ctx->res.n_hsp);
    CK(cudaMemcpyAsync(out, ctx->d_hits_out, (size_t)take * sizeof(mcx_hit), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    return MCX_OK;
}

extern "C" int mcx_get_classified(mcx_ctx *ctx, int32_t *best_subject, int64_t n) {
    if (!ctx || !best_subject) return fail(ctx, MCX_EINVAL, "mcx_get_classified: null argument");
    if (!ctx->searched) return fail(ctx, MCX_ESTATE, "mcx_get_classified: no search has run");
    if (n > ctx->n_reads) n = ctx->n_reads;
    CK(cudaSetDevice(ctx->device));
    if (n > 0) CK(cudaMemcpyAsync(best_subject, ctx->d_best, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return MCX_OK;
}

// ------------------------------------------------------------------------------------------------
// DPX issue-rate microbenchmark (SURVEY 8d: the denominator the north star asks for next to the gapped stage's
// GCUPS).  Eight independent chains per thread of viaddmax / vimax3_relu, the two DPX forms an affine-gap cell uses.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dpx_bench(int iters, int seed, int *out) {
    int a[8], b = seed + threadIdx.x, c = seed * 3 + blockIdx.x;
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = seed + k * 17 + threadIdx.x;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            a[k] = __viaddmax_s32(a[k], b, c);            // max(a + b, c): the E / F update
            a[k] = __vimax3_s32_relu(a[k], c, b);         // max(a, c, b, 0): the H update
        }
        b ^= it; c += it;
    }
    int r = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) r ^= a[k];
    if (r == 0x7fffffff) out[0] = r;                      // keeps the chains alive
}

// best rate of reps 1..3 of a microbenchmark launch: `work` units over its device time, in 1e9 per second
template <typename F>
static int bench_rate(mcx_ctx *ctx, double work, F launch, double *rate) {
    cudaStream_t st = ctx->stream;
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        CK(cudaEventRecord(ctx->ev[EV_BENCH0], st));
        launch(rep);
        CK(cudaEventRecord(ctx->ev[EV_BENCH1], st));
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->ev[EV_BENCH0], ctx->ev[EV_BENCH1]));
        if (rep > 0) best = std::max(best, work / (ms * 1e-3) / 1e9);
    }
    *rate = best;
    return MCX_OK;
}

extern "C" int mcx_dpx_peak(mcx_ctx *ctx, double *gops_per_s) {
    if (!ctx || !gops_per_s) return fail(ctx, MCX_EINVAL, "mcx_dpx_peak: null argument");
    CK(cudaSetDevice(ctx->device));
    const int blocks = ctx->n_sm * 8, iters = 1 << 14;
    int *d_out = reinterpret_cast<int *>(ctx->d_cnt.p);   // never written in practice
    const double ops = (double)blocks * 256.0 * (double)iters * 16.0;    // DPX thread-instructions
    return bench_rate(ctx, ops, [&](int rep) { k_dpx_bench<<<blocks, 256, 0, ctx->stream>>>(iters, 12345 + rep, d_out); }, gops_per_s);
}

// ------------------------------------------------------------------------------------------------
// L2 random-access microbenchmark (SURVEY 8d: the seed-word lookup is bound by the random-access transaction rate, not
// by bandwidth).  Every thread issues independent 4-byte loads at pseudo-random words of the context's own 32 MB
// presence filter -- the access pattern of k_probe's filter probes, with nothing else in the way: one 32-byte sector per
// load, eight loads in flight per thread, full occupancy.  The result is the rate k_probe's probes/s are quoted against.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_l2_bench(const uint32_t *__restrict__ words, uint32_t mask, int iters, uint32_t seed, uint32_t *out) {
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + seed, acc = 0;
    for (int it = 0; it < iters; ++it) {
        uint32_t v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { x = x * 1664525u + 1013904223u; v[k] = __ldg(words + ((x >> 7) & mask)); }
#pragma unroll
        for (int k = 0; k < 8; ++k) acc ^= v[k];
    }
    if (acc == 0x9e3779b9u) out[0] = acc;                 // keeps the loads alive
}

extern "C" int mcx_l2_peak(mcx_ctx *ctx, double *gsectors_per_s) {
    if (!ctx || !gsectors_per_s) return fail(ctx, MCX_EINVAL, "mcx_l2_peak: null argument");
    CK(cudaSetDevice(ctx->device));
    const int blocks = ctx->n_sm * 8, iters = 512;
    uint32_t *d_out = reinterpret_cast<uint32_t *>(ctx->d_cnt + C_N - 1);
    const double loads = (double)blocks * 256.0 * (double)iters * 8.0;
    return bench_rate(ctx, loads, [&](int rep) {
        k_l2_bench<<<blocks, 256, 0, ctx->stream>>>(reinterpret_cast<const uint32_t *>(ctx->db.filt_a), (4u << FILT_BITS) - 1u, iters, 777u + rep, d_out);
    }, gsectors_per_s);
}

extern "C" int mcx_search_counters(mcx_ctx *ctx, int64_t out[8]) {
    if (!ctx || !out) return fail(ctx, MCX_EINVAL, "mcx_search_counters: null argument");
    memcpy(out, ctx->work, sizeof ctx->work);
    return MCX_OK;
}

extern "C" int mcx_timings_detail(mcx_ctx *ctx, float ms[4]) {
    if (!ctx || !ms) return fail(ctx, MCX_EINVAL, "mcx_timings_detail: null argument");
    memcpy(ms, ctx->ms_detail, sizeof ctx->ms_detail);
    return MCX_OK;
}

extern "C" int mcx_timings(mcx_ctx *ctx, float ms[12], int64_t *launches) {
    if (!ctx || !ms) return fail(ctx, MCX_EINVAL, "mcx_timings: null argument");
    memcpy(ms, ctx->ms, sizeof ctx->ms);
    if (launches) *launches = ctx->launches;
    return MCX_OK;
}
