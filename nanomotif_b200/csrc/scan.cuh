// Bit-parallel motif matcher shared by K2 (scan_count) and K3 (match_plane).
//
// Each lane owns one 512-bp chunk = NW (16) consecutive 32-bit words of the two sequence bit-planes
// x (high code bit) and y (low code bit), plus H halo words on both sides.  For a motif with
// constrained positions j_0 < ... < j_{K-1} the start-aligned match plane
//     S[p] = AND_i  ind_{j_i}( base[p + j_i] )
// is evaluated as ONE Horner chain from the last constrained position to the first, so that every
// constrained position costs one funnel shift of the running plane plus one lop3 per word:
//     C <- ind_{j_K-1};   C <- ind_{j_i} & (C >> (j_{i+1} - j_i))   for i = K-2 .. 0
// and the plane aligned at the modified base is M = C << mod_pos (one more funnel shift).  The chain
// runs over words [-H, NW + H): the right halo feeds the >> shifts, the left halo the final <<.
// Two register representations of the sequence:
//   XY   the raw planes; the indicator of ANY allowed-set is a two-variable boolean function of (x, y),
//        so it is folded into the lop3 immediate: C <- lop3<set>(x, y, shifted C).  Used by warps whose
//        chunks hold no non-ACGT letter.  Inter-contig padding is stored as code 0 and kept out by
//        CLIPPING the finished chains (LaneEdge below): padding runs are >= 64 > motif length, so an
//        occurrence overlaps padding iff its first or last position does, i.e. iff its start lies outside
//        [contig start, contig end - len].  That is ~3 integer ops per word and motif, only in warps that
//        touch a contig edge, instead of a second code path.
//   XYN  additionally the non-ACGT plane n, ANDed out of every indicator so that such letters fail every
//        constrained position and only match '.', the regex semantics of the reference (SURVEY.md
//        Appendix B item 5).  One extra logic op per word and step; used only by warps whose chunks (or
//        neighbouring chunks) hold a non-ACGT letter of a contig -- rare.  Padding fails every constrained
//        position here too, but a flanking '.' of an unstripped motif (K3, K5) is never tested, so callers
//        that may see one clip these chains as well (LaneEdge with edge set); K2's stripped motifs need not.
// The branch on the base is uniform across the CTA (it depends on the motif only).
#pragma once
#include "common.cuh"

namespace nmb {

constexpr int NW = kChunkWords;  // words per lane

template <int H, bool HASN>
struct LaneSeq;

// lop3 immediates over inputs (a, b, c) = (0xF0, 0xCC, 0xAA)
constexpr int kLutAndNot = 0x30;    // a & ~b

// ind_M(x, y) & s for an allowed-set M (bit0=A bit1=T bit2=G bit3=C) is ONE lop3 whose immediate is the
// set's truth table.  Every indicator is written so that it depends on the running (shifted) plane s:
// otherwise the compiler hoists the step-invariant part (e.g. ind(x, y) & ~n) out of the motif loop and
// keeps one extra register per word and plane alive.
template <int H>
struct LaneSeq<H, false> {
    static constexpr int XW = NW + 2 * H;  // words held per plane: [-H, NW + H)
    uint32_t x[XW], y[XW];
    template <int M>
    __device__ __forceinline__ uint32_t and_code(int i, uint32_t s) const {
        return lop3<(set_truth(M) & 0xAA)>(x[i], y[i], s);
    }
};

template <int H>
struct LaneSeq<H, true> {
    static constexpr int XW = NW + 2 * H;
    uint32_t x[XW], y[XW], n[XW];  // n = non-ACGT plane (inter-contig padding included)
    template <int M>
    __device__ __forceinline__ uint32_t and_code(int i, uint32_t s) const {
        return lop3<(set_truth(M) & 0xAA)>(x[i], y[i], lop3<kLutAndNot>(s, n[i], 0u));
    }
};

// Where the lane's chunk sits in its contig (meaningful in warps that touch inter-contig padding).
struct LaneEdge {
    int hi;      // contig end relative to the chunk's first position (clamped; >= 32 * (NW + 2) when far away)
    bool first;  // the chunk is the first of its contig: everything left of it is padding
    bool edge;   // warp-uniform: some lane of the warp touches padding, clip the chains
};

// bits k of a word starting at bit offset b (relative to the chunk) with b + k < hi / b + k >= lo
__device__ __forceinline__ uint32_t bits_below(int b, int hi) {
    return __funnelshift_rc(0xFFFFFFFFu, 0u, max(b + 32 - hi, 0));  // shift clamps at 32 -> 0
}
__device__ __forceinline__ uint32_t bits_from(int b, int lo) {
    return __funnelshift_lc(0u, 0xFFFFFFFFu, max(lo - b, 0));
}

// Start-aligned chain of a motif of `len` positions: keep starts p with contig_start <= p <= contig_end - len.
template <int H>
__device__ __forceinline__ void clip_start_aligned(uint32_t (&c)[NW + 2 * H], const LaneEdge &e, int len) {
    const int hi = e.hi - (len - 1);
#pragma unroll
    for (int i = 0; i < NW + 2 * H; ++i) {
        c[i] &= bits_below(32 * (i - H), hi);
        if (i < H && e.first) c[i] = 0u;
    }
}
// End-aligned chain (reverse-complement twin), stored reversed (dr[j] = D[CW-1-j]): keep ends q with
// contig_start + len - 1 <= q < contig_end.  Words left of the chunk are never read (aligned_word_rc).
template <int H>
__device__ __forceinline__ void clip_end_aligned_rev(uint32_t (&dr)[NW + 2 * H], const LaneEdge &e, int len) {
    constexpr int CW = NW + 2 * H;
#pragma unroll
    for (int i = H; i < CW; ++i) {
        uint32_t m = bits_below(32 * (i - H), e.hi);
        if (i < 2 * H && e.first) m &= bits_from(32 * (i - H), len - 1);  // len - 1 <= 32 * H - 1
        dr[CW - 1 - i] &= m;
    }
}

// Program (common.cuh): header n | mod_pos << 8 | len << 16, then n entries in processing order
// (last constrained position first).  entry = set code | (distance to the previous entry) << 8.
struct ProgramView {
    const uint16_t *ent;
    int n, mod_pos, len;
};

__device__ __forceinline__ ProgramView load_program(const Program *p) {
    const uint32_t hdr = __ldg(reinterpret_cast<const uint32_t *>(p));
    ProgramView v;
    v.n = hdr & 0xFF;
    v.mod_pos = (hdr >> 8) & 0xFF;
    v.len = (hdr >> 16) & 0xFF;
    v.ent = p->ent;
    return v;
}

template <int H>
__device__ __forceinline__ uint32_t shifted(const uint32_t (&c)[NW + 2 * H], int i, int s) {
    return __funnelshift_r(c[i], (i + 1 < NW + 2 * H) ? c[i + 1] : 0u, s);
}

template <int M, int H, bool HASN>
__device__ __forceinline__ void step_code(uint32_t (&c)[NW + 2 * H], const LaneSeq<H, HASN> &q, int s) {
#pragma unroll
    for (int i = 0; i < NW + 2 * H; ++i) c[i] = q.template and_code<M>(i, shifted<H>(c, i, s));
}

// Entry codes: 1..14 allowed-set (all fourteen have their own lop3 immediate, so degenerate positions
// cost the same as single bases), kEntShift32 = "shift the chain by one word" (emitted by the motif
// compiler for gaps >= 32), 0 = empty set (nothing matches), 15 = wildcard (pure shift; only produced
// for a leading wildcard of an unstripped motif).  All shifts are < 32 and the first entry's shift is 0.
constexpr int kEntShift32 = 0x10;

// Single-strand chain (K3 match planes): start-aligned match words of the lane's words [-H, NW + H);
// valid for words [-H, NW).
template <int H, bool HASN>
__device__ __forceinline__ void run_chain(const ProgramView &pv, const LaneSeq<H, HASN> &q,
                                          uint32_t (&c)[NW + 2 * H], const LaneEdge &edge) {
#pragma unroll
    for (int i = 0; i < NW + 2 * H; ++i) c[i] = 0xFFFFFFFFu;
    uint32_t e = __ldg(pv.ent);
#pragma unroll 1
    for (int i = 0; i < pv.n; ++i) {
        const uint32_t cur = e;
        if (i + 1 < pv.n) e = __ldg(pv.ent + i + 1);  // prefetch the next entry
        const int s = cur >> 8;
        switch (cur & 0xFF) {
#define NMB_CASE(m) case m: step_code<m, H, HASN>(c, q, s); break;
            NMB_CASE(1) NMB_CASE(2) NMB_CASE(3) NMB_CASE(4) NMB_CASE(5) NMB_CASE(6) NMB_CASE(7)
            NMB_CASE(8) NMB_CASE(9) NMB_CASE(10) NMB_CASE(11) NMB_CASE(12) NMB_CASE(13) NMB_CASE(14)
#undef NMB_CASE
            case 15:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) c[k] = shifted<H>(c, k, s);
                break;
            case kEntShift32:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) c[k] = (k + 1 < NW + 2 * H) ? c[k + 1] : 0u;
                break;
            default:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) c[k] = 0u;
                break;
        }
    }
    if (edge.edge) clip_start_aligned<H>(c, edge, pv.len);
}

// Allowed-set of the complementary bases: A<->T (bits 0,1), G<->C (bits 2,3).
__host__ __device__ constexpr int comp_set(int m) { return ((m & 5) << 1) | ((m & 10) >> 1); }

// The reverse-complement chain D is kept in REVERSED word order (dr[j] = D[CW-1-j]) so that its in-place
// update has the same shape as the forward chain's (new[j] from old[j] and old[j+1], ascending j); written
// the natural way the compiler rotates the whole array through registers with 18 moves per step.
template <int H>
__device__ __forceinline__ uint32_t shifted_l(const uint32_t (&dr)[NW + 2 * H], int j, int s) {
    return __funnelshift_l((j + 1 < NW + 2 * H) ? dr[j + 1] : 0u, dr[j], s);
}

// Both strands in one pass.  The reverse-complement motif has the complementary set at the mirrored
// position, so walking the SAME program (last constrained position first, same distances) with the
// complementary lop3 immediate and the OPPOSITE shift direction yields its END-aligned match plane:
//     C <- ind_S(x, y)       & (C >> d)     forward motif, start-aligned, valid on words [-H, NW)
//     D <- ind_comp(S)(x, y) & (D << d)     reverse complement, end-aligned, valid on words [0, NW + H)
// One dispatch per constrained position serves both chains (half the loop / branch overhead per chain
// step) and the two dependency chains interleave (twice the ILP).
template <int M, int H, bool HASN>
__device__ __forceinline__ void step_pair(uint32_t (&c)[NW + 2 * H], uint32_t (&dr)[NW + 2 * H],
                                          const LaneSeq<H, HASN> &q, int s) {
    constexpr int CW = NW + 2 * H;
#pragma unroll
    for (int i = 0; i < CW; ++i) c[i] = q.template and_code<M>(i, shifted<H>(c, i, s));
#pragma unroll
    for (int j = 0; j < CW; ++j) dr[j] = q.template and_code<comp_set(M)>(CW - 1 - j, shifted_l<H>(dr, j, s));
}

// First entry of a program: both chains start as the plain indicator planes (no shift, no AND).
template <int M, int H, bool HASN>
__device__ __forceinline__ void init_pair(uint32_t (&c)[NW + 2 * H], uint32_t (&dr)[NW + 2 * H],
                                          const LaneSeq<H, HASN> &q) {
    constexpr int CW = NW + 2 * H;
#pragma unroll
    for (int i = 0; i < CW; ++i) c[i] = q.template and_code<M>(i, 0xFFFFFFFFu);
#pragma unroll
    for (int j = 0; j < CW; ++j) dr[j] = q.template and_code<comp_set(M)>(CW - 1 - j, 0xFFFFFFFFu);
}

// True when any lane of the warp still has a candidate occurrence on either strand.
template <int H>
__device__ __forceinline__ bool chains_alive(const uint32_t (&c)[NW + 2 * H], const uint32_t (&d)[NW + 2 * H]) {
    uint32_t any = 0;
#pragma unroll
    for (int i = 0; i < NW + 2 * H; ++i) any |= c[i] | d[i];
    return __any_sync(0xFFFFFFFFu, any != 0);
}

// Returns false when both chains died in every lane of the warp (no occurrence in the warp's 16 384
// positions): after 8 constrained positions that is the common case, so the remaining steps and the
// whole popcount stage are skipped.  The test is warp-uniform.
template <int H, bool HASN>
__device__ __forceinline__ bool run_chain_pair(const ProgramView &pv, const LaneSeq<H, HASN> &q,
                                               uint32_t (&c)[NW + 2 * H], uint32_t (&d)[NW + 2 * H],
                                               const LaneEdge &edge) {
    uint32_t e = __ldg(pv.ent);
    {   // first entry (shift 0 by construction): the chains ARE the indicator planes
        const int code = e & 0xFF;
        if (pv.n > 1) e = __ldg(pv.ent + 1);
        switch (code) {
#define NMB_CASE(m) case m: init_pair<m, H, HASN>(c, d, q); break;
            NMB_CASE(1) NMB_CASE(2) NMB_CASE(3) NMB_CASE(4) NMB_CASE(5) NMB_CASE(6) NMB_CASE(7)
            NMB_CASE(8) NMB_CASE(9) NMB_CASE(10) NMB_CASE(11) NMB_CASE(12) NMB_CASE(13) NMB_CASE(14)
#undef NMB_CASE
            case 15:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) c[k] = d[k] = 0xFFFFFFFFu;
                break;
            default:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) c[k] = d[k] = 0u;
                break;
        }
    }
#pragma unroll 1
    for (int i = 1; i < pv.n; ++i) {
        const uint32_t cur = e;
        if (i + 1 < pv.n) e = __ldg(pv.ent + i + 1);  // prefetch the next entry
        const int s = cur >> 8;
        if (i >= 8 && !(i & 1) && !chains_alive<H>(c, d)) return false;
        switch (cur & 0xFF) {
#define NMB_CASE(m) case m: step_pair<m, H, HASN>(c, d, q, s); break;
            NMB_CASE(1) NMB_CASE(2) NMB_CASE(3) NMB_CASE(4) NMB_CASE(5) NMB_CASE(6) NMB_CASE(7)
            NMB_CASE(8) NMB_CASE(9) NMB_CASE(10) NMB_CASE(11) NMB_CASE(12) NMB_CASE(13) NMB_CASE(14)
#undef NMB_CASE
            case 15:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) c[k] = shifted<H>(c, k, s);
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) d[k] = shifted_l<H>(d, k, s);
                break;
            case kEntShift32:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) {
                    c[k] = (k + 1 < NW + 2 * H) ? c[k + 1] : 0u;
                    d[k] = (k + 1 < NW + 2 * H) ? d[k + 1] : 0u;
                }
                break;
            default:
#pragma unroll
                for (int k = 0; k < NW + 2 * H; ++k) {
                    c[k] = 0u;
                    d[k] = 0u;
                }
                break;
        }
    }
    if (pv.n >= 8 && !chains_alive<H>(c, d)) return false;
    if (edge.edge) {  // warp-uniform
        clip_start_aligned<H>(c, edge, pv.len);
        clip_end_aligned_rev<H>(d, edge, pv.len);
    }
    return true;
}

// Word k of the reverse-complement match plane aligned at ITS modified base: M_rc[p] = D[p + mod_pos]
// (mod_pos = the forward motif's; the rc motif's is len - 1 - mod_pos, motif.py:264).  dr is the reversed
// storage of D: D[i] = dr[CW - 1 - i].
template <int H>
__device__ __forceinline__ uint32_t aligned_word_rc(const uint32_t (&dr)[NW + 2 * H], int k, int sh, bool far) {
    constexpr int CW = NW + 2 * H;
    const int i = (H == 1 || !far) ? k + H : k + H + 1;  // D word holding the low part
    return __funnelshift_r(dr[CW - 1 - i], (i + 1 < CW) ? dr[CW - 2 - i] : 0u, sh);
}

// Word k (0 <= k < NW) of the match plane aligned at mod_pos: M[p] = S[p - mod_pos].
template <int H>
__device__ __forceinline__ uint32_t aligned_word(const uint32_t (&c)[NW + 2 * H], int k, int sh, bool far) {
    if (H == 1 || !far) return __funnelshift_l(c[k + H - 1], c[k + H], sh);
    return __funnelshift_l(c[k + H - 2], c[k + H - 1], sh);
}

template <int H, bool HASN>
__device__ __forceinline__ void match_words(const ProgramView &pv, const LaneSeq<H, HASN> &q,
                                            uint32_t (&m)[NW], const LaneEdge &edge) {
    uint32_t c[NW + 2 * H];
    run_chain<H, HASN>(pv, q, c, edge);
    const bool far = pv.mod_pos >= 32;  // only possible when H == 2
    const int sh = pv.mod_pos & 31;
#pragma unroll
    for (int k = 0; k < NW; ++k) m[k] = aligned_word<H>(c, k, sh, far);
}

// Load chunk t's words [-H, NW+H) of one record plane (shared or global memory).  `plane` points at the
// plane's left halo (16-byte aligned): kHalo halo words in natural order, the 2048 body words
// lane-interleaved (nmb200.h NMB_WORD_SLOT: the four uint4 vectors of chunk t sit at body + v*512 + t*4,
// so the lanes of a warp read consecutive 16-byte vectors), then kHalo right halo words.
template <int H>
__device__ __forceinline__ void load_plane(const uint32_t *plane, int t, uint32_t (&w)[NW + 2 * H]) {
    const uint32_t *body = plane + kHalo;
#pragma unroll
    for (int v = 0; v < NW / 4; ++v) {
        const uint4 a = *reinterpret_cast<const uint4 *>(body + v * kSlotStride + t * 4);
        w[H + 4 * v + 0] = a.x; w[H + 4 * v + 1] = a.y; w[H + 4 * v + 2] = a.z; w[H + 4 * v + 3] = a.w;
    }
    // halo: the last H words of chunk t-1 / the first H words of chunk t+1 (record halo at the tile edges)
    const uint32_t *pl = t > 0 ? body + (NW / 4 - 1) * kSlotStride + (t - 1) * 4 + (4 - H) : plane + (kHalo - H);
    const uint32_t *pr = t + 1 < kTileChunks ? body + (t + 1) * 4 : body + kTileWords;
#pragma unroll
    for (int i = 0; i < H; ++i) {
        w[i] = pl[i];
        w[NW + H + i] = pr[i];
    }
}

// px / py point at the x and y planes of a sequence record (shared or global); gn at word -H of the
// chunk in the flat non-ACGT plane (global).
template <int H>
__device__ __forceinline__ void load_xy(const uint32_t *px, const uint32_t *py, int t, LaneSeq<H, false> &q) {
    load_plane<H>(px, t, q.x);
    load_plane<H>(py, t, q.y);
}
template <int H>
__device__ __forceinline__ void load_xyn(const uint32_t *px, const uint32_t *py, int t, const uint32_t *gn,
                                         LaneSeq<H, true> &q) {
    load_plane<H>(px, t, q.x);
    load_plane<H>(py, t, q.y);
#pragma unroll
    for (int i = 0; i < NW + 2 * H; ++i) q.n[i] = __ldg(gn + i);
}

// Position of global chunk `chunk` (info = its chunk_info word) inside its contig.
__device__ __forceinline__ LaneEdge lane_edge(bool warp_edge, int info, int64_t chunk, const int64_t *contig_start,
                                              const int64_t *contig_len) {
    LaneEdge e;
    e.edge = warp_edge;
    e.hi = 1 << 20;
    e.first = false;
    if (warp_edge && info >= 0) {
        const int c = info & kChunkIdMask;
        const int64_t start = __ldg(contig_start + c), pos = chunk * NMB_CHUNK_BP;
        e.hi = (int)min(start + __ldg(contig_len + c) - pos, (int64_t)(1 << 20));
        e.first = pos == start;
    }
    return e;
}

}  // namespace nmb
