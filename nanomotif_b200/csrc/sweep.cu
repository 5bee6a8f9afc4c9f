// K8 -- exhaustive candidate sweep (BASELINE.json configs[4]): the counts of EVERY IUPAC motif of length 4..8
// at every modified position, without scanning per motif.
//
// Brute force is motif x bp work: 15^4 + ... + 15^8 = 2.7e9 motifs over a 2 Gbp assembly is ~5e18 motif*bp.  The
// counts that motif_model_bin returns (find_motifs_bin.py:1265-1331: pileup rows classified methylated /
// unmethylated whose position is the modified base of an occurrence, both strands) are additive over the
// CONCRETE sequence contexts of the rows, so one pass over the assembly suffices:
//   sweep_hist_kernel    for every window of 8 letters inside a contig and every classified row under it:
//                        hist[8][o][class][window] += 1, o = offset of the row in the window ('+' rows use
//                        the window, '-' rows its reverse complement with the offset mirrored -- the reference
//                        scans the reverse-complement motif on the forward text, find_motifs_bin.py:1317).
//                        Letters have FIVE states: A, T, G, C and "other" (non-ACGT), because the regex
//                        wildcard matches any character while sets do not (SURVEY App. B item 5).
//                        Only k = 8 is counted row by row (8 REDs per row instead of 4+5+6+7+8 = 30): a motif of
//                        k < 8 letters is the PREFIX of the (k+1)-letter motifs that extend it by one letter, so
//                            hist[k][o][c][w] = sum_j hist[k+1][o][c][5 w + j]  +  the k-windows that have no
//                                                                                  (k+1)-extension inside the contig
//                        ('+' rows: the one window that ends at the contig end; '-' rows, whose motif is the
//                        reverse complement and therefore extends to the LEFT in contig coordinates: the one window
//                        that starts at the contig start).  The kernel adds those edge windows directly (a handful
//                        per contig) and sweep_marginalise_kernel folds the levels 8 -> 7 -> ... -> 4 afterwards
//                        (nmb_sweep_finalize).
//   sweep_expand_kernel  subset-sum (zeta) transform, one axis at a time: 5 letter states -> 15 IUPAC letters
//                        (N includes "other").  After all axes, table[L_0 .. L_{k-1}] is the count of motif L.
//   sweep_filter_kernel  posterior-mean / support filter over a finished table -> candidate list.
// The modified position's own letter is fixed to one concrete base by the caller (a row under any other base
// cannot exist), which keeps the largest table at 15^7 entries.
#include "scan.cuh"

namespace nmb {

constexpr int kSweepMinK = 4, kSweepMaxK = 8;
__host__ __device__ constexpr int pow5(int k) { return k == 0 ? 1 : 5 * pow5(k - 1); }
// first counter of length k in the histogram array: sum_{j<k} j * 2 * 5^j
__host__ __device__ constexpr int64_t sweep_hist_offset(int k) {
    return k <= kSweepMinK ? 0 : sweep_hist_offset(k - 1) + (int64_t)(k - 1) * 2 * pow5(k - 1);
}
constexpr int64_t kSweepHistSize = sweep_hist_offset(kSweepMaxK + 1);  // 7 567 500 counters

// contig_slot == nullptr: one histogram, contigs [contig_begin, contig_end) counted.  Otherwise a chunk of contig c
// counts into histogram slot contig_slot[c] (skipped when outside [0, n_slots)), slots stacked at the histogram size.
struct SweepParams {
    const uint32_t *seq_records, *nonacgt, *cls;  // cls: the class records of ONE mod type
    const int64_t *contig_start, *contig_len;
    uint32_t *hist;
    const int32_t *contig_slot;
    int tile_begin, n_tiles_total, contig_begin, contig_end, n_slots;
};

// word w (0..16) of chunk t in a lane-interleaved plane; word 16 = first word of chunk t + 1
// (`next` supplies it for the last chunk of the tile)
__device__ __forceinline__ uint32_t chunk_word(const uint32_t *body, int t, int w, uint32_t next) {
    if (w < NW) return body[(w >> 2) * kSlotStride + t * 4 + (w & 3)];
    return t + 1 < kTileChunks ? body[(t + 1) * 4] : next;
}

template <int K>
__device__ __forceinline__ void sweep_add(uint32_t *hist, int code8, int rc8, unsigned plus, unsigned minus, int cls,
                                          int rem) {
    if (rem < K) return;  // the window of K letters must lie inside the contig
    uint32_t *h = hist + sweep_hist_offset(K);
    const int code = code8 / pow5(kSweepMaxK - K);  // first K letters
    const int rc = rc8 % pow5(K);                   // reverse complement of the first K letters
    for (unsigned b = plus & ((1u << K) - 1u); b; b &= b - 1) {
        const int o = __ffs(b) - 1;
        atomicAdd(h + (size_t)(o * 2 + cls) * pow5(K) + code, 1u);
    }
    for (unsigned b = minus & ((1u << K) - 1u); b; b &= b - 1) {
        const int o = K - 1 - (__ffs(b) - 1);  // offset of the row in the reverse-complement window
        atomicAdd(h + (size_t)(o * 2 + cls) * pow5(K) + rc, 1u);
    }
}

// ---- bipartite shapes X{3,4} N{4..8} Y{3,4} over ACGT (the second half of BASELINE config 5) ----
// Shape (a, g, b): a concrete letters, g wildcards, b concrete letters.  Block of shape (a, g, b):
// [o = 0..a+b-1][class][4^(a+b)], o counted over the concrete letters only; window index =
// xL | yL << a | xR << 2a | yR << (2a + b) with x / y the high / low code bits of the letters, letter i at bit i.
constexpr int kBipMinGap = 4, kBipMaxGap = 8;
__host__ __device__ constexpr int64_t bip_block(int a, int b) { return (int64_t)(a + b) * 2 * (1 << (2 * (a + b))); }
__host__ __device__ constexpr int64_t bip_offset(int a, int g, int b) {
    // order: g major, then (3,3) (3,4) (4,3) (4,4)
    return (int64_t)(g - kBipMinGap) * (bip_block(3, 3) + bip_block(3, 4) + bip_block(4, 3) + bip_block(4, 4)) +
           (a == 3 ? (b == 3 ? 0 : bip_block(3, 3)) : bip_block(3, 3) + bip_block(3, 4) + (b == 3 ? 0 : bip_block(4, 3)));
}
constexpr int64_t kBipHistSize = bip_offset(3, kBipMaxGap + 1, 3);

__device__ __forceinline__ unsigned rev_bits(unsigned v, int n) { return __brev(v) >> (32 - n); }

// Window of shape (A, G, B) starting at bit `s` of the 64-bit planes: '+' rows count under the window, '-' rows
// under its reverse complement, whose shape is (B, G, A).
template <int A, int G, int B>
__device__ __forceinline__ void bip_add(uint32_t *hist, uint64_t X, uint64_t Y, uint64_t N, uint64_t plus, uint64_t minus,
                                        int s, int cls, int rem, bool do_plus = true, bool do_minus = true) {
    constexpr int span = A + G + B;
    if (rem < span) return;
    constexpr unsigned ma = (1u << A) - 1u, mb = (1u << B) - 1u;
    const unsigned nl = (unsigned)(N >> s) & ma, nr = (unsigned)(N >> (s + A + G)) & mb;
    if (nl | nr) return;  // a concrete letter cannot match a non-ACGT letter
    const unsigned pl = do_plus ? (unsigned)(plus >> s) & ma : 0u, pr = do_plus ? (unsigned)(plus >> (s + A + G)) & mb : 0u;
    const unsigned ql = do_minus ? (unsigned)(minus >> s) & ma : 0u, qr = do_minus ? (unsigned)(minus >> (s + A + G)) & mb : 0u;
    if (!(pl | pr | ql | qr)) return;
    const unsigned xl = (unsigned)(X >> s) & ma, yl = (unsigned)(Y >> s) & ma;
    const unsigned xr = (unsigned)(X >> (s + A + G)) & mb, yr = (unsigned)(Y >> (s + A + G)) & mb;
    if (pl | pr) {
        uint32_t *h = hist + bip_offset(A, G, B);
        const unsigned code = xl | (yl << A) | (xr << (2 * A)) | (yr << (2 * A + B));
        for (unsigned b = pl | (pr << A); b; b &= b - 1) {
            const int o = __ffs(b) - 1;
            atomicAdd(h + (size_t)(o * 2 + cls) * (1u << (2 * (A + B))) + code, 1u);
        }
    }
    if (ql | qr) {  // the motif is the reverse complement of the window: shape (B, G, A), letters reversed, A<->T G<->C
        uint32_t *h = hist + bip_offset(B, G, A);
        const unsigned code = rev_bits(xr, B) | (rev_bits(~yr & mb, B) << B) | (rev_bits(xl, A) << (2 * B)) |
                              (rev_bits(~yl & ma, A) << (2 * B + A));
        // forward offset j (left part) -> motif offset B + (A - 1 - j); right part j -> B - 1 - j
        for (unsigned b = ql; b; b &= b - 1) {
            const int o = B + (A - 1 - (__ffs(b) - 1));
            atomicAdd(h + (size_t)(o * 2 + cls) * (1u << (2 * (A + B))) + code, 1u);
        }
        for (unsigned b = qr; b; b &= b - 1) {
            const int o = B - 1 - (__ffs(b) - 1);
            atomicAdd(h + (size_t)(o * 2 + cls) * (1u << (2 * (A + B))) + code, 1u);
        }
    }
}

// Only the shape (4, G, 4) is counted row by row.  The three shorter shapes are prefixes / suffixes of it at the MOTIF
// level -- (4,G,3) drops the motif's last letter, (3,G,4) its first, (3,G,3) then the last letter of (3,G,4) -- so
// nmb_sweep_bipartite_finalize gets them by summing over the dropped letter (4 concrete letters).  A window is counted
// directly only when the letter that would extend it is not a concrete letter of the same contig (non-ACGT, or past
// the contig's edge: inter-contig padding is flagged in the non-ACGT plane), because then no longer window covers it.
// '+' rows: motif = window, so "last letter" extends to the right and "first" to the left; '-' rows: motif = reverse
// complement, so the directions swap.  left_n = the letter left of the window start is not concrete.
template <int G>
__device__ __forceinline__ void bip_add_gap(uint32_t *hist, uint64_t X, uint64_t Y, uint64_t N, uint64_t plus,
                                            uint64_t minus, int s, int cls, int rem, bool left_n) {
    bip_add<4, G, 4>(hist, X, Y, N, plus, minus, s, cls, rem);
    const bool right4_n = (N >> (s + 7 + G)) & 1;  // the letter after a (4,G,3) window
    const bool right3_n = (N >> (s + 6 + G)) & 1;  // the letter after a (3,G,3) / before-last of (3,G,4)
    // fwd (4,G,3): '+' motif (4,G,3) and '-' motif (3,G,4) both extend to the right
    if (right4_n) bip_add<4, G, 3>(hist, X, Y, N, plus, minus, s, cls, rem);
    // fwd (3,G,4): '+' motif (3,G,4) and '-' motif (4,G,3) both extend to the left
    if (left_n) bip_add<3, G, 4>(hist, X, Y, N, plus, minus, s, cls, rem);
    // fwd (3,G,3): '+' motif comes from (3,G,4) at the same start (right extension), '-' motif from the reverse
    // complement of fwd (4,G,3) one letter to the left
    if (right3_n | left_n) bip_add<3, G, 3>(hist, X, Y, N, plus, minus, s, cls, rem, right3_n, left_n);
}

// One CTA per tile, one lane per 512-bp chunk, positions in order: the 8-letter window code slides by one letter
// per position (base-5 digits, most significant first; the reverse-complement code slides the other way).
// The minimum-blocks bound keeps the register counts the kernels had before slot routing (48 / 56: 10 / 9 CTAs per SM);
// unbounded, the routed histogram pointer costs the IUPAC variant 6 registers and one resident CTA.
template <bool BIPARTITE>
__global__ void __launch_bounds__(kTileChunks, BIPARTITE ? 9 : 10) sweep_hist_kernel(const SweepParams p) {
    // The records are read straight from global memory / L2 (the lane-interleaved layout keeps the lanes' words
    // adjacent): every word is used once, and without a 50 KB tile per CTA in shared memory three times as many
    // warps are resident to cover the latency of the divergent REDs (ncu on the staged version: issue-active 16 %,
    // long-scoreboard 16 per issue).
    const int tid = threadIdx.x;
    const int tile = p.tile_begin + blockIdx.x;
    const uint32_t *sx = p.seq_records + (size_t)tile * kSeqRecWords;
    const uint32_t *sy = sx + kSeqPlaneWords;
    const int info = reinterpret_cast<const int32_t *>(sy + kSeqPlaneWords)[tid];
    if (info < 0) return;
    const int contig = info & kChunkIdMask;
    // A lane's chunk lies in one contig and no window leaves its contig, so routing per lane keeps bins apart even
    // when their contigs share a tile.
    uint32_t *hist = p.hist;
    if (p.contig_slot) {
        const int slot = __ldg(p.contig_slot + contig);
        if (slot < 0 || slot >= p.n_slots) return;
        hist += (size_t)slot * (BIPARTITE ? kBipHistSize : kSweepHistSize);
    } else if (contig < p.contig_begin || contig >= p.contig_end) {
        return;
    }
    const uint32_t *scls = p.cls + (size_t)tile * kClsRecWords;
    const int64_t chunk_pos = ((int64_t)tile * kTileChunks + tid) * NMB_CHUNK_BP;
    const int64_t contig_start_pos = __ldg(p.contig_start + contig);
    const int64_t contig_end_pos = contig_start_pos + __ldg(p.contig_len + contig);
    const int n_here = (int)min((int64_t)NMB_CHUNK_BP, contig_end_pos - chunk_pos);  // window starts in this chunk
    // word 16 of every plane: the record halo / the next tile's class record for the last chunk
    const bool last_chunk = tid + 1 == kTileChunks;
    const bool has_next = tile + 1 < p.n_tiles_total;
    uint32_t next_cls[4] = {0, 0, 0, 0};
    if (last_chunk && has_next)
        for (int k = 0; k < 4; ++k) next_cls[k] = __ldg(p.cls + (size_t)(tile + 1) * kClsRecWords + k * kTileWords);
    const uint32_t next_x = sx[kHalo + kTileWords], next_y = sy[kHalo + kTileWords];
    const uint32_t *gn = p.nonacgt + kHalo + (size_t)tile * kTileWords + tid * NW;

    uint64_t X = 0, Y = 0, N = 0, C0 = 0, C1 = 0, C2 = 0, C3 = 0;  // bit i = position (32 * word + i) of the current pair
    auto load_pair = [&](int w) {  // words w and w + 1 of the seven planes
        const uint64_t x0 = chunk_word(sx + kHalo, tid, w, next_x), x1 = w + 1 <= NW ? chunk_word(sx + kHalo, tid, w + 1, next_x) : 0;
        const uint64_t y0 = chunk_word(sy + kHalo, tid, w, next_y), y1 = w + 1 <= NW ? chunk_word(sy + kHalo, tid, w + 1, next_y) : 0;
        X = x0 | (x1 << 32);
        Y = y0 | (y1 << 32);
        N = (uint64_t)__ldg(gn + w) | ((uint64_t)(w + 1 <= NW ? __ldg(gn + w + 1) : 0xFFFFFFFFu) << 32);
        const uint64_t a0 = chunk_word(scls, tid, w, next_cls[0]), a1 = w + 1 <= NW ? chunk_word(scls, tid, w + 1, next_cls[0]) : 0;
        const uint64_t b0 = chunk_word(scls + kTileWords, tid, w, next_cls[1]), b1 = w + 1 <= NW ? chunk_word(scls + kTileWords, tid, w + 1, next_cls[1]) : 0;
        const uint64_t c0 = chunk_word(scls + 2 * kTileWords, tid, w, next_cls[2]), c1 = w + 1 <= NW ? chunk_word(scls + 2 * kTileWords, tid, w + 1, next_cls[2]) : 0;
        const uint64_t d0 = chunk_word(scls + 3 * kTileWords, tid, w, next_cls[3]), d1 = w + 1 <= NW ? chunk_word(scls + 3 * kTileWords, tid, w + 1, next_cls[3]) : 0;
        C0 = a0 | (a1 << 32);
        C1 = b0 | (b1 << 32);
        C2 = c0 | (c1 << 32);
        C3 = d0 | (d1 << 32);
    };
    auto letter = [&](int i) -> int {  // state of position i (0..63) of the current pair: A T G C other
        return ((N >> i) & 1) ? 4 : (int)((((X >> i) & 1) << 1) | ((Y >> i) & 1));
    };
    auto comp = [](int d) -> int { return d < 4 ? (d ^ 1) : 4; };  // A<->T, G<->C

    load_pair(0);
    bool left_n = (__ldg(gn - 1) >> 31) & 1;  // the letter before the chunk (padding and pad words are flagged)
    int code8 = 0, rc8 = 0, first = 0;  // first = the window's leading letter (leaves on the next slide)
    for (int i = 0; i < kSweepMaxK; ++i) {
        const int d = letter(i);
        code8 = code8 * 5 + d;
        rc8 += comp(d) * pow5(i);
        if (i == 0) first = d;
    }
    for (int s = 0; s < n_here; ++s) {
        const int b = s & 31;
        if (b == 0 && s) load_pair(s >> 5);
        if (BIPARTITE) {  // spans of 10..16 letters: bits b .. b + 15 of the pairs
            const int rem16 = (int)min((int64_t)16, contig_end_pos - (chunk_pos + s));
            if ((C0 | C2) >> b & 0xFFFF) {
                bip_add_gap<4>(hist, X, Y, N, C0, C2, b, 0, rem16, left_n);
                bip_add_gap<5>(hist, X, Y, N, C0, C2, b, 0, rem16, left_n);
                bip_add_gap<6>(hist, X, Y, N, C0, C2, b, 0, rem16, left_n);
                bip_add_gap<7>(hist, X, Y, N, C0, C2, b, 0, rem16, left_n);
                bip_add_gap<8>(hist, X, Y, N, C0, C2, b, 0, rem16, left_n);
            }
            if ((C1 | C3) >> b & 0xFFFF) {
                bip_add_gap<4>(hist, X, Y, N, C1, C3, b, 1, rem16, left_n);
                bip_add_gap<5>(hist, X, Y, N, C1, C3, b, 1, rem16, left_n);
                bip_add_gap<6>(hist, X, Y, N, C1, C3, b, 1, rem16, left_n);
                bip_add_gap<7>(hist, X, Y, N, C1, C3, b, 1, rem16, left_n);
                bip_add_gap<8>(hist, X, Y, N, C1, C3, b, 1, rem16, left_n);
            }
            left_n = (N >> b) & 1;
            continue;
        }
        const int rem = (int)min((int64_t)kSweepMaxK, contig_end_pos - (chunk_pos + s));
        const unsigned mp = (unsigned)(C0 >> b) & 0xFF, np = (unsigned)(C1 >> b) & 0xFF;  // rows under the window, '+'
        const unsigned mm = (unsigned)(C2 >> b) & 0xFF, nm = (unsigned)(C3 >> b) & 0xFF;  // '-'
        if (rem >= kSweepMaxK) {  // the common case: the 8-window lies inside the contig
            if (mp | mm) sweep_add<8>(hist, code8, rc8, mp, mm, 0, rem);
            if (np | nm) sweep_add<8>(hist, code8, rc8, np, nm, 1, rem);
        }
        // k < 8 comes from marginalising k + 1 (nmb_sweep_finalize) except for the windows without an extension inside
        // the contig: '+' rows under the k-window that ENDS at the contig end (rem == k), '-' rows under the k-window
        // that STARTS at the contig start
        const bool at_start = s == 0 && chunk_pos == contig_start_pos;
        if (rem < kSweepMaxK || at_start) {
#define NMB_EDGE(K)                                                                                              \
            {                                                                                                    \
                const unsigned pm = rem == K ? mp : 0u, pn = rem == K ? np : 0u;                                 \
                const unsigned qm = at_start ? mm : 0u, qn = at_start ? nm : 0u;                                 \
                if (pm | qm) sweep_add<K>(hist, code8, rc8, pm, qm, 0, rem);                                     \
                if (pn | qn) sweep_add<K>(hist, code8, rc8, pn, qn, 1, rem);                                     \
            }
            NMB_EDGE(4) NMB_EDGE(5) NMB_EDGE(6) NMB_EDGE(7)
#undef NMB_EDGE
        }
        // slide: drop the leading letter, append the letter at s + 8
        const int d_new = letter(b + kSweepMaxK);
        code8 = (code8 - first * pow5(kSweepMaxK - 1)) * 5 + d_new;
        rc8 = (rc8 - comp(first)) / 5 + comp(d_new) * pow5(kSweepMaxK - 1);
        first = letter(b + 1);
    }
}

// hist[k][o][c][w] += sum_{j < 5} hist[k + 1][o][c][5 w + j] for o < k: a k-letter motif is the prefix of its five
// one-letter extensions (the trailing letter is the least significant base-5 digit).  blockIdx.y = histogram slot.
__global__ void __launch_bounds__(256) sweep_marginalise_kernel(uint32_t *__restrict__ hist, int k) {
    hist += (size_t)blockIdx.y * kSweepHistSize;
    int n5 = 1;
    for (int i = 0; i < k; ++i) n5 *= 5;
    const int64_t n = (int64_t)k * 2 * n5;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t oc = i / n5, w = i - oc * n5;  // oc = o * 2 + class, the same index in both levels (o < k)
    int64_t off_k = 0, off_k1 = 0;               // sweep_hist_offset(k), sweep_hist_offset(k + 1)
    for (int j = kSweepMinK, p5 = pow5(kSweepMinK); j <= k; ++j, p5 *= 5) {
        if (j < k) off_k += (int64_t)j * 2 * p5;
        off_k1 += (int64_t)j * 2 * p5;
    }
    const uint32_t *src = hist + off_k1 + oc * (int64_t)n5 * 5 + w * 5;
    hist[off_k + i] += src[0] + src[1] + src[2] + src[3] + src[4];
}

// Bipartite marginals (see bip_add_gap).  mode 0: shape (a, b) += sum over the LAST right letter of shape (a, b + 1),
// same offsets; mode 1: shape (a, b) += sum over the FIRST left letter of shape (a + 1, b), offset o <- o + 1.
// blockIdx.y = histogram slot.
__global__ void __launch_bounds__(256) bip_marginalise_kernel(uint32_t *__restrict__ hist, int g, int a, int b, int mode) {
    hist += (size_t)blockIdx.y * kBipHistSize;
    const int n_code = 1 << (2 * (a + b));
    const int64_t n = (int64_t)(a + b) * 2 * n_code;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int oc = (int)(i / n_code), code = (int)(i - (int64_t)oc * n_code);
    const int o = oc >> 1, cls = oc & 1;
    const unsigned xl = code & ((1u << a) - 1), yl = (code >> a) & ((1u << a) - 1);
    const unsigned xr = (code >> (2 * a)) & ((1u << b) - 1), yr = (code >> (2 * a + b)) & ((1u << b) - 1);
    const int sa = mode ? a + 1 : a, sb = mode ? b : b + 1;
    const uint32_t *src = hist + bip_offset(sa, g, sb) + (size_t)(((mode ? o + 1 : o) * 2 + cls)) * (1u << (2 * (sa + sb)));
    uint32_t sum = 0;
    for (unsigned t = 0; t < 4; ++t) {
        const unsigned tx = t >> 1, ty = t & 1;
        unsigned sxl = xl, syl = yl, sxr = xr, syr = yr;
        if (mode) { sxl = (xl << 1) | tx; syl = (yl << 1) | ty; }
        else { sxr = xr | (tx << b); syr = yr | (ty << b); }
        sum += src[sxl | (syl << sa) | (sxr << (2 * sa)) | (syr << (2 * sa + sb))];
    }
    hist[bip_offset(a, g, b) + i] += sum;
}

// The sums of the 4 concrete letter states over the 14 IUPAC letters other than N: A T G C R Y S W K M B D H V.
__device__ __forceinline__ void acgt_sums(uint32_t a, uint32_t t, uint32_t g, uint32_t c, uint32_t *v) {
    v[0] = a; v[1] = t; v[2] = g; v[3] = c;
    v[4] = a + g; v[5] = c + t; v[6] = g + c; v[7] = a + t; v[8] = g + t; v[9] = a + c;
    v[10] = c + g + t; v[11] = a + g + t; v[12] = a + c + t; v[13] = a + c + g;
}

// The 15 IUPAC sums of the 5 letter states s[0], s[inner], ..., s[4 * inner] (A T G C other).
__device__ __forceinline__ void iupac_sums(const uint32_t *s, int64_t inner, uint32_t v[15]) {
    const uint32_t a = s[0], t = s[inner], g = s[2 * inner], c = s[3 * inner], x = s[4 * inner];
    // N also takes the "other" state: the regex wildcard matches non-ACGT letters
    acgt_sums(a, t, g, c, v);
    v[14] = a + c + g + t + x;
}

__device__ __forceinline__ bool sweep_pass(uint32_t m, uint32_t n, double min_mean, uint32_t min_mod) {
    return m >= min_mod && (5.0 + m) / (10.0 + m + n) >= min_mean;
}

// dst[outer][15][inner] = subset sums of src[outer][5][inner] over the letters of each IUPAC code.
// Letter states: A T G C other; IUPAC order = nanomotif/constants.py:2 (A T G C R Y S W K M B D H V N).
__global__ void __launch_bounds__(256) sweep_expand_kernel(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst,
                                                           int64_t outer, int64_t inner) {
    const int64_t n = outer * inner;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t o = i / inner, r = i - o * inner;
        uint32_t v[15];
        iupac_sums(src + o * 5 * inner + r, inner, v);
        uint32_t *d = dst + o * 15 * inner + r;
        for (int l = 0; l < 15; ++l) d[l * inner] = v[l];
    }
}

// dst[...] = src[... with the digit of axis `axis_stride` fixed to `digit` ...]: drops one base-5 axis.
// blockIdx.y = slot: src at slot * src_slot_stride, dst stacked [slot][n_out].
__global__ void __launch_bounds__(256) sweep_slice_kernel(const uint32_t *__restrict__ src, int64_t src_slot_stride,
                                                          uint32_t *__restrict__ dst, int64_t n_out, int64_t axis_stride,
                                                          int digit) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_out) return;
    src += blockIdx.y * src_slot_stride;
    dst += blockIdx.y * n_out;
    const int64_t hi = i / axis_stride, lo = i - hi * axis_stride;
    dst[i] = src[(hi * 5 + digit) * axis_stride + lo];
}

// ---- degenerate bipartite halves: X{a} N{g} Y{b} with any of the 14 IUPAC letters other than N in X and Y ----
// A half letter other than N matches only the four concrete contig letters, and bip_add skips every window with a
// non-ACGT letter in a half, so the count of such a motif is the sum of the finished ACGT counters over the concrete
// letters each of its letters stands for: a 4-state -> 14-letter subset sum, one axis per letter, on the bit-planar
// blocks.  N in a half would need a fifth ("other") state in the histogram pass.

// dst[slot][w] = the (shape (a, b), offset o, class cls) block of slot `slot` of finished bipartite histograms stacked
// at kBipHistSize (`block` = bip_offset(a, g, b)), with the letter at offset o fixed to `canonical` and the other
// a + b - 1 letters written as base-4 digits w (A=0 T=1 G=2 C=3), first letter most significant.  blockIdx.y = slot.
__global__ void __launch_bounds__(256) bip_iupac_slice_kernel(const uint32_t *__restrict__ hist, int64_t block, int a,
                                                              int b, int o, int cls, int canonical,
                                                              uint32_t *__restrict__ dst) {
    const int n_out = 1 << (2 * (a + b - 1));
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_out) return;
    const uint32_t *h = hist + (size_t)blockIdx.y * kBipHistSize + block + (size_t)(o * 2 + cls) * (1u << (2 * (a + b)));
    unsigned code = 0;
    for (int p = a + b - 1, w = i; p >= 0; --p) {  // last letter = least significant digit
        int d = canonical;
        if (p != o) { d = w & 3; w >>= 2; }
        const int xbit = p < a ? p : 2 * a + (p - a), ybit = p < a ? a + p : 2 * a + b + (p - a);
        code |= (unsigned)(d >> 1) << xbit | (unsigned)(d & 1) << ybit;
    }
    dst[(size_t)blockIdx.y * n_out + i] = h[code];
}

// dst[outer][14][inner] = sums of src[outer][4][inner] over the concrete letters of each IUPAC letter but N.
__global__ void __launch_bounds__(256) bip_iupac_expand_kernel(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst,
                                                               int64_t outer, int64_t inner) {
    const int64_t n = outer * inner;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t o = i / inner, r = i - o * inner;
        const uint32_t *s = src + o * 4 * inner + r;
        uint32_t v[14];
        acgt_sums(s[0], s[inner], s[2 * inner], s[3 * inner], v);
        uint32_t *d = dst + o * 14 * inner + r;
        for (int l = 0; l < 14; ++l) d[l * inner] = v[l];
    }
}

// Candidates of one finished table pair: posterior mean (5 + n_mod) / (10 + n_mod + n_nomod) >= min_mean and
// n_mod >= min_mod (Beta(5, 5) prior, nanomotif/model.py:8-9).  Appends the table index; *n_out counts all hits.
__global__ void __launch_bounds__(256) sweep_filter_kernel(const uint32_t *__restrict__ n_mod,
                                                           const uint32_t *__restrict__ n_nomod, int64_t n,
                                                           double min_mean, uint32_t min_mod, int64_t *__restrict__ out,
                                                           int64_t capacity, unsigned long long *__restrict__ n_out) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (!sweep_pass(n_mod[i], n_nomod[i], min_mean, min_mod)) continue;
        const unsigned long long slot = atomicAdd(n_out, 1ull);
        if ((int64_t)slot < capacity) out[slot] = i;
    }
}

// ---- pruning (ABI 7): drop candidates that are a redundant specialisation or a mixture of a neighbour ----
// A candidate M (it passes sweep_pass) is widened at one letter other than the modified one by one base (P) or
// narrowed by one (C); Q is the difference of the counts, P - M or M - C.  M is pruned when
//   (a) some widening P passes and Q's posterior mean is >= min_mean (the added base is methylated too), or
//   (b) some narrowing C passes and Q's posterior mean is < min_mean (the removed base is not methylated).
// Widening and narrowing follow the covering relation of a lattice of letters, each a set of letter states:
//   contiguous: the 15 IUPAC letters over A T G C other (N = every state: a 3-base letter widens to N, which adds a
//               base and "other", as iupac_sums counts it);
//   bipartite ACGT halves: A T G C and the pseudo-letter * = {A, C, G, T}, which is never a row;
//   bipartite IUPAC halves: the 14 letters other than N and * above the 3-base letters.
struct PruneLattice {
    int n;               // letters; index n - 1 is the widest (N or *)
    uint32_t states[15];  // bit s: the letter stands for state s (A=0 T=1 G=2 C=3 other=4)
    uint32_t widen[15];   // bit e: letter e covers this letter (the smallest supersets in the lattice)
    uint32_t narrow[15];  // bit e: this letter covers letter e
};

__host__ __device__ constexpr bool strict_subset(uint32_t x, uint32_t y) { return x != y && (x & y) == x; }

__host__ __device__ constexpr PruneLattice prune_lattice(int n, const uint32_t (&states)[15]) {
    PruneLattice L{n, {}, {}, {}};
    for (int i = 0; i < n; ++i) L.states[i] = states[i];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            if (!strict_subset(states[i], states[j])) continue;
            bool between = false;
            for (int l = 0; l < n; ++l)
                between = between || (strict_subset(states[i], states[l]) && strict_subset(states[l], states[j]));
            if (!between) {
                L.widen[i] |= 1u << j;
                L.narrow[j] |= 1u << i;
            }
        }
    return L;
}

// letter states in table order: IUPAC_ORDER (A T G C R Y S W K M B D H V N), the 14 without N + *, A T G C + *
constexpr uint32_t kPruneStatesIupac[15] = {1, 2, 4, 8, 5, 10, 12, 3, 6, 9, 14, 7, 11, 13, 31};
constexpr uint32_t kPruneStatesBipIupac[15] = {1, 2, 4, 8, 5, 10, 12, 3, 6, 9, 14, 7, 11, 13, 15};
constexpr uint32_t kPruneStatesBipAcgt[15] = {1, 2, 4, 8, 15};
constexpr PruneLattice kPruneLattices[3] = {prune_lattice(15, kPruneStatesIupac), prune_lattice(5, kPruneStatesBipAcgt),
                                            prune_lattice(15, kPruneStatesBipIupac)};
enum { kLatticeIupac = 0, kLatticeBipAcgt = 1, kLatticeBipIupac = 2 };
__constant__ PruneLattice c_prune_lattices[3] = {kPruneLattices[0], kPruneLattices[1], kPruneLattices[2]};

// Q's posterior mean, with the arithmetic of sweep_pass
__device__ __forceinline__ double prune_q_mean(uint32_t q_mod, uint32_t q_nomod) {
    return (5.0 + q_mod) / (10.0 + q_mod + q_nomod);
}

// Whether the candidate (m, u) is pruned by the neighbour (nm, nu) that widens it (`wider`) or that it widens.
__device__ __forceinline__ bool pruned_by(bool wider, uint32_t m, uint32_t u, uint32_t nm, uint32_t nu, double min_mean,
                                          uint32_t min_mod) {
    if (!sweep_pass(nm, nu, min_mean, min_mod)) return false;
    return wider ? prune_q_mean(nm - m, nu - u) >= min_mean : prune_q_mean(m - nm, u - nu) < min_mean;
}

// Sum of s[t * inner] over the states t of `states` (the register axis of one table entry).
template <int S>
__device__ __forceinline__ uint32_t state_sum(const uint32_t *s, int64_t inner, uint32_t states) {
    uint32_t v = 0;
#pragma unroll
    for (int t = 0; t < S; ++t)
        if (states >> t & 1) v += s[t * inner];
    return v;
}

// v[l] for a letter l known only at run time, without moving v out of registers.
template <int N>
__device__ __forceinline__ uint32_t pick(const uint32_t (&v)[N], int l) {
    uint32_t x = 0;
#pragma unroll
    for (int j = 0; j < N; ++j) x = j == l ? v[j] : x;
    return x;
}

// Whether letter d of the register axis at entry r of one slot's [S][inner] input is pruned (mb / ub: n_mod / n_nomod
// of the slot; m / u: the register sums of entry r, index L.n - 1 the widest letter).  The other axes are the base-B
// digits of r, most significant first; a neighbour letter e >= B on such an axis (*) is the sum of the entries with
// its states' digits, which are the concrete letters 0..S-1 of the table.
template <int S, int B>
__device__ __forceinline__ bool expand_pruned(const PruneLattice &L, const uint32_t *mb, const uint32_t *ub,
                                              int64_t inner, int64_t r, int d, const uint32_t (&m)[15],
                                              const uint32_t (&u)[15], double min_mean, uint32_t min_mod) {
    const uint32_t md = pick(m, d), ud = pick(u, d);
    for (uint32_t e = L.widen[d] | L.narrow[d]; e; e &= e - 1) {
        const int l = __ffs(e) - 1;
        if (pruned_by(L.widen[d] >> l & 1, md, ud, pick(m, l), pick(u, l), min_mean, min_mod)) return true;
    }
    const uint32_t sd = L.states[d];
    for (int64_t pv = inner / B; pv >= 1; pv /= B) {
        const int c = (int)(r / pv % B);
        for (uint32_t e = L.widen[c] | L.narrow[c]; e; e &= e - 1) {
            const int l = __ffs(e) - 1;
            uint32_t nm = 0, nu = 0;
            if (l < B) {
                const int64_t r2 = r + (int64_t)(l - c) * pv;
                nm = state_sum<S>(mb + r2, inner, sd);
                nu = state_sum<S>(ub + r2, inner, sd);
            } else {
                for (uint32_t t = L.states[l]; t; t &= t - 1) {
                    const int64_t r2 = r + (int64_t)(__ffs(t) - 1 - c) * pv;
                    nm += state_sum<S>(mb + r2, inner, sd);
                    nu += state_sum<S>(ub + r2, inner, sd);
                }
            }
            if (pruned_by(L.widen[c] >> l & 1, md, ud, nm, nu, min_mean, min_mod)) return true;
        }
    }
    return false;
}

// v[0..14] = the letter sums of the S states s[0], s[inner], ..., s[(S - 1) * inner]: for S = 5 the 15 IUPAC letters
// (iupac_sums), for S = 4 the 14 letters other than N and, at index 14, the pseudo-letter * = the sum of the 4 states.
template <int S>
__device__ __forceinline__ void letter_sums(const uint32_t *s, int64_t inner, uint32_t (&v)[15]) {
    if constexpr (S == 5) {
        iupac_sums(s, inner, v);
    } else {
        acgt_sums(s[0], s[inner], s[2 * inner], s[3 * inner], v);
        v[14] = s[0] + s[inner] + s[2 * inner] + s[3 * inner];
    }
}

// Appends (slot, index r + d * inner, m[d], u[d]) for every letter d < N set in `hits`.  *n_out counts all hits, at
// most `capacity` records are written (count-then-fill).
template <int N>
__device__ __forceinline__ void append_hits(uint32_t hits, int64_t slot, int64_t inner, int64_t r, const uint32_t *m,
                                            const uint32_t *u, nmb_sweep_hit *__restrict__ out, int64_t capacity,
                                            unsigned long long *__restrict__ n_out) {
    unsigned long long at = atomicAdd(n_out, (unsigned long long)__popc(hits));
    for (int d = 0; d < N; ++d) {
        if (!(hits >> d & 1)) continue;
        if ((int64_t)at < capacity) out[at] = nmb_sweep_hit{(int32_t)slot, (uint32_t)(d * inner + r), m[d], u[d]};
        ++at;
    }
}

// The last expansion pass fused with the filter: the most significant table axis of src[slot][S][inner] is expanded
// in registers and every entry that passes sweep_filter_kernel's test (same arithmetic) is appended as (slot, table
// index = letter * inner + r, n_mod, n_nomod); the expanded table is never written.
//   S = 5: the 15 IUPAC letters of nmb_sweep_expand (contiguous k-mers, inner = 15^(k-2)).  Motifs whose first or
//          last letter is N are skipped (canonical form) unless that letter is the modified position's fixed base.
//   S = 4: the 14 letters of nmb_sweep_bip_iupac_expand (degenerate bipartite halves, inner = 14^(a+b-2)).
// PRUNE drops the candidates that expand_pruned prunes: neighbours on the register axis come from the register sums
// (index 14: N, or for S = 4 the pseudo-letter * = the sum of the 4 states), those on the other axes from the entry
// with that digit of r replaced (a flanking N included: GATCN prunes GATCB; * is the sum of the entries with A, T, G
// and C there).  Only candidates that pass look at their neighbours.
template <int S, bool PRUNE>
__global__ void __launch_bounds__(256) expand_filter_kernel(const uint32_t *__restrict__ n_mod,
                                                            const uint32_t *__restrict__ n_nomod, int64_t n_slots,
                                                            int64_t inner, bool skip_first_n, bool skip_last_n,
                                                            double min_mean, uint32_t min_mod,
                                                            nmb_sweep_hit *__restrict__ out, int64_t capacity,
                                                            unsigned long long *__restrict__ n_out) {
    constexpr int L = S == 5 ? 15 : 14;  // letters of the register axis
    const int64_t n = n_slots * inner;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t slot = i / inner, r = i - slot * inner;
        const uint32_t *mb = n_mod + slot * S * inner, *ub = n_nomod + slot * S * inner;
        uint32_t m[15], u[15];
        letter_sums<S>(mb + r, inner, m);
        uint32_t hits = 0;  // bit d: letter d passes
        const int last = S == 5 && skip_last_n && r % 15 == 14 ? 0 : L;
        for (int d = 0; d < last; ++d)
            if (m[d] >= min_mod) hits |= 1u << d;
        if (S == 5 && skip_first_n) hits &= ~(1u << 14);
        if (!hits) continue;
        letter_sums<S>(ub + r, inner, u);
        for (int d = 0; d < L; ++d)
            if ((hits >> d & 1) && !sweep_pass(m[d], u[d], min_mean, min_mod)) hits &= ~(1u << d);
        if constexpr (PRUNE) {
            const PruneLattice &lat = c_prune_lattices[S == 5 ? kLatticeIupac : kLatticeBipIupac];
#pragma unroll 1
            for (uint32_t h = hits; h; h &= h - 1) {
                const int d = __ffs(h) - 1;
                if (expand_pruned<S, L>(lat, mb, ub, inner, r, d, m, u, min_mean, min_mod)) hits &= ~(1u << d);
            }
        }
        if (!hits) continue;
        append_hits<L>(hits, slot, inner, r, m, u, out, capacity, n_out);
    }
}

// Candidates of finished bipartite histograms stacked [slot][kBipHistSize]: every n_mod counter (class 0) whose
// concrete letter at the counter's offset is `canonical` (A=0 T=1 G=2 C=3) and that passes the test of
// sweep_filter_kernel; index = the counter's position in its slot's histogram.  PRUNE: every letter but the modified
// one widens to *, the sum of the 4 counters whose code differs only in that letter's x and y bits (same block,
// offset and class).
template <bool PRUNE>
__global__ void __launch_bounds__(256) bip_filter_kernel(const uint32_t *__restrict__ hist, int64_t n_slots, int canonical,
                                                         double min_mean, uint32_t min_mod, nmb_sweep_hit *__restrict__ out,
                                                         int64_t capacity, unsigned long long *__restrict__ n_out) {
    constexpr int64_t b33 = bip_block(3, 3), b34 = bip_block(3, 4), b43 = bip_block(4, 3);
    constexpr int64_t per_gap = bip_offset(3, kBipMinGap + 1, 3);
    const int64_t n = n_slots * kBipHistSize;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint32_t m = hist[i];
        if (m < min_mod) continue;
        const int64_t slot = i / kBipHistSize, j = i - slot * kBipHistSize;
        int64_t rem = j % per_gap;
        int a, b;
        if (rem < b33) { a = 3; b = 3; }
        else if (rem < b33 + b34) { a = 3; b = 4; rem -= b33; }
        else if (rem < b33 + b34 + b43) { a = 4; b = 3; rem -= b33 + b34; }
        else { a = 4; b = 4; rem -= b33 + b34 + b43; }
        const int bits = 2 * (a + b);
        const int oc = (int)(rem >> bits), code = (int)(rem & ((1 << bits) - 1));
        if (oc & 1) continue;  // an n_nomod counter
        const int o = oc >> 1;
        auto xbit = [&](int p) { return p < a ? p : 2 * a + (p - a); };
        auto ybit = [&](int p) { return p < a ? a + p : 2 * a + b + (p - a); };
        auto letter = [&](int p) { return ((code >> xbit(p)) & 1) << 1 | ((code >> ybit(p)) & 1); };
        if (letter(o) != canonical) continue;
        const uint32_t u = hist[i + (1 << bits)];
        if (!sweep_pass(m, u, min_mean, min_mod)) continue;
        if constexpr (PRUNE) {
            const PruneLattice &L = c_prune_lattices[kLatticeBipAcgt];
            const uint32_t *block = hist + (i - code);  // code 0 of this (shape, offset, class 0) block
            bool pruned = false;
            for (int p = 0; p < a + b && !pruned; ++p) {
                if (p == o) continue;
                const int c = letter(p), rest = code & ~(1 << xbit(p) | 1 << ybit(p));
                for (uint32_t e = L.widen[c] | L.narrow[c]; e && !pruned; e &= e - 1) {
                    const int l = __ffs(e) - 1;
                    uint32_t nm = 0, nu = 0;
                    for (uint32_t t = L.states[l]; t; t &= t - 1) {
                        const int x = __ffs(t) - 1;
                        const int c2 = rest | (x >> 1) << xbit(p) | (x & 1) << ybit(p);
                        nm += block[c2];
                        nu += block[c2 + (1 << bits)];
                    }
                    pruned = pruned_by(L.widen[c] >> l & 1, m, u, nm, nu, min_mean, min_mod);
                }
            }
            if (pruned) continue;
        }
        append_hits<1>(1u, slot, 0, j, &m, &u, out, capacity, n_out);
    }
}

// ---- lookup (ABI 9): the counts of listed motifs, gathered from the finished histograms (nmb_sweep_query) ----
// One warp per (query, run of kLookupRun output rows).  A query of >= 32 cells spreads its cells over the 32 lanes and
// takes the run's rows one after the other; a smaller one puts 32 / cells rows side by side, one cell per lane.  Each
// lane sums its cells in uint64, the lanes of a row are reduced with shuffles and the row's first lane writes the pair:
// no atomics, so the sums do not depend on the schedule.  The cost is proportional to the cells read.
constexpr int kLookupRun = 32, kLookupWarps = 8;
constexpr int kLookupMaxPos = 7, kLookupQueryWords = (int)(sizeof(nmb_sweep_query) / 4);
static_assert(sizeof(nmb_sweep_query) == 168, "nmb_sweep_query layout is fixed by the header");

// Whether every counter the record addresses lies inside its slot's histogram (both classes).
__device__ __forceinline__ bool lookup_readable(const nmb_sweep_query &q, const uint32_t *table, int64_t size) {
    if (!table || q.kind < 0 || q.kind > 1 || q.n_pos < 0 || q.n_pos > kLookupMaxPos || q.base < 0 || q.class_step < 0)
        return false;
    const int max_states = q.kind == 0 ? 5 : 4;
    int64_t last = q.base + q.class_step;
    for (int p = 0; p < q.n_pos; ++p) {
        if (q.n_states[p] < 1 || q.n_states[p] > max_states) return false;
        int32_t hi = 0;
        for (int d = 0; d < q.n_states[p]; ++d) {
            if (q.offset[p][d] < 0) return false;
            hi = max(hi, q.offset[p][d]);
        }
        last += hi;
    }
    return last < size;
}

__global__ void __launch_bounds__(kLookupWarps * 32) sweep_lookup_kernel(const uint32_t *__restrict__ hist,
                                                                          const uint32_t *__restrict__ bip,
                                                                          const int32_t *__restrict__ slots, int n_rows,
                                                                          const nmb_sweep_query *__restrict__ queries,
                                                                          int64_t n_queries, int64_t *__restrict__ out) {
    __shared__ nmb_sweep_query sq[kLookupWarps];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const nmb_sweep_query &q = sq[w];
    const int runs = (n_rows + kLookupRun - 1) / kLookupRun;
    const int64_t items = n_queries * runs, warps = (int64_t)gridDim.x * kLookupWarps;
    for (int64_t item = (int64_t)blockIdx.x * kLookupWarps + w; item < items; item += warps) {
        const int64_t qi = item / runs;
        const int r0 = (int)(item - qi * runs) * kLookupRun, r1 = min(r0 + kLookupRun, n_rows);
        __syncwarp();  // the lanes are done with the previous record
        const uint32_t *src = reinterpret_cast<const uint32_t *>(queries + qi);
        for (int i = lane; i < kLookupQueryWords; i += 32) reinterpret_cast<uint32_t *>(&sq[w])[i] = __ldg(src + i);
        __syncwarp();
        const uint32_t *table = q.kind == 1 ? bip : hist;
        const int64_t size = q.kind == 1 ? kBipHistSize : kSweepHistSize;
        if (!lookup_readable(q, table, size)) {
            for (int r = r0 + lane; r < r1; r += 32) {
                int64_t *o = out + ((int64_t)r * n_queries + qi) * 2;
                o[0] = o[1] = -1;
            }
            continue;
        }
        const int n_pos = q.n_pos;
        uint32_t radix[kLookupMaxPos], magic[kLookupMaxPos];
        int cells = 1;
#pragma unroll
        for (int p = 0; p < kLookupMaxPos; ++p) {
            radix[p] = p < n_pos ? q.n_states[p] : 1u;
            magic[p] = 0xFFFFFFFFu / radix[p] + 1u;  // x / radix = umulhi(x, magic), exact for x < 2^17 (radix > 1)
            cells *= (int)radix[p];
        }
        const int span = min(cells, 32), per = 32 / span, seg = lane / span, j0 = lane - seg * span;
        const uint32_t *base = table + q.base;
        const int64_t step = q.class_step;
        for (int r = r0; r < r1; r += per) {  // uniform over the warp: the shuffles below see every lane
            const int row = r + seg;
            const bool mine = seg < per && row < r1;
            uint64_t s0 = 0, s1 = 0;
            const int slot = mine ? (slots ? __ldg(slots + row) : row) : -1;
            if (slot >= 0) {
                const uint32_t *h = base + (int64_t)slot * size;
                for (int c = j0; c < cells; c += span) {
                    uint32_t x = (uint32_t)c;
                    int32_t off = 0;
#pragma unroll
                    for (int p = kLookupMaxPos - 1; p >= 0; --p) {  // the last position is the least significant digit
                        if (p >= n_pos) continue;
                        const uint32_t qt = radix[p] == 1u ? x : __umulhi(x, magic[p]);
                        off += q.offset[p][x - qt * radix[p]];
                        x = qt;
                    }
                    s0 += __ldg(h + off);
                    s1 += __ldg(h + off + step);
                }
            }
            // segmented tree reduction: after offset o, lane j0 of a row holds the sum of its row's lanes [j0, j0 + 2o)
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t t0 = __shfl_down_sync(0xFFFFFFFFu, s0, o), t1 = __shfl_down_sync(0xFFFFFFFFu, s1, o);
                if (j0 + o < span) {
                    s0 += t0;
                    s1 += t1;
                }
            }
            if (mine && j0 == 0) {
                int64_t *o = out + ((int64_t)row * n_queries + qi) * 2;
                o[0] = (int64_t)s0;
                o[1] = (int64_t)s1;
            }
        }
    }
}

}  // namespace nmb

extern "C" {

int64_t nmb_sweep_hist_size(void) { return nmb::kSweepHistSize; }

int64_t nmb_sweep_bipartite_size(void) { return nmb::kBipHistSize; }

// One launch of sweep_hist_kernel; SweepParams says how contig_slot / the contig range select the counted contigs.
static int sweep_launch(bool bipartite, const nmb_assembly *a, const uint32_t *class_records_of_modtype,
                        int32_t tile_begin, int32_t tile_count, int32_t contig_begin, int32_t contig_end,
                        const int32_t *contig_slot, int32_t n_slots, uint32_t *hist, void *stream) {
    const char *what = bipartite ? "nmb_sweep_bipartite" : "nmb_sweep_hist";
    NMB_REQUIRE(a && class_records_of_modtype && hist, "%s: null argument", what);
    NMB_REQUIRE(contig_slot ? n_slots > 0 : n_slots == 1, "%s: bad slot map", what);
    NMB_REQUIRE(tile_begin >= 0 && tile_count >= 0 && tile_begin + tile_count <= a->n_tiles,
                "%s: tiles [%d, %d) outside the assembly", what, tile_begin, tile_begin + tile_count);
    if (tile_count == 0) return NMB_OK;
    nmb::SweepParams p{a->seq_records, a->nonacgt, class_records_of_modtype, a->contig_start, a->contig_len, hist,
                       contig_slot, tile_begin, a->n_tiles, contig_begin, contig_end, n_slots};
    if (bipartite)
        nmb::sweep_hist_kernel<true><<<tile_count, nmb::kTileChunks, 0, (cudaStream_t)stream>>>(p);
    else
        nmb::sweep_hist_kernel<false><<<tile_count, nmb::kTileChunks, 0, (cudaStream_t)stream>>>(p);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_hist(const nmb_assembly *a, const uint32_t *class_records_of_modtype, int32_t tile_begin,
                   int32_t tile_count, int32_t contig_begin, int32_t contig_end, const int32_t *contig_slot,
                   int32_t n_slots, uint32_t *hist, void *stream) {
    return sweep_launch(false, a, class_records_of_modtype, tile_begin, tile_count, contig_begin, contig_end,
                        contig_slot, n_slots, hist, stream);
}

int nmb_sweep_bipartite(const nmb_assembly *a, const uint32_t *class_records_of_modtype, int32_t tile_begin,
                        int32_t tile_count, int32_t contig_begin, int32_t contig_end, const int32_t *contig_slot,
                        int32_t n_slots, uint32_t *hist, void *stream) {
    return sweep_launch(true, a, class_records_of_modtype, tile_begin, tile_count, contig_begin, contig_end,
                        contig_slot, n_slots, hist, stream);
}

int nmb_sweep_finalize(uint32_t *hist, int32_t n_slots, void *stream) {
    NMB_REQUIRE(hist && n_slots > 0 && n_slots <= 65535, "nmb_sweep_finalize: bad argument");
    for (int k = nmb::kSweepMaxK - 1; k >= nmb::kSweepMinK; --k) {  // 8 -> 7, then 7 -> 6, ... each level complete first
        const int64_t n = (int64_t)k * 2 * nmb::pow5(k);
        const dim3 grid((unsigned)((n + 255) / 256), (unsigned)n_slots);
        nmb::sweep_marginalise_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(hist, k);
        NMB_CUDA(cudaGetLastError());
    }
    return NMB_OK;
}

int nmb_sweep_bipartite_finalize(uint32_t *hist, int32_t n_slots, void *stream) {
    NMB_REQUIRE(hist && n_slots > 0 && n_slots <= 65535, "nmb_sweep_bipartite_finalize: bad argument");
    auto run = [&](int g, int a, int b, int mode) {
        const int64_t n = (int64_t)(a + b) * 2 * (1ll << (2 * (a + b)));
        const dim3 grid((unsigned)((n + 255) / 256), (unsigned)n_slots);
        nmb::bip_marginalise_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(hist, g, a, b, mode);
    };
    for (int g = nmb::kBipMinGap; g <= nmb::kBipMaxGap; ++g) {
        run(g, 4, 3, 0);  // (4,g,3) from (4,g,4): last letter
        run(g, 3, 4, 1);  // (3,g,4) from (4,g,4): first letter
        run(g, 3, 3, 0);  // (3,g,3) from the now complete (3,g,4): last letter
        NMB_CUDA(cudaGetLastError());
    }
    return NMB_OK;
}

int nmb_sweep_slice(const uint32_t *src, int64_t src_slot_stride, int32_t n_slots, uint32_t *dst, int64_t n_out,
                    int64_t axis_stride, int32_t digit, void *stream) {
    NMB_REQUIRE(src && dst && n_out > 0 && axis_stride > 0 && digit >= 0 && digit < 5 && n_slots > 0 &&
                    n_slots <= 65535 && src_slot_stride >= 0,
                "nmb_sweep_slice: bad argument");
    const dim3 grid((unsigned)((n_out + 255) / 256), (unsigned)n_slots);
    nmb::sweep_slice_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, src_slot_stride, dst, n_out, axis_stride, digit);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

static uint32_t clamp_min_mod(int64_t min_mod) { return (uint32_t)(min_mod > 0xFFFFFFFFll ? 0xFFFFFFFFll : min_mod); }

// What the three candidate filters share before their launch: the checks of the filter and output arguments, *n_out
// zeroed, and *blocks = the grid for n entries (0: nothing to launch).
static int filter_begin(const char *what, int64_t min_mod, int32_t prune, nmb_sweep_hit *out, int64_t capacity,
                        int64_t *n_out, int64_t n, void *stream, unsigned *blocks) {
    NMB_REQUIRE(n_out && capacity >= 0 && min_mod >= 0 && (prune == 0 || prune == 1), "%s: bad argument", what);
    NMB_REQUIRE(capacity == 0 || out, "%s: null output", what);
    NMB_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int64_t), (cudaStream_t)stream));
    const int64_t grid = (n + 255) / 256;
    *blocks = (unsigned)(grid < 148 * 32 ? grid : 148 * 32);
    return NMB_OK;
}

int nmb_sweep_expand_filter(const uint32_t *n_mod, const uint32_t *n_nomod, int64_t n_slots, int64_t inner, int32_t k,
                            int32_t mod_pos, double min_mean, int64_t min_mod, int32_t prune, nmb_sweep_hit *out,
                            int64_t capacity, int64_t *n_out, void *stream) {
    NMB_REQUIRE(n_mod && n_nomod && n_slots >= 0 && k >= nmb::kSweepMinK && k <= nmb::kSweepMaxK && mod_pos >= 0 &&
                    mod_pos < k,
                "nmb_sweep_expand_filter: bad argument");
    int64_t want = 1;
    for (int i = 0; i < k - 2; ++i) want *= 15;
    NMB_REQUIRE(inner == want, "nmb_sweep_expand_filter: inner %lld is not 15^(k-2) for k = %d", (long long)inner, k);
    unsigned blocks;
    const int rc = filter_begin("nmb_sweep_expand_filter", min_mod, prune, out, capacity, n_out, n_slots * inner,
                                stream, &blocks);
    if (rc != NMB_OK || blocks == 0) return rc;
    // the first motif letter is the expanded (most significant) axis unless it is the modified position; the last one
    // is the least significant digit of r unless it is the modified position
    (prune ? nmb::expand_filter_kernel<5, true> : nmb::expand_filter_kernel<5, false>)<<<blocks, 256, 0,
                                                                                        (cudaStream_t)stream>>>(
        n_mod, n_nomod, n_slots, inner, mod_pos != 0, mod_pos != k - 1, min_mean, clamp_min_mod(min_mod), out, capacity,
        (unsigned long long *)n_out);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_bipartite_filter(const uint32_t *hist, int32_t n_slots, int32_t canonical, double min_mean,
                               int64_t min_mod, int32_t prune, nmb_sweep_hit *out, int64_t capacity, int64_t *n_out,
                               void *stream) {
    NMB_REQUIRE(hist && n_slots >= 0 && canonical >= 0 && canonical < 4, "nmb_sweep_bipartite_filter: bad argument");
    unsigned blocks;
    const int rc = filter_begin("nmb_sweep_bipartite_filter", min_mod, prune, out, capacity, n_out,
                                (int64_t)n_slots * nmb::kBipHistSize, stream, &blocks);
    if (rc != NMB_OK || blocks == 0) return rc;
    (prune ? nmb::bip_filter_kernel<true> : nmb::bip_filter_kernel<false>)<<<blocks, 256, 0, (cudaStream_t)stream>>>(
        hist, n_slots, canonical, min_mean, clamp_min_mod(min_mod), out, capacity, (unsigned long long *)n_out);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_bip_iupac_slice(const uint32_t *hist, int32_t n_slots, int32_t a, int32_t g, int32_t b, int32_t mod_pos,
                              int32_t cls, int32_t canonical, uint32_t *dst, void *stream) {
    NMB_REQUIRE((a == 3 || a == 4) && (b == 3 || b == 4) && g >= nmb::kBipMinGap && g <= nmb::kBipMaxGap,
                "nmb_sweep_bip_iupac_slice: shape (%d, %d, %d) is not X{3,4} N{4..8} Y{3,4}", a, g, b);
    NMB_REQUIRE(mod_pos >= 0 && mod_pos < a + g + b && !(mod_pos >= a && mod_pos < a + g),
                "nmb_sweep_bip_iupac_slice: modified position %d outside the halves", mod_pos);
    NMB_REQUIRE(hist && dst && n_slots > 0 && n_slots <= 65535 && (cls == 0 || cls == 1) && canonical >= 0 &&
                    canonical < 4,
                "nmb_sweep_bip_iupac_slice: bad argument");
    const int n_out = 1 << (2 * (a + b - 1));
    const dim3 grid((unsigned)((n_out + 255) / 256), (unsigned)n_slots);
    nmb::bip_iupac_slice_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
        hist, nmb::bip_offset(a, g, b), a, b, mod_pos < a ? mod_pos : mod_pos - g, cls, canonical, dst);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_bip_iupac_expand(const uint32_t *src, uint32_t *dst, int64_t outer, int64_t inner, void *stream) {
    NMB_REQUIRE(src && dst && outer > 0 && inner > 0, "nmb_sweep_bip_iupac_expand: bad argument");
    int64_t blocks = (outer * inner + 255) / 256;
    if (blocks > 148 * 64) blocks = 148 * 64;
    nmb::bip_iupac_expand_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(src, dst, outer, inner);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_bip_iupac_expand_filter(const uint32_t *n_mod, const uint32_t *n_nomod, int64_t n_slots, int64_t inner,
                                      double min_mean, int64_t min_mod, int32_t prune, nmb_sweep_hit *out,
                                      int64_t capacity, int64_t *n_out, void *stream) {
    NMB_REQUIRE(n_mod && n_nomod && n_slots >= 0 && inner > 0 && inner <= 0xFFFFFFFFll / 14,
                "nmb_sweep_bip_iupac_expand_filter: bad argument");
    int64_t p = 1;
    while (p < inner) p *= 14;
    NMB_REQUIRE(p == inner, "nmb_sweep_bip_iupac_expand_filter: inner %lld is not a power of 14", (long long)inner);
    unsigned blocks;
    const int rc = filter_begin("nmb_sweep_bip_iupac_expand_filter", min_mod, prune, out, capacity, n_out,
                                n_slots * inner, stream, &blocks);
    if (rc != NMB_OK || blocks == 0) return rc;
    (prune ? nmb::expand_filter_kernel<4, true> : nmb::expand_filter_kernel<4, false>)<<<blocks, 256, 0,
                                                                                        (cudaStream_t)stream>>>(
        n_mod, n_nomod, n_slots, inner, false, false, min_mean, clamp_min_mod(min_mod), out, capacity,
        (unsigned long long *)n_out);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_lookup(const uint32_t *hist, const uint32_t *bip, const int32_t *slots, int32_t n_rows,
                     const nmb_sweep_query *queries, int64_t n_queries, int64_t *out, void *stream) {
    NMB_REQUIRE(hist && n_rows >= 0 && n_rows <= 65535 && n_queries >= 0 && n_queries <= ((int64_t)1 << 40),
                "nmb_sweep_lookup: bad argument");
    NMB_REQUIRE(n_queries == 0 || queries, "nmb_sweep_lookup: null queries");
    NMB_REQUIRE(n_rows == 0 || n_queries == 0 || out, "nmb_sweep_lookup: null output");
    if (n_rows == 0 || n_queries == 0) return NMB_OK;
    const int64_t items = n_queries * ((n_rows + nmb::kLookupRun - 1) / nmb::kLookupRun);
    int64_t blocks = (items + nmb::kLookupWarps - 1) / nmb::kLookupWarps;
    if (blocks > 148 * 64) blocks = 148 * 64;
    nmb::sweep_lookup_kernel<<<(unsigned)blocks, nmb::kLookupWarps * 32, 0, (cudaStream_t)stream>>>(
        hist, bip, slots, n_rows, queries, n_queries, out);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_prune_lattice(int32_t lattice, uint32_t *states, uint32_t *widen, uint32_t *narrow) {
    NMB_REQUIRE(lattice >= 0 && lattice < 3 && states && widen && narrow, "nmb_sweep_prune_lattice: bad argument");
    const nmb::PruneLattice &L = nmb::kPruneLattices[lattice];
    for (int i = 0; i < L.n; ++i) {
        states[i] = L.states[i];
        widen[i] = L.widen[i];
        narrow[i] = L.narrow[i];
    }
    return L.n;
}

int nmb_sweep_expand(const uint32_t *src, uint32_t *dst, int64_t outer, int64_t inner, void *stream) {
    NMB_REQUIRE(src && dst && outer > 0 && inner > 0, "nmb_sweep_expand: bad argument");
    int64_t blocks = (outer * inner + 255) / 256;
    if (blocks > 148 * 64) blocks = 148 * 64;
    nmb::sweep_expand_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(src, dst, outer, inner);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_sweep_filter(const uint32_t *n_mod, const uint32_t *n_nomod, int64_t n, double min_mean, int64_t min_mod,
                     int64_t *out_index, int64_t capacity, int64_t *n_out, void *stream) {
    NMB_REQUIRE(n_mod && n_nomod && n_out && n >= 0 && capacity >= 0 && min_mod >= 0, "nmb_sweep_filter: bad argument");
    NMB_REQUIRE(capacity == 0 || out_index, "nmb_sweep_filter: null output");
    NMB_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int64_t), (cudaStream_t)stream));
    if (n == 0) return NMB_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    nmb::sweep_filter_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        n_mod, n_nomod, n, min_mean, clamp_min_mod(min_mod), out_index, capacity,
        (unsigned long long *)n_out);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

}  // extern "C"
