// K2 -- fused motif scan + gather-join + segmented reduce, and the motif compiler.
//
// Replaces, for a whole batch of (motif, contig-set) pairs in one launch:
//   utils.subseq_indices                      nanomotif/utils.py:44-67        (regex scan)
//   methylated_motif_occourances              nanomotif/find_motifs_bin.py:1234-1263 (np.isin join)
//   motif_model_contig (count step)           nanomotif/find_motifs_bin.py:1285-1331
//   motif_model_bin (sum over contigs)        nanomotif/find_motifs_bin.py:1265-1283
//
// Persistent CTAs draw work items (tile, block of <=32 motifs) from a device counter.  A tile is one
// self-contained 17 KB sequence record + one 32 KB class record, brought into shared memory by two
// cp.async.bulk (TMA) copies, each completing on its own mbarrier; the next item's sequence record is
// copied while the current item's motifs are evaluated.  Four CTAs of 128 threads are resident per
// SM, so the remaining copy latency is hidden by the other CTAs' bit-parallel evaluation.  Counts are popcounts of
// match & class-plane, reduced with warp REDUX, accumulated per CTA in shared memory and flushed
// with one 64-bit atomic per (motif, counter) per item.
#include "scan.cuh"

namespace nmb {

constexpr int kScanThreads = kTileChunks;                                       // 128
constexpr int kMaxMpi = NMB_MAX_MOTIFS_PER_ITEM;

// A SIBLING RUN is a maximal sequence (>= 2) of consecutive motifs of one work item's block that have the same len and
// mod_pos and the same allowed set at every position but one common position j -- the children of one search expansion
// (find_motifs_bin.py:1116-1145 adds one base at one position to the same parent).  The run is scored as ONE parent
// chain pair (a member with j made a wildcard, same len and mod_pos, so run_chain_pair's clip keeps exactly the members'
// starts, contig edges included) plus a four-base split: every parent occurrence is counted by the base it has at j.
// A member with set S at j counts the sum over S.  Exact wherever every in-contig position holds one of A, C, G, T, i.e.
// in all but the non-ACGT warps, which score the members one by one.
//
// Sibling word of motif i (written by the motif compiler; link = motif i against motif i - 1 in the motif array):
//   bits 0-5 j, bits 6-7 link (0 none, kSibSame identical, kSibDiff differ at j only, both sets there non-empty),
//   bits 8-11 motif i's set at j, bits 12-15 motif i-1's set at j.
// parents[i] is motif i with the position where it differs from motif i + 1 made a wildcard (when they are linked).
constexpr uint32_t kSibSame = 1, kSibDiff = 2;
static_assert(NMB_MAX_MOTIFS_PER_ITEM == 32, "one lane per motif of a block holds its sibling word");

struct ScanParams {
    const uint32_t *seq_records;
    const uint32_t *nonacgt;
    const uint32_t *cls;
    const Program *programs;
    const nmb_job *jobs;
    const int32_t *contig_group;
    const int64_t *contig_start, *contig_len;
    unsigned long long *out;
    int *counter;             // dynamic item scheduling: {next item, finished CTAs}, zero at launch and at exit; or null
    const uint32_t *sib;      // per motif: sibling word; or null (every motif scored on its own)
    const Program *parents;   // per motif: parent program towards the right neighbour
    int n_jobs, n_items, mpi, n_tiles;
};

struct ItemMeta {
    int job, tile, mblk, pad;
};

__device__ __forceinline__ ItemMeta decode_item(const ScanParams &p, int item) {
    int lo = 0, hi = p.n_jobs;  // largest j with item_offset[j] <= item
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(&p.jobs[mid].item_offset) <= item) lo = mid; else hi = mid;
    }
    const int local = item - __ldg(&p.jobs[lo].item_offset);
    const int nblk = (__ldg(&p.jobs[lo].motif_count) + p.mpi - 1) / p.mpi;
    ItemMeta m;
    m.job = lo;
    m.tile = __ldg(&p.jobs[lo].tile_begin) + local / nblk;  // tile-major: concurrent CTAs share a tile in L2
    m.mblk = local % nblk;
    m.pad = 0;
    return m;
}

__device__ __forceinline__ int group_of(const nmb_job &job, int contig, const int32_t *contig_group) {
    if (contig < job.contig_begin || contig >= job.contig_end) return -1;
    if (job.group_mode == 0) return 0;
    if (job.group_mode == 1) return contig - job.contig_begin;
    return __ldg(contig_group + contig);
}

// Run of siblings that starts at block lane `a` (warp-uniform), formed from the block's sibling words (lane l holds
// motif l's word, 0 past the block) with ballots: the lanes after `a` that are linked to their left neighbour, cut at
// the first one that differs at another position.  Identical motifs carry their neighbour's set along.
struct SibRun {
    int run;    // members; 1 = motif a scored on its own
    int first;  // first lane whose link differs at j: parents[first - 1] is the parent
    int j;      // the split position
    int set;    // this lane's allowed set at j (lanes of the run)
};

__device__ __forceinline__ SibRun sibling_run(uint32_t sw, int a) {
    SibRun r = {1, 0, 0, 0};
    const int lane = threadIdx.x & 31;
    const uint32_t link = (sw >> 6) & 3;
    const unsigned gt = ~((2u << a) - 1u);  // lanes after a
    const unsigned linked = __ballot_sync(0xFFFFFFFFu, link != 0) & gt;
    const unsigned diff = __ballot_sync(0xFFFFFFFFu, link == kSibDiff) & linked;
    const unsigned stop = ~linked & gt;
    unsigned span = stop ? gt & ((1u << (__ffs(stop) - 1)) - 1u) : gt;
    if (!(diff & span)) return r;  // nothing linked, or identical motifs only: no position to split at
    r.first = __ffs(diff & span) - 1;
    r.j = __shfl_sync(0xFFFFFFFFu, sw & 63, r.first);
    const unsigned bad = __ballot_sync(0xFFFFFFFFu, link == kSibDiff && (int)(sw & 63) != r.j) & span;
    if (bad) span &= (1u << (__ffs(bad) - 1)) - 1u;
    r.run = 1 + __popc(span);
    // up to the first differing link a member has that link's left set at j, after it the set of its last one
    const unsigned upto = diff & span & ((2u << lane) - 1u);
    const uint32_t ws = __shfl_sync(0xFFFFFFFFu, sw, upto ? 31 - __clz(upto) : r.first);
    r.set = (ws >> (upto ? 8 : 12)) & 0xF;
    return r;
}

// Word k of a sequence plane seen o positions to the right (0 <= o < 32 * H): bit b = plane[32 k + b + o].
template <int H>
__device__ __forceinline__ uint32_t plane_right(const uint32_t (&w)[NW + 2 * H], int k, int o) {
    if (H == 1 || o < 32) return __funnelshift_r(w[k + H], w[k + H + 1], o);
    return __funnelshift_r(w[k + H + 1], w[k + H + 2], o);
}
// ... o positions to the left (0 <= o < 32 * H): bit b = plane[32 k + b - o] (the clamped shift of 32 is the word itself).
template <int H>
__device__ __forceinline__ uint32_t plane_left(const uint32_t (&w)[NW + 2 * H], int k, int o) {
    if (H == 1 || o <= 32) return __funnelshift_rc(w[k + H - 1], w[k + H], 32 - o);
    return __funnelshift_rc(w[k + H - 2], w[k + H - 1], 64 - o);
}

// Popcounts of P, P & x, P & y, P & x & y: by inclusion-exclusion the occurrences in P with each base (x, y) at j.
__device__ __forceinline__ void tally(uint32_t pw, uint32_t xs, uint32_t ys, uint32_t *t) {
    t[0] += __popc(pw);
    t[1] += __popc(pw & xs);
    t[2] += __popc(pw & ys);
    t[3] += __popc(lop3<0x80>(pw, xs, ys));
}

// Four-base split of a parent's finished chains: for each of the four counters (n_mod / n_nomod per strand) the number
// of the lane's parent occurrences with A, T, G, C at the split position, delta = j - mod_pos positions from the
// modified base on the forward strand and -delta on the reverse strand (the reverse-complement occurrence sees the
// complementary base there).  base[col][b]: b = set bit (A, T, G, C), forward coordinates.
template <int H>
__device__ __forceinline__ void split_counts(const LaneSeq<H, false> &q, const uint32_t (&c)[NW + 2 * H],
                                             const uint32_t (&d)[NW + 2 * H], int sh, bool far, int delta,
                                             const uint32_t *cl, uint32_t (&base)[4][4]) {
    // the strand that looks right (delta >= 0: forward) and the one that looks left, so that one pair of windows
    // serves both signs of delta
    const bool neg = delta < 0;
    const int o = neg ? -delta : delta;
    const uint32_t *cr = neg ? cl + 2 * kTileWords : cl, *cf = neg ? cl : cl + 2 * kTileWords;
    uint32_t t[4][4] = {};  // [right mod, right nomod, left mod, left nomod][all, x, y, xy]
#pragma unroll
    for (int h = 0; h < NW; h += 4) {
        const uint4 r0 = *reinterpret_cast<const uint4 *>(cr + (h >> 2) * kSlotStride);
        const uint4 r1 = *reinterpret_cast<const uint4 *>(cr + kTileWords + (h >> 2) * kSlotStride);
        const uint4 l0 = *reinterpret_cast<const uint4 *>(cf + (h >> 2) * kSlotStride);
        const uint4 l1 = *reinterpret_cast<const uint4 *>(cf + kTileWords + (h >> 2) * kSlotStride);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t mf = aligned_word<H>(c, h + k, sh, far);
            const uint32_t mr = aligned_word_rc<H>(d, h + k, sh, far);
            const uint32_t mR = neg ? mr : mf, mL = neg ? mf : mr;
            const uint32_t xr = plane_right<H>(q.x, h + k, o), yr = plane_right<H>(q.y, h + k, o);
            const uint32_t xl = plane_left<H>(q.x, h + k, o), yl = plane_left<H>(q.y, h + k, o);
            const uint32_t w0 = k == 0 ? r0.x : k == 1 ? r0.y : k == 2 ? r0.z : r0.w;
            const uint32_t w1 = k == 0 ? r1.x : k == 1 ? r1.y : k == 2 ? r1.z : r1.w;
            const uint32_t w2 = k == 0 ? l0.x : k == 1 ? l0.y : k == 2 ? l0.z : l0.w;
            const uint32_t w3 = k == 0 ? l1.x : k == 1 ? l1.y : k == 2 ? l1.z : l1.w;
            tally(mR & w0, xr, yr, t[0]);
            tally(mR & w1, xr, yr, t[1]);
            tally(mL & w2, xl, yl, t[2]);
            tally(mL & w3, xl, yl, t[3]);
        }
    }
#pragma unroll
    for (int col = 0; col < 4; ++col) {
        uint32_t u[4];  // right = forward unless delta < 0
#pragma unroll
        for (int e = 0; e < 4; ++e) u[e] = neg ? t[col ^ 2][e] : t[col][e];
        base[col][0] = u[0] - u[1] - u[2] + u[3];               // A = (0, 0)
        base[col][1] = u[2] - u[3];                             // T = (0, 1)
        base[col][2] = u[1] - u[3];                             // G = (1, 0)
        base[col][3] = u[3];                                    // C = (1, 1)
    }
}

__device__ __forceinline__ uint32_t sum_over_set(const uint32_t (&b)[4], int s) {
    return ((s & 1) ? b[0] : 0u) + ((s & 2) ? b[1] : 0u) + ((s & 4) ? b[2] : 0u) + ((s & 8) ? b[3] : 0u);
}

// Evaluate the item's motifs on this lane's chunk and accumulate the four counters.
template <int H, bool PLANES>
__device__ __forceinline__ void score_motifs(const ScanParams &p, const nmb_job &job, const ItemMeta &meta,
                                             const LaneSeq<H, PLANES> &q, const LaneEdge &edge, const uint32_t *cl,
                                             bool valid,
                                             bool uniform, unsigned peers, bool leader, int g, int primary,
                                             uint32_t (*acc)[4]) {
    const int m_begin = job.motif_begin + meta.mblk * p.mpi;
    const int m_count = min(p.mpi, job.motif_count - meta.mblk * p.mpi);
    // sibling words of the whole block in ONE coalesced load (lane l holds motif l's word; kMaxMpi == 32): the runs
    // are formed with ballots and shuffles below, so no motif waits for a dependent global load before its program
    // can be fetched.  Warps with a non-ACGT letter in reach score every motif on its own.
    const bool siblings = !PLANES && p.sib != nullptr;  // warp-uniform
    uint32_t sw = 0;
    if (siblings && (int)(threadIdx.x & 31) < m_count) sw = __ldg(p.sib + m_begin + (threadIdx.x & 31));

    // per-lane counts of one motif -> warp sums -> the CTA's accumulators / the output
    auto flush = [&](int mi, uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) {
        // n_mod | n_nomod << 16 per strand (per-lane counts are <= 512)
        uint32_t pk_f = valid ? (c0 | (c1 << 16)) : 0u;
        uint32_t pk_r = valid ? (c2 | (c3 << 16)) : 0u;
        const long long row = job.out_base + (long long)(meta.mblk * p.mpi + mi) * job.n_groups;
        // two 16-bit fields per word survive a 32-lane sum (<= 8192)
        if (uniform) {  // all counted lanes of the warp feed the same output row (the common case)
            pk_f = __reduce_add_sync(0xFFFFFFFFu, pk_f);
            pk_r = __reduce_add_sync(0xFFFFFFFFu, pk_r);
        } else {  // contig / group boundary inside the warp: segmented sums over equal-group lanes
            pk_f = __reduce_add_sync(peers, pk_f);
            pk_r = __reduce_add_sync(peers, pk_r);
        }
        if (leader && (pk_f | pk_r)) {
            const uint32_t v[4] = {pk_f & 0xFFFFu, pk_f >> 16, pk_r & 0xFFFFu, pk_r >> 16};
            if (g == primary) {
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (v[c]) atomicAdd(&acc[mi][c], v[c]);
            } else {
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (v[c]) atomicAdd(p.out + (row + g) * 4 + c, (unsigned long long)v[c]);
            }
        }
    };

    int mi = 0;
#pragma unroll 1
    while (mi < m_count) {
        SibRun sr = {1, 0, 0, 0};
        if (siblings) sr = sibling_run(sw, mi);
        // ONE program serves both strands (scan.cuh: run_chain_pair) -- the motif's own, or the run's parent
        const ProgramView pv = load_program(sr.run > 1 ? p.parents + (m_begin + sr.first - 1)
                                                       : p.programs + (size_t)(m_begin + mi) * 2);
        uint32_t c[NW + 2 * H], d[NW + 2 * H];
        if (run_chain_pair<H, PLANES>(pv, q, c, d, edge)) {  // else: no occurrence in this warp's chunks
            const bool far = pv.mod_pos >= 32;  // only possible when H == 2
            const int sh = pv.mod_pos & 31;
            if constexpr (!PLANES) {
                if (sr.run > 1) {
                    uint32_t base[4][4];
                    split_counts<H>(q, c, d, sh, far, sr.j - pv.mod_pos, cl, base);
#pragma unroll 1
                    for (int k = 0; k < sr.run; ++k) {
                        const int s = __shfl_sync(0xFFFFFFFFu, sr.set, mi + k);
                        flush(mi + k, sum_over_set(base[0], s), sum_over_set(base[1], s),
                              sum_over_set(base[2], comp_set(s)), sum_over_set(base[3], comp_set(s)));
                    }
                    mi += sr.run;
                    continue;
                }
            }
            uint32_t cnt[4] = {0, 0, 0, 0};  // n_mod '+', n_nomod '+', n_mod '-', n_nomod '-'
#pragma unroll
            for (int h = 0; h < NW; h += 4) {
                uint4 pl[4];
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    pl[k] = *reinterpret_cast<const uint4 *>(cl + k * kTileWords + (h >> 2) * kSlotStride);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t mf = aligned_word<H>(c, h + k, sh, far);
                    const uint32_t mr = aligned_word_rc<H>(d, h + k, sh, far);
                    const uint32_t w0 = k == 0 ? pl[0].x : k == 1 ? pl[0].y : k == 2 ? pl[0].z : pl[0].w;
                    const uint32_t w1 = k == 0 ? pl[1].x : k == 1 ? pl[1].y : k == 2 ? pl[1].z : pl[1].w;
                    const uint32_t w2 = k == 0 ? pl[2].x : k == 1 ? pl[2].y : k == 2 ? pl[2].z : pl[2].w;
                    const uint32_t w3 = k == 0 ? pl[3].x : k == 1 ? pl[3].y : k == 2 ? pl[3].z : pl[3].w;
                    cnt[0] += __popc(mf & w0);  // occurrences whose modified base is methylated, '+'
                    cnt[1] += __popc(mf & w1);  // ... unmethylated, '+'
                    cnt[2] += __popc(mr & w2);  // reverse-complement occurrences, '-' strand rows
                    cnt[3] += __popc(mr & w3);
                }
            }
            flush(mi, cnt[0], cnt[1], cnt[2], cnt[3]);
        }
        mi += sr.run;
    }
}

// One tile (sequence record + class record = 49.7 KB) per CTA in shared memory; four CTAs of four warps are resident
// per SM, so while one CTA waits for its bulk copies the other three keep the ALUs busy.  (Measured alternatives on
// B200: a 2-stage ring with two resident CTAs, and a split ring with three, were both slower -- profiles/r01_notes.md.)
constexpr int kScanSmemBytes = kSeqRecBytes + kClsRecBytes;

__device__ __forceinline__ void bar_sync_1(int n_threads) { asm volatile("bar.sync 1, %0;" ::"r"(n_threads) : "memory"); }

// The two records of a tile arrive on SEPARATE mbarriers.  The lanes copy their sequence words into registers at the
// start of an item, after which the sequence half of the buffer is dead: the next item's index is decoded and its
// sequence record is already on its way while this item's motifs are evaluated; only the class record (2/3 of the
// bytes) has to wait for the end of the item.  ncu's source view had 19 % of all warp samples on the mbarrier spin in
// front of a tile (profiles/r02_notes.md).
template <int H, int STAGES>
__global__ void __launch_bounds__(kScanThreads, 4) scan_count_kernel(const ScanParams p) {
    static_assert(STAGES == 1, "one tile buffer per CTA");
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t seq_bar, cls_bar;
    __shared__ ItemMeta s_meta[2];
    __shared__ uint32_t s_acc[2][kMaxMpi][4];

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    if (tid == 0) {
        mbar_init(&seq_bar, 1);
        mbar_init(&cls_bar, 1);
        fence_barrier_init();
    }
    for (int i = tid; i < 2 * kMaxMpi * 4; i += kScanThreads) (&s_acc[0][0][0])[i] = 0;
    __syncthreads();

    // Items are handed out through a global counter when the caller provides one: a CTA that drew cheap items (3
    // instead of 4 motifs, dead chains) simply takes more of them, so the launch ends when the WORK runs out, not
    // when the unluckiest CTA of a static round-robin finishes.  Items still start in tile-major order.  The index
    // of the next item is drawn as soon as the previous draw has been used, so the atomic's round trip is hidden.
    const bool dynamic = p.counter != nullptr;
    int next_item = 0, n_drawn = 0;  // thread 0 only
    auto draw = [&]() {
        next_item = dynamic ? atomicAdd(p.counter, 1) : (int)blockIdx.x + n_drawn * (int)gridDim.x;
        ++n_drawn;
    };
    // thread 0: decode the drawn item into s_meta[slot] and start the copy of its sequence record; an exhausted
    // work list is signalled through an empty phase of the sequence barrier
    auto issue_seq = [&](int slot) {
        const int item = next_item;
        if (item >= p.n_items) {
            s_meta[slot].job = -1;
            mbar_arrive(&seq_bar);
            return;
        }
        const ItemMeta m = decode_item(p, item);
        s_meta[slot] = m;
        fence_proxy_async();  // order the earlier generic reads of this buffer before the async writes
        mbar_expect_tx(&seq_bar, kSeqRecBytes);
        bulk_g2s(smem, p.seq_records + (size_t)m.tile * kSeqRecWords, kSeqRecBytes, &seq_bar);
        draw();
    };
    auto issue_cls = [&](int slot) {
        const ItemMeta m = s_meta[slot];
        if (m.job < 0) return;
        const int modtype = __ldg(&p.jobs[m.job].modtype);
        fence_proxy_async();
        mbar_expect_tx(&cls_bar, kClsRecBytes);
        bulk_g2s(smem + kSeqRecBytes, p.cls + ((size_t)modtype * p.n_tiles + m.tile) * kClsRecWords, kClsRecBytes, &cls_bar);
    };
    if (tid == 0) {
        draw();
        issue_seq(0);
        issue_cls(0);
    }

    const uint32_t *sx = reinterpret_cast<const uint32_t *>(smem);
    const uint32_t *sy = sx + kSeqPlaneWords;
    const int32_t *sinfo = reinterpret_cast<const int32_t *>(sy + kSeqPlaneWords);
    const uint32_t *scls = sx + kSeqRecWords;
    for (int k = 0;; ++k) {
        const int par = k & 1;
        mbar_wait(&seq_bar, (uint32_t)par);
        const ItemMeta meta = s_meta[par];
        if (meta.job < 0) break;  // CTA-uniform: every thread reads the same word
        const nmb_job job = p.jobs[meta.job];

        const int info = sinfo[tid];
        const int contig = info < 0 ? -1 : (info & kChunkIdMask);
        const int g = contig < 0 ? -1 : group_of(job, contig, p.contig_group);
        const bool valid = g >= 0;
        // group whose counts go through the CTA's shared accumulators: the one of the tile's first chunk
        const int info0 = sinfo[0];
        const int primary = info0 < 0 ? -1 : group_of(job, info0 & kChunkIdMask, p.contig_group);

        const unsigned vmask = __ballot_sync(0xFFFFFFFFu, valid);
        // lanes that are not counted (padding, contigs outside the job) contribute zeros, so the warp
        // is uniform when all COUNTED lanes share one group
        const int first = vmask ? __ffs(vmask) - 1 : 0;
        const int g0 = __shfl_sync(0xFFFFFFFFu, g, first);
        const bool uniform = __all_sync(0xFFFFFFFFu, !valid || g == g0);
        unsigned peers = 0xFFFFFFFFu;
        bool leader = lane == first;
        if (!uniform) {
            peers = __match_any_sync(0xFFFFFFFFu, g);
            leader = valid && lane == __ffs(peers) - 1;
        }
        // matcher variant (scan.cuh): non-ACGT letters of a contig in reach -> full test at every step
        // (rare); inter-contig padding in reach -> plain steps, finished chains clipped to the contig
        const bool warp_n = __any_sync(0xFFFFFFFFu, valid && (info & kChunkFlagN));
        const bool warp_edge = __any_sync(0xFFFFFFFFu, valid && (info & kChunkFlagEdge));
        const uint32_t *cl = scls + tid * 4;  // lane-interleaved planes: vector v at cl + v * kSlotStride

        // after this point nobody reads the sequence half of the buffer any more
        auto seq_done_prefetch_next = [&]() {
            bar_sync_1(kScanThreads);
            if (tid == 0) issue_seq(par ^ 1);
            mbar_wait(&cls_bar, (uint32_t)par);
        };
        if (!vmask) {
            seq_done_prefetch_next();
        } else if (warp_n) {
            LaneSeq<H, true> q;
            load_xyn<H>(sx, sy, tid, p.nonacgt + kHalo + (size_t)meta.tile * kTileWords + tid * NW - H, q);
            seq_done_prefetch_next();
            const LaneEdge edge = {0, false, false};
            score_motifs<H, true>(p, job, meta, q, edge, cl, valid, uniform, peers, leader, g, primary, s_acc[par]);
        } else {
            LaneSeq<H, false> q;
            load_xy<H>(sx, sy, tid, q);
            seq_done_prefetch_next();
            const LaneEdge edge = lane_edge(warp_edge, info, (int64_t)meta.tile * kTileChunks + tid,
                                            p.contig_start, p.contig_len);
            score_motifs<H, false>(p, job, meta, q, edge, cl, valid, uniform, peers, leader, g, primary, s_acc[par]);
        }
        __syncthreads();  // everyone is done with the class record and with s_acc[par]
        if (tid == 0) issue_cls(par ^ 1);
        if (tid < kMaxMpi * 4) {
            const int mi = tid >> 2, c = tid & 3;
            const uint32_t v = s_acc[par][mi][c];
            if (v) {
                s_acc[par][mi][c] = 0;
                const long long row =
                    job.out_base + (long long)(meta.mblk * p.mpi + mi) * job.n_groups + primary;
                atomicAdd(p.out + row * 4 + c, (unsigned long long)v);
            }
        }
    }
    // every CTA has drawn its last (empty) item before it gets here: the last one to leave re-arms the counter
    if (dynamic && tid == 0 && atomicAdd(p.counter + 1, 1) == (int)gridDim.x - 1) {
        p.counter[0] = 0;
        p.counter[1] = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// motif compiler: nmb_motif -> forward and reverse-complement Programs
// ---------------------------------------------------------------------------------------------
// Program of a motif strand given as allowed-sets per position (0xF = wildcard) in reading order.
// Gaps of 32 or more positions become "shift one word" pseudo entries so that every real entry carries a shift < 32.
// The first processed entry is the last motif position (shift 0); a stripped motif starts with a constrained position,
// so the chain ends aligned at position 0.
__device__ void build_program(const uint8_t *allowed, int len, int mp, Program &pr) {
    for (int i = 0; i < kMaxLen; ++i) pr.ent[i] = 0;
    pr.reserved = 0;
    int n = 0, prev = -1;
    for (int j = len - 1; j >= 0; --j) {
        const int a = allowed[j] & 0xF;
        if (a == 0xF && j != 0) continue;
        int d = prev < 0 ? 0 : prev - j;
        for (; d >= 32 && n < kMaxLen - 1; d -= 32) pr.ent[n++] = kEntShift32;
        if (n < kMaxLen) pr.ent[n++] = (uint16_t)(a | (d << 8));  // a == 0xF at j == 0: pure shift
        prev = j;
    }
    pr.n = (uint8_t)n; pr.mod_pos = (uint8_t)mp; pr.len = (uint8_t)len;
}

__device__ __forceinline__ bool motif_ok(const nmb_motif &m) { return m.len >= 1 && m.len <= kMaxLen && m.mod_pos < m.len; }

// Link of motif b to its left neighbour a (sibling word layout above; 0 = not siblings): same len and mod_pos, the same
// allowed set at every position but at most one, and there both sets non-empty.
__device__ uint32_t sibling_link(const nmb_motif &a, const nmb_motif &b) {
    if (!motif_ok(a) || !motif_ok(b) || a.len != b.len || a.mod_pos != b.mod_pos) return 0;
    int j = -1;
    for (int i = 0; i < a.len; ++i) {
        if ((a.allowed[i] & 0xF) == (b.allowed[i] & 0xF)) continue;
        if (j >= 0) return 0;
        j = i;
    }
    if (j < 0) return kSibSame << 6;
    const uint32_t sa = a.allowed[j] & 0xF, sb = b.allowed[j] & 0xF;
    if (!sa || !sb) return 0;
    return (uint32_t)j | kSibDiff << 6 | sb << 8 | sa << 12;
}

// Two threads per motif (forward and reverse-complement program); with `siblings`, the forward thread also writes the
// motif's sibling word and its parent program towards the right neighbour.
__global__ void compile_motifs_kernel(const nmb_motif *__restrict__ motifs, int n_motifs,
                                      Program *__restrict__ programs, uint32_t *__restrict__ siblings,
                                      Program *__restrict__ parents) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * n_motifs) return;
    const int m = t >> 1;
    const nmb_motif mt = motifs[m];
    const bool rc = t & 1;
    Program pr;
    int len = mt.len, mp = mt.mod_pos;
    if (siblings && !rc) {
        siblings[m] = m > 0 ? sibling_link(motifs[m - 1], mt) : 0u;
        const uint32_t right = m + 1 < n_motifs ? sibling_link(mt, motifs[m + 1]) : 0u;
        if (((right >> 6) & 3) == kSibDiff) {
            uint8_t allowed[kMaxLen];
            for (int j = 0; j < len; ++j) allowed[j] = mt.allowed[j] & 0xF;
            allowed[right & 63] = 0xF;
            build_program(allowed, len, mp, pr);
            parents[m] = pr;
        }
    }
    if (!motif_ok(mt)) {  // invalid: compile to "never matches"
        for (int i = 0; i < kMaxLen; ++i) pr.ent[i] = 0;
        pr.reserved = 0;
        pr.n = 1; pr.mod_pos = 0; pr.len = 1;
        programs[t] = pr;
        return;
    }
    uint8_t allowed[kMaxLen];
    for (int j = 0; j < len; ++j) {
        int a = mt.allowed[rc ? (len - 1 - j) : j] & 0xF;
        if (rc) a = ((a & 5) << 1) | ((a & 10) >> 1);  // A<->T, G<->C (constants.py:14-20)
        allowed[j] = (uint8_t)a;
    }
    if (rc) mp = len - 1 - mp;  // motif.py:264
    build_program(allowed, len, mp, pr);
    programs[t] = pr;
}

}  // namespace nmb

extern "C" {

static int compile_impl(const nmb_motif *motifs, int32_t n_motifs, void *programs, void *siblings, void *stream) {
    NMB_REQUIRE(n_motifs >= 0, "nmb_compile_motifs: n_motifs=%d", n_motifs);
    if (n_motifs == 0) return NMB_OK;
    NMB_REQUIRE(motifs && programs, "nmb_compile_motifs: null argument");
    nmb::Program *parents =
        siblings ? (nmb::Program *)((uint8_t *)siblings + ((n_motifs * (int64_t)sizeof(uint32_t) + 127) / 128) * 128)
                 : nullptr;
    nmb::compile_motifs_kernel<<<(2 * n_motifs + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        motifs, n_motifs, (nmb::Program *)programs, (uint32_t *)siblings, parents);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_compile_motifs(const nmb_motif *motifs, int32_t n_motifs, void *programs, void *stream) {
    return compile_impl(motifs, n_motifs, programs, nullptr, stream);
}

int64_t nmb_sibling_bytes(int32_t n_motifs) {
    const int64_t n = n_motifs > 0 ? n_motifs : 0;
    return ((n * (int64_t)sizeof(uint32_t) + 127) / 128) * 128 + n * (int64_t)sizeof(nmb::Program);
}

int nmb_compile_motifs_siblings(const nmb_motif *motifs, int32_t n_motifs, void *programs, void *siblings,
                                void *stream) {
    NMB_REQUIRE(siblings || n_motifs == 0, "nmb_compile_motifs_siblings: null siblings");
    return compile_impl(motifs, n_motifs, programs, siblings, stream);
}

static int scan_count_impl(const nmb_assembly *a, const uint32_t *class_records, const void *programs,
                           const nmb_job *jobs, int32_t n_jobs, int32_t n_items, int32_t motifs_per_item,
                           int32_t max_motif_len, const int32_t *contig_group, int64_t *out, int32_t grid_ctas,
                           const void *siblings, int32_t n_motifs, int32_t *work_counter, void *stream);

int nmb_scan_count(const nmb_assembly *a, const uint32_t *class_records, const void *programs,
                   const nmb_job *jobs, int32_t n_jobs, int32_t n_items, int32_t motifs_per_item,
                   int32_t max_motif_len, const int32_t *contig_group, int64_t *out,
                   int32_t grid_ctas, void *stream) {
    return scan_count_impl(a, class_records, programs, jobs, n_jobs, n_items, motifs_per_item, max_motif_len,
                           contig_group, out, grid_ctas, nullptr, 0, nullptr, stream);
}

int nmb_scan_count_balanced(const nmb_assembly *a, const uint32_t *class_records, const void *programs,
                            const nmb_job *jobs, int32_t n_jobs, int32_t n_items, int32_t motifs_per_item,
                            int32_t max_motif_len, const int32_t *contig_group, int64_t *out, int32_t grid_ctas,
                            int32_t *work_counter, void *stream) {
    NMB_REQUIRE(work_counter, "nmb_scan_count_balanced: null work counter");
    return scan_count_impl(a, class_records, programs, jobs, n_jobs, n_items, motifs_per_item, max_motif_len,
                           contig_group, out, grid_ctas, nullptr, 0, work_counter, stream);
}

int nmb_scan_count_siblings(const nmb_assembly *a, const uint32_t *class_records, const void *programs,
                            const void *siblings, int32_t n_motifs, const nmb_job *jobs, int32_t n_jobs,
                            int32_t n_items, int32_t motifs_per_item, int32_t max_motif_len,
                            const int32_t *contig_group, int64_t *out, int32_t grid_ctas, int32_t *work_counter,
                            void *stream) {
    NMB_REQUIRE(siblings && n_motifs > 0, "nmb_scan_count_siblings: null argument");
    return scan_count_impl(a, class_records, programs, jobs, n_jobs, n_items, motifs_per_item, max_motif_len,
                           contig_group, out, grid_ctas, siblings, n_motifs, work_counter, stream);
}

static int scan_count_impl(const nmb_assembly *a, const uint32_t *class_records, const void *programs,
                           const nmb_job *jobs, int32_t n_jobs, int32_t n_items, int32_t motifs_per_item,
                           int32_t max_motif_len, const int32_t *contig_group, int64_t *out, int32_t grid_ctas,
                           const void *siblings, int32_t n_motifs, int32_t *work_counter, void *stream) {
    NMB_REQUIRE(a && class_records && programs && jobs && out, "nmb_scan_count: null argument");
    NMB_REQUIRE(n_jobs > 0 && n_items >= 0, "nmb_scan_count: n_jobs=%d n_items=%d", n_jobs, n_items);
    NMB_REQUIRE(motifs_per_item >= 1 && motifs_per_item <= NMB_MAX_MOTIFS_PER_ITEM,
                "nmb_scan_count: motifs_per_item=%d not in 1..%d", motifs_per_item,
                NMB_MAX_MOTIFS_PER_ITEM);
    NMB_REQUIRE(max_motif_len >= 1 && max_motif_len <= NMB_MAX_MOTIF_LEN,
                "nmb_scan_count: max_motif_len=%d not in 1..%d", max_motif_len, NMB_MAX_MOTIF_LEN);
    if (n_items == 0) return NMB_OK;
    nmb::ScanParams p;
    p.seq_records = a->seq_records;
    p.nonacgt = a->nonacgt;
    p.cls = class_records;
    p.programs = (const nmb::Program *)programs;
    p.jobs = jobs;
    p.contig_group = contig_group;
    p.contig_start = a->contig_start;
    p.contig_len = a->contig_len;
    p.out = (unsigned long long *)out;
    p.n_jobs = n_jobs;
    p.n_items = n_items;
    p.mpi = motifs_per_item;
    p.n_tiles = a->n_tiles;
    p.counter = work_counter;
    p.sib = siblings ? (const uint32_t *)siblings : nullptr;
    p.parents = siblings ? (const nmb::Program *)((const uint8_t *)siblings +
                                                  ((n_motifs * (int64_t)sizeof(uint32_t) + 127) / 128) * 128)
                         : nullptr;

    int grid = grid_ctas;
    if (grid <= 0) {
        int sms = nmb_device_sm_count();
        if (sms < 0) return sms;
        grid = 4 * sms;  // resident CTAs per SM (49.7 KB of shared memory, <= 128 registers)
    }
    if (grid > n_items) grid = n_items;
    cudaStream_t s = (cudaStream_t)stream;
    const int smem_bytes = nmb::kScanSmemBytes;
#define NMB_LAUNCH_SCAN(H, S)                                                                                         \
    do {                                                                                                              \
        NMB_CUDA(cudaFuncSetAttribute(nmb::scan_count_kernel<H, S>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                      smem_bytes));                                                                   \
        nmb::scan_count_kernel<H, S><<<grid, nmb::kScanThreads, smem_bytes, s>>>(p);                                   \
    } while (0)
    if (max_motif_len <= 32) NMB_LAUNCH_SCAN(1, 1);  // one halo word covers a total shift (and a mod_pos) of at most 31
    else NMB_LAUNCH_SCAN(2, 1);
#undef NMB_LAUNCH_SCAN
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

}  // extern "C"
