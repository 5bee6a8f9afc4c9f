// K5 (tile-driven) -- contig x motif methylation-pattern table for MANY motifs per launch.
//
// The row-driven kernels of pattern.cu read every pileup row once per motif (~21 B per row and motif).
// Here the join runs the other way round, like K2: the pileup rows of one mod type that pass the
// read-coverage filters become two bit-planes per tile (valid '+', valid '-', lane-interleaved like the
// class planes) plus a rank directory (rows before each 32-bp word) and a (n_mod, n_valid_cov) payload
// array in (strand, position) order.  A persistent CTA brings a tile's sequence record and valid record
// into shared memory by TMA, evaluates a block of motifs with the K2 matcher (both strands per pass) and
// touches the payload only at the set bits of match & valid -- occurrences that have a pileup row --
// which are sparse.  Per (motif, contig): n_motif_obs, sum n_mod, sum n_valid_cov (phase 0) and, for the
// median, the per-occurrence fractions written into per-(motif, contig) segments (phase 1).
// Spec: DESIGN.md section 4 (K5); reference call site nanomotif/main.py:167-178.
#include "scan.cuh"

namespace nmb {

constexpr int kValidRecWords = 2 * kTileWords;                  // valid '+', valid '-'
constexpr int kValidRecBytes = kValidRecWords * 4;              // 16 KB
constexpr int kPatSmemBytes = kSeqRecBytes + kValidRecBytes + 2 * kChunkWords * kTileChunks * 2;  // 33.3 KB + 8 KB prefix counts
constexpr int kPatThreads = kTileChunks;

// ---- index build ------------------------------------------------------------------------------

struct RowFilter {
    const int32_t *contig_id;
    const int64_t *pos;
    const uint8_t *strand, *mod_type;  // mod_type may be null (all rows are of the wanted type)
    const int64_t *n_mod, *n_cov, *n_diff;
    int64_t n_rows;
    int want_modtype;
    int64_t min_cov;
    double min_fraction;
    const int64_t *contig_start, *contig_len;
    int n_contigs;
};

// Global position of row r when it takes part in the table, else -1 (spec: n_valid_cov >= min and
// n_valid_cov / (n_valid_cov + n_diff) >= min_fraction, compared in float64 like the oracle).
__device__ __forceinline__ int64_t row_gpos(const RowFilter &f, int64_t r) {
    if (f.mod_type && f.mod_type[r] != f.want_modtype) return -1;
    const int c = f.contig_id[r];
    if (c < 0 || c >= f.n_contigs || f.strand[r] > 1) return -1;
    const int64_t p = f.pos[r];
    if (p < 0 || p >= __ldg(f.contig_len + c)) return -1;
    const int64_t cov = f.n_cov[r], diff = f.n_diff[r];
    if (cov < f.min_cov || cov >= (1ll << 31) || f.n_mod[r] < 0 || f.n_mod[r] >= (1ll << 31)) return -1;
    if (!((double)cov / (double)(cov + diff) >= f.min_fraction)) return -1;  // NaN (0/0) fails like numpy
    return __ldg(f.contig_start + c) + p;
}

__global__ void __launch_bounds__(256) pattern_valid_kernel(const RowFilter f, uint32_t *__restrict__ valid) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < f.n_rows; r += stride) {
        const int64_t g = row_gpos(f, r);
        if (g < 0) continue;
        uint32_t *w = valid + (g >> 16) * kValidRecWords + (f.strand[r] ? kTileWords : 0) +
                      word_slot((int)((g >> 5) & (kTileWords - 1)));
        atomicOr(w, 1u << (g & 31));
    }
}

// valid word of flat index i = strand * n_words + tile * 2048 + natural word
__device__ __forceinline__ uint32_t valid_word(const uint32_t *__restrict__ valid, int64_t i, int64_t n_words) {
    const int strand = i >= n_words;
    const int64_t gw = i - (strand ? n_words : 0);
    return valid[(gw >> 11) * kValidRecWords + (strand ? kTileWords : 0) + word_slot((int)(gw & (kTileWords - 1)))];
}

constexpr int kRankWordsPerThread = 8;
constexpr int kRankBlockWords = 256 * kRankWordsPerThread;

__global__ void __launch_bounds__(256) pattern_rank_count_kernel(const uint32_t *__restrict__ valid, int64_t n_words,
                                                                 int64_t *__restrict__ block_counts) {
    __shared__ int s_warp[8];
    const int64_t i0 = ((int64_t)blockIdx.x * 256 + threadIdx.x) * kRankWordsPerThread;
    int c = 0;
    for (int k = 0; k < kRankWordsPerThread; ++k)
        if (i0 + k < 2 * n_words) c += __popc(valid_word(valid, i0 + k, n_words));
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int i = 0; i < 8; ++i) t += s_warp[i];
        block_counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(256) pattern_rank_write_kernel(const uint32_t *__restrict__ valid, int64_t n_words,
                                                                 const int64_t *__restrict__ block_offsets,
                                                                 uint32_t *__restrict__ rank_dir) {
    __shared__ int s_warp[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i0 = ((int64_t)blockIdx.x * 256 + threadIdx.x) * kRankWordsPerThread;
    int cnt[kRankWordsPerThread], c = 0;
    for (int k = 0; k < kRankWordsPerThread; ++k) {
        cnt[k] = i0 + k < 2 * n_words ? __popc(valid_word(valid, i0 + k, n_words)) : 0;
        c += cnt[k];
    }
    int incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int before = 0;
    for (int i = 0; i < warp; ++i) before += s_warp[i];
    int64_t run = block_offsets[blockIdx.x] + before + incl - c;
    for (int k = 0; k < kRankWordsPerThread; ++k) {
        if (i0 + k < 2 * n_words) rank_dir[i0 + k] = (uint32_t)run;
        run += cnt[k];
    }
}

__global__ void __launch_bounds__(256) pattern_payload_kernel(const RowFilter f, const uint32_t *__restrict__ valid,
                                                              const uint32_t *__restrict__ rank_dir, int64_t n_words,
                                                              int2 *__restrict__ payload) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < f.n_rows; r += stride) {
        const int64_t g = row_gpos(f, r);
        if (g < 0) continue;
        const int64_t i = (f.strand[r] ? n_words : 0) + (g >> 5);
        const uint32_t v = valid_word(valid, i, n_words);
        const int64_t row = (int64_t)rank_dir[i] + __popc(v & ((1u << (g & 31)) - 1u));
        payload[row] = make_int2((int)f.n_mod[r], (int)f.n_cov[r]);
    }
}

// ---- scan ---------------------------------------------------------------------------------------

struct PatParams {
    const uint32_t *seq_records, *nonacgt;
    const int64_t *contig_start, *contig_len;
    const uint32_t *valid, *rank_dir;
    const int2 *payload;
    const Program *programs;
    unsigned long long *stats;    // [n_motifs][n_contigs][3]
    const long long *offsets;     // [n_motifs * n_contigs + 1]   (phase 1)
    int *cursor;                  // [n_motifs * n_contigs]       (phase 1)
    double *fractions;            //                              (phase 1)
    int *counter;                 // dynamic item scheduling {next item, finished CTAs} (see scan.cu), or null
    int64_t n_words;
    int n_motifs, mpi, n_mblk, n_tiles, n_contigs, n_items, write;
};

// ---- warp hit queue ---------------------------------------------------------------------------
// Occurrences that have a pileup row ("hits") are found lane by lane, but fetching their payload lane by
// lane would leave one dependent load in flight per warp.  Instead every lane pushes its hits (payload row,
// contig, motif) into a per-warp queue in shared memory that lives across the motifs of a work item;
// whenever 32 are waiting the warp drains them together: 32 independent payload loads, then one masked
// warp reduction (REDUX) and one update per distinct (motif, contig) among them.
constexpr int kQueueLen = 64;
static_assert(NMB_MAX_MOTIFS_PER_ITEM == 32, "WarpQueue::acc is reset and flushed one motif per lane");

struct WarpQueue {
    uint32_t row[kQueueLen];
    int32_t contig[kQueueLen];
    uint8_t mi[kQueueLen];
    int n;                                                // entries waiting (warp-uniform)
    unsigned long long acc[NMB_MAX_MOTIFS_PER_ITEM][3];   // phase 0: counts of the warp's first contig, per motif
};

__device__ __forceinline__ unsigned long long redux_u64_of_u32(unsigned x) {  // sum over the warp, no overflow
    return (unsigned long long)__reduce_add_sync(0xFFFFFFFFu, x & 0xFFFFu) +
           ((unsigned long long)__reduce_add_sync(0xFFFFFFFFu, x >> 16) << 16);
}

// Drain the first n (<= 32) queue entries.  Phase 0: {obs, sum n_mod, sum n_valid_cov} per (motif, contig)
// -- into q.acc for the warp's first contig c0 (flushed once per work item), straight to global for the
// other contigs of a warp that straddles contigs.  Phase 1: the fractions go to their (motif, contig)
// segment; one cursor update per group, ranks inside the group give the slots.
__device__ __noinline__ void drain_hits(const PatParams *p, WarpQueue *q, int n, int m_begin, int c0) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    const bool on = lane < n;
    const int c = on ? q->contig[lane] : -1;
    const int mi = on ? q->mi[lane] : 0;
    int2 pl = make_int2(0, 0);
    if (on) pl = __ldg(p->payload + q->row[lane]);
    unsigned remaining = __ballot_sync(0xFFFFFFFFu, on);
    while (remaining) {  // one round per distinct (motif, contig); warp-uniform control flow
        const int src = __ffs(remaining) - 1;
        const int cl = __shfl_sync(0xFFFFFFFFu, c, src), ml = __shfl_sync(0xFFFFFFFFu, mi, src);
        const bool in = on && c == cl && mi == ml;
        const unsigned grp = __ballot_sync(0xFFFFFFFFu, in);
        remaining &= ~grp;
        const size_t seg = (size_t)(m_begin + ml) * p->n_contigs + cl;
        if (p->write) {
            int slot0 = 0;
            if (lane == src) slot0 = atomicAdd(p->cursor + seg, __popc(grp));
            slot0 = __shfl_sync(0xFFFFFFFFu, slot0, src);
            if (in) p->fractions[p->offsets[seg] + slot0 + __popc(grp & lt)] = (double)pl.x / (double)pl.y;
        } else {
            const unsigned long long sm = redux_u64_of_u32(in ? (unsigned)pl.x : 0u);
            const unsigned long long sc = redux_u64_of_u32(in ? (unsigned)pl.y : 0u);
            if (lane == src) {
                const unsigned long long cnt = __popc(grp);
                if (cl == c0) {  // only this warp touches q->acc, one lane per round
                    q->acc[ml][0] += cnt;
                    q->acc[ml][1] += sm;
                    q->acc[ml][2] += sc;
                } else {
                    unsigned long long *st = p->stats + seg * 3;
                    atomicAdd(st + 0, cnt);
                    atomicAdd(st + 1, sm);
                    atomicAdd(st + 2, sc);
                }
            }
        }
    }
    __syncwarp();
}

// Every lane pushes the set bits of `hits` (word-local occurrences with a valid row; v = the word of the
// valid plane, base = rows before the word); drains whenever 32 entries wait.
__device__ __noinline__ void push_hits(const PatParams *p, WarpQueue *q, uint32_t hits, uint32_t v, uint32_t base,
                                       int contig, int mi, int m_begin, int c0) {
    const int lane = threadIdx.x & 31;
    const unsigned lt = (1u << lane) - 1u;
    int qn = q->n;
    unsigned any = __ballot_sync(0xFFFFFFFFu, hits != 0);
    while (any) {  // every lane with hits left pushes one
        if (hits) {
            const int b = __ffs(hits) - 1;
            hits &= hits - 1;
            const int slot = qn + __popc(any & lt);
            q->row[slot] = base + __popc(v & ((1u << b) - 1u));
            q->contig[slot] = contig;
            q->mi[slot] = (uint8_t)mi;
        }
        qn += __popc(any);
        __syncwarp();
        if (qn >= 32) {
            drain_hits(p, q, 32, m_begin, c0);
            const int rest = qn - 32;  // <= 31: move the tail to the front
            uint32_t r = 0;
            int cc = 0, mm = 0;
            if (lane < rest) { r = q->row[32 + lane]; cc = q->contig[32 + lane]; mm = q->mi[32 + lane]; }
            __syncwarp();
            if (lane < rest) { q->row[lane] = r; q->contig[lane] = cc; q->mi[lane] = (uint8_t)mm; }
            __syncwarp();
            qn = rest;
        }
        any = __ballot_sync(0xFFFFFFFFu, hits != 0);
    }
    if (lane == 0) q->n = qn;
    __syncwarp();
}

// s_pref[(strand * NW + word) * 128 + chunk] = valid rows of the chunk's strand before that word (uint16)
template <int H, bool HASN>
__device__ __forceinline__ void pattern_motifs(const PatParams &p, int mblk, const LaneSeq<H, HASN> &q,
                                               const LaneEdge &edge, const uint32_t *sv, const uint16_t *s_pref,
                                               WarpQueue &wq, uint32_t rank_p, uint32_t rank_m, int contig, int c0) {
    const int tid = threadIdx.x, lane = tid & 31;
    const int m_begin = mblk * p.mpi;
    const int m_count = min(p.mpi, p.n_motifs - m_begin);
    wq.acc[lane][0] = wq.acc[lane][1] = wq.acc[lane][2] = 0;  // NMB_MAX_MOTIFS_PER_ITEM == 32 lanes
    if (lane == 0) wq.n = 0;
    __syncwarp();
#pragma unroll 1
    for (int mi = 0; mi < m_count; ++mi) {
        const ProgramView pv = load_program(p.programs + (size_t)(m_begin + mi) * 2);
        uint32_t c[NW + 2 * H], d[NW + 2 * H];
        if (!run_chain_pair<H, HASN>(pv, q, c, d, edge)) continue;
        const bool far = pv.mod_pos >= 32;
        const int sh = pv.mod_pos & 31;
        // occurrences WITH a pileup row, all 16 words of both strands first (the chains are dead after this): most
        // (warp, motif) pairs of a specific motif have none, and ONE vote then skips the whole push stage
        uint32_t hit0[NW], hit1[NW], any = 0;
#pragma unroll
        for (int h = 0; h < NW; h += 4) {
            const uint4 vp = *reinterpret_cast<const uint4 *>(sv + (h >> 2) * kSlotStride);
            const uint4 vm = *reinterpret_cast<const uint4 *>(sv + kTileWords + (h >> 2) * kSlotStride);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t v0 = k == 0 ? vp.x : k == 1 ? vp.y : k == 2 ? vp.z : vp.w;
                const uint32_t v1 = k == 0 ? vm.x : k == 1 ? vm.y : k == 2 ? vm.z : vm.w;
                hit0[h + k] = contig < 0 ? 0u : aligned_word<H>(c, h + k, sh, far) & v0;
                hit1[h + k] = contig < 0 ? 0u : aligned_word_rc<H>(d, h + k, sh, far) & v1;
                any |= hit0[h + k] | hit1[h + k];
            }
        }
        if (!__any_sync(0xFFFFFFFFu, any != 0)) continue;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            if (!__any_sync(0xFFFFFFFFu, (hit0[w] | hit1[w]) != 0)) continue;
            const uint32_t v0 = sv[(w >> 2) * kSlotStride + (w & 3)];
            const uint32_t v1 = sv[kTileWords + (w >> 2) * kSlotStride + (w & 3)];
            push_hits(&p, &wq, hit0[w], v0, rank_p + s_pref[w * kTileChunks + tid], contig, mi, m_begin, c0);
            push_hits(&p, &wq, hit1[w], v1, rank_m + s_pref[(NW + w) * kTileChunks + tid], contig, mi, m_begin, c0);
        }
    }
    if (wq.n) drain_hits(&p, &wq, wq.n, m_begin, c0);
    __syncwarp();
    if (!p.write && lane < m_count && wq.acc[lane][0]) {
        unsigned long long *st = p.stats + ((size_t)(m_begin + lane) * p.n_contigs + c0) * 3;
        atomicAdd(st + 0, wq.acc[lane][0]);
        atomicAdd(st + 1, wq.acc[lane][1]);
        atomicAdd(st + 2, wq.acc[lane][2]);
    }
    __syncwarp();
}

constexpr int kPrefBytes = 2 * NW * kTileChunks * 2;  // uint16 prefix counts: 8 KB

template <int H>
__global__ void __launch_bounds__(kPatThreads, 4) pattern_scan_kernel(const __grid_constant__ PatParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t full_bar;
    __shared__ WarpQueue s_queue[kPatThreads / 32];
    const int tid = threadIdx.x;
    __shared__ int s_item;
    if (tid == 0) {
        mbar_init(&full_bar, 1);
        fence_barrier_init();
    }
    __syncthreads();
    uint16_t *s_pref = reinterpret_cast<uint16_t *>(smem + kSeqRecBytes + kValidRecBytes);
    // items come from a device counter when the caller provides one (tiles differ in rows and hits: a static
    // round-robin ends with the unluckiest CTA), else blockIdx.x + k * gridDim.x
    for (int k = 0;; ++k) {
        if (tid == 0) {
            const int item = p.counter ? atomicAdd(p.counter, 1) : (int)blockIdx.x + k * (int)gridDim.x;
            s_item = item < p.n_items ? item : -1;
            if (item < p.n_items) {
                const int tile = item / p.n_mblk;
                fence_proxy_async();
                mbar_expect_tx(&full_bar, kSeqRecBytes + kValidRecBytes);
                bulk_g2s(smem, p.seq_records + (size_t)tile * kSeqRecWords, kSeqRecBytes, &full_bar);
                bulk_g2s(smem + kSeqRecBytes, p.valid + (size_t)tile * kValidRecWords, kValidRecBytes, &full_bar);
            } else {
                mbar_arrive(&full_bar);  // nothing left: wake the CTA with an empty phase
            }
        }
        mbar_wait(&full_bar, (uint32_t)(k & 1));
        const int item = s_item;
        if (item < 0) break;  // CTA-uniform
        const int tile = item / p.n_mblk, mblk = item % p.n_mblk;  // tile-major: concurrent CTAs share a tile in L2
        // rows before the lane's chunk on each strand: the only rank-directory reads of the tile
        const int64_t dir0 = (int64_t)tile * kTileWords + tid * NW;
        const uint32_t rank_p = __ldg(p.rank_dir + dir0), rank_m = __ldg(p.rank_dir + p.n_words + dir0);
        const uint32_t *sx = reinterpret_cast<const uint32_t *>(smem);
        const uint32_t *sy = sx + kSeqPlaneWords;
        const int32_t *sinfo = reinterpret_cast<const int32_t *>(sy + kSeqPlaneWords);
        const uint32_t *sv = sx + kSeqRecWords + tid * 4;
        {   // per-word prefix counts of the lane's valid rows (only this lane reads them back)
            int run_p = 0, run_m = 0;
#pragma unroll
            for (int w = 0; w < NW; ++w) {
                s_pref[w * kTileChunks + tid] = (uint16_t)run_p;
                s_pref[(NW + w) * kTileChunks + tid] = (uint16_t)run_m;
                run_p += __popc(sv[(w >> 2) * kSlotStride + (w & 3)]);
                run_m += __popc(sv[kTileWords + (w >> 2) * kSlotStride + (w & 3)]);
            }
        }
        const int info = sinfo[tid];
        const int contig = info < 0 ? -1 : (info & kChunkIdMask);
        const unsigned vmask = __ballot_sync(0xFFFFFFFFu, contig >= 0);
        if (vmask) {
            const int c0 = __shfl_sync(0xFFFFFFFFu, contig, __ffs(vmask) - 1);
            const bool warp_n = __any_sync(0xFFFFFFFFu, contig >= 0 && (info & kChunkFlagN));
            const bool warp_edge = __any_sync(0xFFFFFFFFu, contig >= 0 && (info & kChunkFlagEdge));
            WarpQueue &wq = s_queue[tid >> 5];
            if (warp_n) {
                LaneSeq<H, true> q;
                load_xyn<H>(sx, sy, tid, p.nonacgt + kHalo + (size_t)tile * kTileWords + tid * NW - H, q);
                // motifs are unstripped: a flanking '.' is never tested against the n plane, so clip to the contig
                const LaneEdge edge = lane_edge(true, info, (int64_t)tile * kTileChunks + tid, p.contig_start,
                                                p.contig_len);
                pattern_motifs<H, true>(p, mblk, q, edge, sv, s_pref, wq, rank_p, rank_m, contig, c0);
            } else {
                LaneSeq<H, false> q;
                load_xy<H>(sx, sy, tid, q);
                const LaneEdge edge = lane_edge(warp_edge, info, (int64_t)tile * kTileChunks + tid, p.contig_start,
                                                p.contig_len);
                pattern_motifs<H, false>(p, mblk, q, edge, sv, s_pref, wq, rank_p, rank_m, contig, c0);
            }
        }
        __syncthreads();  // everyone is done with the tile (and has read s_item)
    }
    if (p.counter && tid == 0 && atomicAdd(p.counter + 1, 1) == (int)gridDim.x - 1) {  // last CTA out re-arms the counter
        p.counter[0] = 0;
        p.counter[1] = 0;
    }
}

// offsets[i] = exclusive prefix sum of stats[i][0] over i < n_segments (offsets[n_segments] = total);
// cursor[i] = 0.  One block.
__global__ void __launch_bounds__(1024) segment_offsets_kernel(const unsigned long long *__restrict__ stats,
                                                               int64_t n_segments, long long *__restrict__ offsets,
                                                               int *__restrict__ cursor) {
    __shared__ long long s_part[1024];
    const int t = threadIdx.x;
    const int64_t per = (n_segments + 1023) / 1024;
    const int64_t b = min(n_segments, t * per), e = min(n_segments, b + per);
    long long sum = 0;
    for (int64_t i = b; i < e; ++i) sum += (long long)stats[3 * i];
    s_part[t] = sum;
    __syncthreads();
    if (t == 0) {
        long long run = 0;
        for (int i = 0; i < 1024; ++i) { const long long x = s_part[i]; s_part[i] = run; run += x; }
        offsets[n_segments] = run;
    }
    __syncthreads();
    long long run = s_part[t];
    for (int64_t i = b; i < e; ++i) {
        offsets[i] = run;
        cursor[i] = 0;
        run += (long long)stats[3 * i];
    }
}

}  // namespace nmb

extern "C" {

int nmb_pattern_index_build(const nmb_assembly *a, const int32_t *contig_id, const int64_t *pos, const uint8_t *strand,
                            const uint8_t *mod_type, int32_t want_modtype, const int64_t *n_mod,
                            const int64_t *n_valid_cov, const int64_t *n_diff, int64_t n_rows,
                            int64_t min_valid_read_coverage, double min_valid_cov_to_diff_fraction,
                            uint32_t *valid_records, uint32_t *rank_dir, int64_t *scratch, int32_t *payload,
                            int64_t *n_valid_rows, void *stream) {
    NMB_REQUIRE(a && valid_records && rank_dir && scratch && n_valid_rows, "nmb_pattern_index_build: null argument");
    NMB_REQUIRE(n_rows >= 0 && a->n_tiles > 0, "nmb_pattern_index_build: bad sizes");
    NMB_REQUIRE(n_rows < (1ll << 32), "nmb_pattern_index_build: more than 2^32 rows in one mod type");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n_words = (int64_t)a->n_tiles * nmb::kTileWords;
    NMB_CUDA(cudaMemsetAsync(valid_records, 0, (size_t)a->n_tiles * nmb::kValidRecBytes, s));
    nmb::RowFilter f{contig_id, pos, strand, mod_type, n_mod, n_valid_cov, n_diff, n_rows, want_modtype,
                     min_valid_read_coverage, min_valid_cov_to_diff_fraction, a->contig_start, a->contig_len,
                     a->n_contigs};
    int64_t row_blocks = (n_rows + 255) / 256;
    if (row_blocks > 148 * 32) row_blocks = 148 * 32;
    if (n_rows > 0) {
        NMB_REQUIRE(contig_id && pos && strand && n_mod && n_valid_cov && n_diff && payload,
                    "nmb_pattern_index_build: null column");
        nmb::pattern_valid_kernel<<<(unsigned)row_blocks, 256, 0, s>>>(f, valid_records);
        NMB_CUDA(cudaGetLastError());
    }
    const int64_t n_blocks = (2 * n_words + nmb::kRankBlockWords - 1) / nmb::kRankBlockWords;
    nmb::pattern_rank_count_kernel<<<(unsigned)n_blocks, 256, 0, s>>>(valid_records, n_words, scratch);
    NMB_CUDA(cudaGetLastError());
    nmb::scan_counts_kernel<1024><<<1, 1024, 0, s>>>(scratch, n_blocks, n_valid_rows);
    NMB_CUDA(cudaGetLastError());
    nmb::pattern_rank_write_kernel<<<(unsigned)n_blocks, 256, 0, s>>>(valid_records, n_words, scratch, rank_dir);
    NMB_CUDA(cudaGetLastError());
    if (n_rows > 0) {
        nmb::pattern_payload_kernel<<<(unsigned)row_blocks, 256, 0, s>>>(f, valid_records, rank_dir, n_words,
                                                                        (int2 *)payload);
        NMB_CUDA(cudaGetLastError());
    }
    return NMB_OK;
}

static int pattern_scan_impl(const nmb_assembly *a, const uint32_t *valid_records, const uint32_t *rank_dir,
                             const int32_t *payload, const void *programs, int32_t n_motifs, int32_t motifs_per_item,
                             int32_t max_motif_len, int32_t phase, int64_t *stats, const int64_t *offsets, int32_t *cursor,
                             double *fractions, int32_t grid_ctas, int32_t *work_counter, void *stream);

int nmb_pattern_scan(const nmb_assembly *a, const uint32_t *valid_records, const uint32_t *rank_dir,
                     const int32_t *payload, const void *programs, int32_t n_motifs, int32_t motifs_per_item,
                     int32_t max_motif_len, int32_t phase, int64_t *stats, const int64_t *offsets, int32_t *cursor,
                     double *fractions, int32_t grid_ctas, void *stream) {
    return pattern_scan_impl(a, valid_records, rank_dir, payload, programs, n_motifs, motifs_per_item, max_motif_len, phase,
                             stats, offsets, cursor, fractions, grid_ctas, nullptr, stream);
}

int nmb_pattern_scan_balanced(const nmb_assembly *a, const uint32_t *valid_records, const uint32_t *rank_dir,
                              const int32_t *payload, const void *programs, int32_t n_motifs, int32_t motifs_per_item,
                              int32_t max_motif_len, int32_t phase, int64_t *stats, const int64_t *offsets,
                              int32_t *cursor, double *fractions, int32_t grid_ctas, int32_t *work_counter, void *stream) {
    NMB_REQUIRE(work_counter, "nmb_pattern_scan_balanced: null work counter");
    return pattern_scan_impl(a, valid_records, rank_dir, payload, programs, n_motifs, motifs_per_item, max_motif_len, phase,
                             stats, offsets, cursor, fractions, grid_ctas, work_counter, stream);
}

static int pattern_scan_impl(const nmb_assembly *a, const uint32_t *valid_records, const uint32_t *rank_dir,
                             const int32_t *payload, const void *programs, int32_t n_motifs, int32_t motifs_per_item,
                             int32_t max_motif_len, int32_t phase, int64_t *stats, const int64_t *offsets, int32_t *cursor,
                             double *fractions, int32_t grid_ctas, int32_t *work_counter, void *stream) {
    NMB_REQUIRE(a && valid_records && rank_dir && programs && stats, "nmb_pattern_scan: null argument");
    NMB_REQUIRE(n_motifs >= 0 && (phase == 0 || phase == 1), "nmb_pattern_scan: n_motifs=%d phase=%d", n_motifs, phase);
    NMB_REQUIRE(motifs_per_item >= 1 && motifs_per_item <= NMB_MAX_MOTIFS_PER_ITEM, "nmb_pattern_scan: motifs_per_item=%d",
                motifs_per_item);
    NMB_REQUIRE(max_motif_len >= 1 && max_motif_len <= NMB_MAX_MOTIF_LEN, "nmb_pattern_scan: max_motif_len=%d",
                max_motif_len);
    NMB_REQUIRE(phase == 0 || (offsets && cursor && fractions), "nmb_pattern_scan: phase 1 needs offsets, cursor, fractions");
    if (n_motifs == 0) return NMB_OK;
    NMB_REQUIRE(payload, "nmb_pattern_scan: null payload");
    nmb::PatParams p;
    p.seq_records = a->seq_records;
    p.nonacgt = a->nonacgt;
    p.contig_start = a->contig_start;
    p.contig_len = a->contig_len;
    p.valid = valid_records;
    p.rank_dir = rank_dir;
    p.payload = (const int2 *)payload;
    p.programs = (const nmb::Program *)programs;
    p.stats = (unsigned long long *)stats;
    p.offsets = (const long long *)offsets;
    p.cursor = cursor;
    p.fractions = fractions;
    p.counter = work_counter;
    p.n_words = (int64_t)a->n_tiles * nmb::kTileWords;
    p.n_motifs = n_motifs;
    p.mpi = motifs_per_item;
    p.n_mblk = (n_motifs + motifs_per_item - 1) / motifs_per_item;
    p.n_tiles = a->n_tiles;
    p.n_contigs = a->n_contigs;
    const int64_t items = (int64_t)p.n_tiles * p.n_mblk;
    NMB_REQUIRE(items < (1ll << 31), "nmb_pattern_scan: too many work items");
    p.n_items = (int)items;
    p.write = phase;
    int grid = grid_ctas;
    if (grid <= 0) {
        int sms = nmb_device_sm_count();
        if (sms < 0) return sms;
        grid = 4 * sms;
    }
    if (grid > p.n_items) grid = p.n_items;
    cudaStream_t s = (cudaStream_t)stream;
    if (max_motif_len <= 32) {
        NMB_CUDA(cudaFuncSetAttribute(nmb::pattern_scan_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      nmb::kPatSmemBytes));
        nmb::pattern_scan_kernel<1><<<grid, nmb::kPatThreads, nmb::kPatSmemBytes, s>>>(p);
    } else {
        NMB_CUDA(cudaFuncSetAttribute(nmb::pattern_scan_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      nmb::kPatSmemBytes));
        nmb::pattern_scan_kernel<2><<<grid, nmb::kPatThreads, nmb::kPatSmemBytes, s>>>(p);
    }
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_segment_offsets(const int64_t *stats, int64_t n_segments, int64_t *offsets, int32_t *cursor, void *stream) {
    NMB_REQUIRE(stats && offsets && cursor && n_segments >= 0, "nmb_segment_offsets: bad argument");
    nmb::segment_offsets_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>((const unsigned long long *)stats, n_segments,
                                                                     (long long *)offsets, cursor);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

}  // extern "C"
