// K3 -- occurrence positions.
//   nmb_match_plane       : match bit-plane of one motif strand (same matcher as K2)
//   nmb_compact_positions : ascending positions of set bits (two-pass, deterministic order) --
//                           the array utils.subseq_indices returns (nanomotif/utils.py:61-66)
//   nmb_test_positions    : np.isin(pileup_positions, motif_index) of
//                           nanomotif/find_motifs_bin.py:1258-1261, in pileup order
#include "scan.cuh"

namespace nmb {

template <int H>
__global__ void __launch_bounds__(kTileChunks) match_plane_kernel(
    const uint32_t *__restrict__ seq_records, const uint32_t *__restrict__ nonacgt,
    const int64_t *__restrict__ contig_start, const int64_t *__restrict__ contig_len,
    const Program *__restrict__ program, int tile_begin, uint32_t *__restrict__ match_plane) {
    const int tid = threadIdx.x;
    const int tile = tile_begin + blockIdx.x;
    const uint32_t *rec = seq_records + (size_t)tile * kSeqRecWords;
    const int info = (int)rec[2 * kSeqPlaneWords + tid];
    uint32_t m[NW];
#pragma unroll
    for (int k = 0; k < NW; ++k) m[k] = 0;
    const bool warp_any = __any_sync(0xFFFFFFFFu, info >= 0);
    if (warp_any) {
        const bool warp_n = __any_sync(0xFFFFFFFFu, info >= 0 && (info & kChunkFlagN));
        const bool warp_edge = __any_sync(0xFFFFFFFFu, info >= 0 && (info & kChunkFlagEdge));
        const ProgramView pv = load_program(program);
        const uint32_t *px = rec, *py = rec + kSeqPlaneWords;
        if (warp_n) {
            LaneSeq<H, true> q;
            load_xyn<H>(px, py, tid, nonacgt + kHalo + (size_t)tile * kTileWords + tid * NW - H, q);
            // programs may be unstripped: a flanking '.' is never tested against the n plane, so clip to the contig
            const LaneEdge edge = lane_edge(true, info, (int64_t)tile * kTileChunks + tid, contig_start, contig_len);
            match_words<H, true>(pv, q, m, edge);
        } else {
            LaneSeq<H, false> q;
            load_xy<H>(px, py, tid, q);
            const LaneEdge edge = lane_edge(warp_edge, info, (int64_t)tile * kTileChunks + tid, contig_start, contig_len);
            match_words<H, false>(pv, q, m, edge);
        }
        if (info < 0) {
#pragma unroll
            for (int k = 0; k < NW; ++k) m[k] = 0;
        }
    }
    uint4 *dst = reinterpret_cast<uint4 *>(match_plane + (size_t)tile * kTileWords + tid * NW);
#pragma unroll
    for (int v = 0; v < NW / 4; ++v) dst[v] = make_uint4(m[4 * v], m[4 * v + 1], m[4 * v + 2], m[4 * v + 3]);
}

// ---- compaction ---------------------------------------------------------------------------------
// A block covers 2048 words (65536 bits) of [pos_begin, pos_end); thread t covers 8 of them.

__device__ __forceinline__ uint32_t masked_word(const uint32_t *plane, const uint32_t *mask,
                                                int64_t word, int64_t pos_end) {
    const int64_t first = word * 32;
    if (first >= pos_end) return 0u;
    uint32_t v = plane[word];
    if (mask) v &= mask[word];
    const int64_t rem = pos_end - first;
    if (rem < 32) v &= (1u << rem) - 1u;
    return v;
}

__global__ void __launch_bounds__(256) count_bits_kernel(const uint32_t *__restrict__ plane,
                                                         const uint32_t *__restrict__ mask,
                                                         int64_t word_begin, int64_t pos_end,
                                                         int64_t *__restrict__ block_counts) {
    __shared__ int s_warp[8];
    const int64_t w0 = word_begin + ((int64_t)blockIdx.x * 256 + threadIdx.x) * 8;
    int c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) c += __popc(masked_word(plane, mask, w0 + k, pos_end));
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int i = 0; i < 8; ++i) t += s_warp[i];
        block_counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(256) write_positions_kernel(
    const uint32_t *__restrict__ plane, const uint32_t *__restrict__ mask, int64_t word_begin,
    int64_t pos_begin, int64_t pos_end, const int64_t *__restrict__ block_offsets,
    int64_t *__restrict__ out_pos, int64_t capacity) {
    __shared__ int s_warp[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t w0 = word_begin + ((int64_t)blockIdx.x * 256 + threadIdx.x) * 8;
    uint32_t w[8];
    int c = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        w[k] = masked_word(plane, mask, w0 + k, pos_end);
        c += __popc(w[k]);
    }
    // warp-inclusive scan of the lane counts, then add the totals of the earlier warps
    int inc = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xFFFFFFFFu, inc, d);
        if (lane >= d) inc += o;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    int before = 0;
    for (int i = 0; i < warp; ++i) before += s_warp[i];
    int64_t o = block_offsets[blockIdx.x] + before + (inc - c);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        uint32_t v = w[k];
        const int64_t base = (w0 + k) * 32 - pos_begin;
        while (v) {
            const int b = __ffs(v) - 1;
            v &= v - 1;
            if (o < capacity) out_pos[o] = base + b;
            ++o;
        }
    }
}

__global__ void __launch_bounds__(256) test_positions_kernel(const uint32_t *__restrict__ plane,
                                                             int64_t base, int64_t limit,
                                                             const int64_t *__restrict__ pos, int64_t n,
                                                             uint8_t *__restrict__ flag) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
        const int64_t p = pos[r];
        uint8_t f = 0;
        if (p >= 0 && p < limit) {
            const int64_t g = base + p;
            f = (plane[g >> 5] >> (g & 31)) & 1u;
        }
        flag[r] = f;
    }
}


// plane[p] &= (upper(ascii[p + shift]) == letter), false outside [0, n): one warp per 32-bit word, lane = bit.
// Serves motif positions that are LITERAL non-ACGT letters (an 'N' in a motif string is the regex literal N,
// nanomotif/utils.py:61-66 -- it matches the contig letter N and nothing else).
__global__ void __launch_bounds__(256) letter_plane_kernel(const uint8_t *__restrict__ ascii, int64_t n, int letter,
                                                           int64_t shift, uint32_t *__restrict__ plane,
                                                           int64_t n_words) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= n_words) return;
    const int64_t q = w * 32 + (threadIdx.x & 31) + shift;
    bool ok = false;
    if (q >= 0 && q < n) {
        int c = ascii[q];
        if (c >= 'a' && c <= 'z') c -= 32;  // the packer upper-cases, like seq.py:55
        ok = c == letter;
    }
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
    if ((threadIdx.x & 31) == 0) plane[w] &= m;
}

}  // namespace nmb

extern "C" {

int nmb_match_plane(const nmb_assembly *a, const void *programs, int32_t motif_index, int32_t strand,
                    int32_t motif_len, int32_t tile_begin, int32_t tile_count, uint32_t *match_plane,
                    void *stream) {
    NMB_REQUIRE(a && programs && match_plane, "nmb_match_plane: null argument");
    NMB_REQUIRE(strand == 0 || strand == 1, "nmb_match_plane: strand=%d", strand);
    NMB_REQUIRE(motif_len >= 1 && motif_len <= NMB_MAX_MOTIF_LEN, "nmb_match_plane: motif_len=%d",
                motif_len);
    NMB_REQUIRE(tile_begin >= 0 && tile_count >= 0 && tile_begin + tile_count <= a->n_tiles,
                "nmb_match_plane: tiles [%d,+%d) outside 0..%d", tile_begin, tile_count, a->n_tiles);
    if (tile_count == 0) return NMB_OK;
    const nmb::Program *prog = (const nmb::Program *)programs + (size_t)motif_index * 2 + strand;
    cudaStream_t s = (cudaStream_t)stream;
    if (motif_len <= 32)  // one halo word covers a total shift (and a mod_pos) of at most 31
        nmb::match_plane_kernel<1><<<tile_count, nmb::kTileChunks, 0, s>>>(
            a->seq_records, a->nonacgt, a->contig_start, a->contig_len, prog, tile_begin, match_plane);
    else
        nmb::match_plane_kernel<2><<<tile_count, nmb::kTileChunks, 0, s>>>(
            a->seq_records, a->nonacgt, a->contig_start, a->contig_len, prog, tile_begin, match_plane);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_compact_positions(const uint32_t *plane, const uint32_t *mask, int64_t pos_begin,
                          int64_t pos_end, int64_t *tile_counts, int64_t *out_pos, int64_t capacity,
                          int64_t *n_out, void *stream) {
    NMB_REQUIRE(plane && tile_counts && n_out, "nmb_compact_positions: null argument");
    NMB_REQUIRE(pos_begin >= 0 && pos_end >= pos_begin && (pos_begin % 32) == 0,
                "nmb_compact_positions: range [%lld,%lld) must start on a word boundary",
                (long long)pos_begin, (long long)pos_end);
    NMB_REQUIRE(capacity >= 0 && (capacity == 0 || out_pos), "nmb_compact_positions: bad capacity");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n_bits = pos_end - pos_begin;
    const int64_t n_blocks = (n_bits + NMB_TILE_BP - 1) / NMB_TILE_BP;
    if (n_blocks == 0) {
        NMB_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int64_t), s));
        return NMB_OK;
    }
    NMB_REQUIRE(n_blocks < (1ll << 31), "nmb_compact_positions: range too large");
    nmb::count_bits_kernel<<<(unsigned)n_blocks, 256, 0, s>>>(plane, mask, pos_begin / 32, pos_end,
                                                             tile_counts);
    NMB_CUDA(cudaGetLastError());
    nmb::scan_counts_kernel<1024><<<1, 1024, 0, s>>>(tile_counts, n_blocks, n_out);
    NMB_CUDA(cudaGetLastError());
    if (capacity > 0) {
        nmb::write_positions_kernel<<<(unsigned)n_blocks, 256, 0, s>>>(
            plane, mask, pos_begin / 32, pos_begin, pos_end, tile_counts, out_pos, capacity);
        NMB_CUDA(cudaGetLastError());
    }
    return NMB_OK;
}

int nmb_test_positions(const uint32_t *plane, int64_t base, int64_t limit, const int64_t *pos,
                       int64_t n, uint8_t *flag, void *stream) {
    NMB_REQUIRE(n >= 0, "nmb_test_positions: n=%lld", (long long)n);
    if (n == 0) return NMB_OK;
    NMB_REQUIRE(plane && pos && flag, "nmb_test_positions: null argument");
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    nmb::test_positions_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(plane, base, limit,
                                                                                 pos, n, flag);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_letter_plane(const uint8_t *ascii, int64_t n, int32_t letter, int64_t shift, uint32_t *plane, int64_t n_words,
                     void *stream) {
    NMB_REQUIRE(ascii && plane && n >= 0 && n_words >= 0 && letter >= 0 && letter < 256, "nmb_letter_plane: bad arguments");
    if (n_words == 0) return NMB_OK;
    const int64_t threads = n_words * 32;
    nmb::letter_plane_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ascii, n, letter, shift,
                                                                                               plane, n_words);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

}  // extern "C"
