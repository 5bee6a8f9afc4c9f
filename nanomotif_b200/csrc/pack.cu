// K1 -- loaders: ASCII contigs -> 2-bit tile records (+ non-ACGT plane), pileup rows -> class
// bit-planes.  Reference behaviour being replaced: nanomotif/fasta.py:35-49 (contig strings),
// nanomotif/seq.py:53-55 (upper-casing), nanomotif/find_motifs_bin.py:1308-1314 (per-call split
// of the pileup into methylated / unmethylated x strand position arrays).
#include "common.cuh"

namespace nmb {

// One warp per 512-bp chunk.  Lane l reads base l of each of the chunk's 16 words (coalesced
// 32-byte reads) and three ballots build the word of each plane.
__global__ void __launch_bounds__(256) pack_sequence_kernel(
    const uint8_t *__restrict__ ascii, const int64_t *__restrict__ ascii_off,
    const int64_t *__restrict__ contig_start, const int64_t *__restrict__ contig_len,
    int n_contigs, int n_tiles, uint32_t *__restrict__ seq_records, uint32_t *__restrict__ nonacgt) {
    const int lane = threadIdx.x & 31;
    const int64_t n_chunks = (int64_t)n_tiles * kTileChunks;
    const int64_t warps_total = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t q = (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); q < n_chunks;
         q += warps_total) {
        const int64_t chunk_pos = q * NMB_CHUNK_BP;
        // largest c with contig_start[c] <= chunk_pos (uniform binary search)
        int lo = 0, hi = n_contigs;  // invariant: start[lo-1] <= chunk_pos < start[hi]
        while (lo < hi) {
            int mid = (lo + hi) >> 1;
            if (__ldg(contig_start + mid) <= chunk_pos) lo = mid + 1; else hi = mid;
        }
        int c = lo - 1;
        int64_t local0 = 0, len = 0, aoff = 0;
        if (c >= 0) {
            local0 = chunk_pos - __ldg(contig_start + c);
            len = __ldg(contig_len + c);
            aoff = __ldg(ascii_off + c);
            if (local0 >= len) c = -1;
        }
        uint32_t my_x = 0, my_y = 0, my_n = 0xFFFFFFFFu;
        bool letter = false;  // a non-ACGT letter INSIDE the contig (padding does not count)
#pragma unroll
        for (int w = 0; w < kChunkWords; ++w) {
            int code = 4;
            if (c >= 0) {
                int64_t local = local0 + w * 32 + lane;
                if (local < len) {
                    int ch = ascii[aoff + local] & 0xDF;  // upper-case (seq.py:55)
                    code = ch == 'A' ? 0 : ch == 'T' ? 1 : ch == 'G' ? 2 : ch == 'C' ? 3 : 4;
                    letter |= code == 4;
                }
            }
            uint32_t xb = __ballot_sync(0xFFFFFFFFu, (code & 2) && code < 4);
            uint32_t yb = __ballot_sync(0xFFFFFFFFu, (code & 1) && code < 4);
            uint32_t nb = __ballot_sync(0xFFFFFFFFu, code == 4);
            if (lane == w) { my_x = xb; my_y = yb; my_n = nb; }
        }
        if (lane < kChunkWords) {
            const int64_t gw = q * kChunkWords + lane;  // global word
            const int64_t tile = gw / kTileWords;
            const int wt = (int)(gw % kTileWords);
            uint32_t *rec = seq_records + tile * kSeqRecWords;
            rec[kHalo + word_slot(wt)] = my_x;
            rec[kSeqPlaneWords + kHalo + word_slot(wt)] = my_y;
            if (wt < kHalo) {  // also the right halo of the previous tile / zero left edge
                if (tile > 0) {
                    uint32_t *prev = rec - kSeqRecWords;
                    prev[kHalo + kTileWords + wt] = my_x;
                    prev[kSeqPlaneWords + kHalo + kTileWords + wt] = my_y;
                } else {
                    rec[wt] = 0;
                    rec[kSeqPlaneWords + wt] = 0;
                }
            }
            if (wt >= kTileWords - kHalo) {  // also the left halo of the next tile / zero right edge
                const int h = wt - (kTileWords - kHalo);
                if (tile + 1 < n_tiles) {
                    uint32_t *next = rec + kSeqRecWords;
                    next[h] = my_x;
                    next[kSeqPlaneWords + h] = my_y;
                } else {
                    rec[kHalo + kTileWords + h] = 0;
                    rec[kSeqPlaneWords + kHalo + kTileWords + h] = 0;
                }
            }
            nonacgt[kHalo + gw] = my_n;
        }
        letter = __any_sync(0xFFFFFFFFu, letter);
        if (lane == 0) {
            const int64_t tile = q / kTileChunks;
            seq_records[tile * kSeqRecWords + 2 * kSeqPlaneWords + (int)(q % kTileChunks)] =
                (uint32_t)(c >= 0 && letter ? (c | kChunkFlagLetter) : c);
        }
    }
}

// Second pass: which matcher a chunk needs.  A lane reads its 16 words plus two halo words on either side
// (motif length <= 62 < 64).  Non-ACGT LETTERS of a contig within that reach (decided per neighbouring
// chunk, conservatively) need the full path that tests every constrained position; inter-contig padding
// alone needs only the cheap edge treatment (first and last motif position must lie in the contig: padding
// runs are >= 64 > motif length, so a match cannot span one).
__device__ __forceinline__ uint32_t *chunk_info_ptr(uint32_t *seq_records, int64_t q) {
    return seq_records + (q / kTileChunks) * kSeqRecWords + 2 * kSeqPlaneWords + (int)(q % kTileChunks);
}

__global__ void __launch_bounds__(256) chunk_flags_kernel(int n_tiles,
                                                          uint32_t *__restrict__ seq_records,
                                                          uint32_t *__restrict__ nonacgt) {
    const int64_t n_chunks = (int64_t)n_tiles * kTileChunks;
    const int64_t n_words = (int64_t)n_tiles * kTileWords;
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q == 0) {
        for (int i = 0; i < kHalo; ++i) {
            nonacgt[i] = 0xFFFFFFFFu;
            nonacgt[kHalo + n_words + i] = 0xFFFFFFFFu;
        }
    }
    if (q >= n_chunks) return;
    uint32_t any = 0;
    const uint32_t *p = nonacgt + kHalo + q * kChunkWords;
    for (int i = -2; i < kChunkWords + 2; ++i) {
        // pad words are written by thread 0 concurrently: treat the array ends as flagged
        int64_t gw = q * kChunkWords + i;
        any |= (gw < 0 || gw >= n_words) ? 0xFFFFFFFFu : p[i];
    }
    uint32_t *info = chunk_info_ptr(seq_records, q);
    // neighbours update their own words concurrently, but only bits 29/30: bit 28 is stable
    const int c = (int)*(volatile uint32_t *)info;
    if (c < 0 || !any) return;
    bool letter = c & kChunkFlagLetter;
    for (int dq = -1; dq <= 1; dq += 2) {
        if (q + dq < 0 || q + dq >= n_chunks) continue;
        const int cn = (int)*(volatile uint32_t *)chunk_info_ptr(seq_records, q + dq);
        letter |= cn >= 0 && (cn & kChunkFlagLetter);
    }
    atomicOr(info, (uint32_t)(letter ? kChunkFlagN : kChunkFlagEdge));
}

__global__ void __launch_bounds__(256) class_planes_kernel(
    const int32_t *__restrict__ contig_id, const int64_t *__restrict__ pos,
    const uint8_t *__restrict__ strand, const uint8_t *__restrict__ modtype,
    const double *__restrict__ fraction, int64_t n_rows, double low, double high,
    const int64_t *__restrict__ contig_start, const int64_t *__restrict__ contig_len, int n_contigs,
    int n_tiles, int n_modtypes, uint32_t *__restrict__ cls, unsigned long long *__restrict__ dup_count) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += stride) {
        const int c = contig_id[r];
        if (c < 0 || c >= n_contigs) continue;
        const int64_t p = pos[r];
        if (p < 0 || p >= __ldg(contig_len + c)) continue;
        const int mt = modtype ? modtype[r] : 0;
        if (mt >= n_modtypes) continue;
        const int st = strand[r];
        if (st > 1) continue;  // modkit's '.' (--combine-strands): the reference's strand == "+" / "-" filters drop it
        const double f = fraction[r];
        const bool is_mod = f >= high;   // find_motifs_bin.py:1308
        const bool is_non = f <= low;    // find_motifs_bin.py:1309
        if (!is_mod && !is_non) continue;
        const int64_t g = __ldg(contig_start + c) + p;
        const int64_t tile = g >> 16;
        const int w = word_slot((int)((g >> 5) & (kTileWords - 1)));
        const uint32_t bit = 1u << (g & 31);
        uint32_t *rec = cls + ((int64_t)mt * n_tiles + tile) * kClsRecWords +
                        (st ? 2 : 0) * kTileWords + w;
        uint32_t old = 0;
        if (is_mod) old |= atomicOr(rec, bit);
        if (is_non) old |= atomicOr(rec + kTileWords, bit);
        if ((old & bit) && dup_count) atomicAdd(dup_count, 1ull);  // a repeated (contig, pos, strand, mod type)
    }
}

// Compact rows (7 bytes each): 32-bit position, flags = strand | mod type << 1, and the modkit percentage
// as an exact fixed-point key (hundredths of a percent, 0..10000).  Rows are grouped by contig
// (row_off[c] .. row_off[c+1]).  key >= key_high / key <= key_low are the host-derived integer images
// of the reference's float64 tests (see nanomotif_b200/device.py::threshold_keys).
__global__ void __launch_bounds__(256) class_planes_compact_kernel(
    const int32_t *__restrict__ pos, const uint8_t *__restrict__ flags, const uint16_t *__restrict__ key,
    const int64_t *__restrict__ row_off, int n_contigs, int64_t n_rows, int key_low, int key_high,
    const int64_t *__restrict__ contig_start, const int64_t *__restrict__ contig_len, int n_tiles,
    int n_modtypes, uint32_t *__restrict__ cls) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n_rows; r += stride) {
        const int k = key[r];
        if (k > 10000) continue;  // off the two-decimal grid (nmb_bed_parse writes 0xFFFF): neither class
        const bool is_mod = k >= key_high, is_non = k <= key_low;
        if (!is_mod && !is_non) continue;
        int lo = 0, hi = n_contigs;  // largest c with row_off[c] <= r
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(row_off + mid) <= r) lo = mid; else hi = mid;
        }
        const int64_t p = pos[r];
        if (p < 0 || p >= __ldg(contig_len + lo)) continue;
        const int f = flags[r];
        const int mt = f >> 1;
        if (mt >= n_modtypes) continue;
        const int64_t g = __ldg(contig_start + lo) + p;
        uint32_t *rec = cls + ((int64_t)mt * n_tiles + (g >> 16)) * kClsRecWords + ((f & 1) ? 2 : 0) * kTileWords +
                        word_slot((int)((g >> 5) & (kTileWords - 1)));
        const uint32_t bit = 1u << (g & 31);
        if (is_mod) atomicOr(rec, bit);
        if (is_non) atomicOr(rec + kTileWords, bit);
    }
}

}  // namespace nmb

extern "C" {

int nmb_pack_sequence(const uint8_t *ascii, const int64_t *ascii_off, const int64_t *contig_start,
                      const int64_t *contig_len, int32_t n_contigs, int32_t n_tiles,
                      uint32_t *seq_records, uint32_t *nonacgt, void *stream) {
    NMB_REQUIRE(n_contigs >= 0 && n_tiles > 0, "nmb_pack_sequence: n_contigs=%d n_tiles=%d", n_contigs,
                n_tiles);
    NMB_REQUIRE(seq_records && nonacgt, "nmb_pack_sequence: null output");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n_chunks = (int64_t)n_tiles * nmb::kTileChunks;
    int64_t blocks = (n_chunks + 7) / 8;  // 8 warps per block
    if (blocks > 148 * 64) blocks = 148 * 64;
    nmb::pack_sequence_kernel<<<(unsigned)blocks, 256, 0, s>>>(ascii, ascii_off, contig_start,
                                                              contig_len, n_contigs, n_tiles,
                                                              seq_records, nonacgt);
    NMB_CUDA(cudaGetLastError());
    nmb::chunk_flags_kernel<<<(unsigned)((n_chunks + 255) / 256), 256, 0, s>>>(n_tiles, seq_records,
                                                                              nonacgt);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_build_class_planes(const int32_t *contig_id, const int64_t *pos, const uint8_t *strand,
                           const uint8_t *modtype, const double *fraction_mod, int64_t n_rows,
                           double low, double high, const nmb_assembly *a, int32_t n_modtypes,
                           uint32_t *class_records, void *stream) {
    const int rc = nmb_clear_class_planes(a, n_modtypes, class_records, stream);
    if (rc != NMB_OK) return rc;
    return nmb_add_class_planes(contig_id, pos, strand, modtype, fraction_mod, n_rows, low, high, a, n_modtypes,
                                class_records, nullptr, stream);
}

int nmb_add_class_planes(const int32_t *contig_id, const int64_t *pos, const uint8_t *strand, const uint8_t *modtype,
                         const double *fraction_mod, int64_t n_rows, double low, double high, const nmb_assembly *a,
                         int32_t n_modtypes, uint32_t *class_records, int64_t *dup_count, void *stream) {
    NMB_REQUIRE(a && class_records, "nmb_add_class_planes: null argument");
    NMB_REQUIRE(n_rows >= 0 && n_modtypes > 0 && a->n_tiles > 0, "nmb_add_class_planes: bad sizes");
    if (n_rows == 0) return NMB_OK;
    NMB_REQUIRE(contig_id && pos && strand && fraction_mod, "nmb_add_class_planes: null column");
    int64_t blocks = (n_rows + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    nmb::class_planes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        contig_id, pos, strand, modtype, fraction_mod, n_rows, low, high, a->contig_start, a->contig_len,
        a->n_contigs, a->n_tiles, n_modtypes, class_records, (unsigned long long *)dup_count);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_clear_class_planes(const nmb_assembly *a, int32_t n_modtypes, uint32_t *class_records, void *stream) {
    NMB_REQUIRE(a && class_records, "nmb_clear_class_planes: null argument");
    NMB_REQUIRE(n_modtypes > 0 && a->n_tiles > 0, "nmb_clear_class_planes: bad sizes");
    NMB_CUDA(cudaMemsetAsync(class_records, 0, (size_t)n_modtypes * a->n_tiles * nmb::kClsRecBytes,
                             (cudaStream_t)stream));
    return NMB_OK;
}

int nmb_add_class_planes_compact(const int32_t *pos, const uint8_t *flags, const uint16_t *percent_x100,
                                 const int64_t *contig_row_off, int64_t n_rows, int32_t key_low, int32_t key_high,
                                 const nmb_assembly *a, int32_t n_modtypes, uint32_t *class_records, void *stream) {
    NMB_REQUIRE(a && class_records, "nmb_add_class_planes_compact: null argument");
    NMB_REQUIRE(n_rows >= 0 && n_modtypes > 0 && n_modtypes <= 128 && a->n_tiles > 0 && a->n_contigs > 0,
                "nmb_add_class_planes_compact: bad sizes");
    if (n_rows == 0) return NMB_OK;
    NMB_REQUIRE(pos && flags && percent_x100 && contig_row_off, "nmb_add_class_planes_compact: null column");
    int64_t blocks = (n_rows + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    nmb::class_planes_compact_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        pos, flags, percent_x100, contig_row_off, a->n_contigs, n_rows, key_low, key_high, a->contig_start,
        a->contig_len, a->n_tiles, n_modtypes, class_records);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_build_class_planes_compact(const int32_t *pos, const uint8_t *flags, const uint16_t *percent_x100,
                                   const int64_t *contig_row_off, int64_t n_rows, int32_t key_low,
                                   int32_t key_high, const nmb_assembly *a, int32_t n_modtypes,
                                   uint32_t *class_records, void *stream) {
    const int rc = nmb_clear_class_planes(a, n_modtypes, class_records, stream);
    if (rc != NMB_OK) return rc;
    return nmb_add_class_planes_compact(pos, flags, percent_x100, contig_row_off, n_rows, key_low, key_high, a,
                                        n_modtypes, class_records, stream);
}

}  // extern "C"
