// K6 -- modkit bedMethyl text -> columnar pileup rows on the device.
//
// Replaces the CSV scan of nanomotif/dataload.py:72-100 (pl.scan_csv, tab separated, 18 columns, keeps
// columns 1, 2, 4, 6, 10, 11 and divides column 11 by 100) and the row materialisation of
// epymetheus.query_pileup_records (dataload.py:109-120).  Three steps, all on the device:
//   nmb_index_bytes   positions of a byte value (here '\n'), ascending -- count / scan / write
//   nmb_bed_parse     one thread per line: split on tabs, parse the kept columns
//   nmb_gather_rows   compaction of the parsed columns by an index list (rows kept by the filters)
// Column 11 is decimal text; its value is taken as mantissa / 10^digits in one IEEE division, which is
// the correctly rounded double for <= 15 significant digits (both operands exact), i.e. what the
// reference's CSV reader returns; fraction_mod = that / 100 like dataload.py:85.
#include "common.cuh"

namespace nmb {

constexpr int kIndexThreads = 256;
constexpr int kIndexBytesPerThread = 16;
constexpr int kIndexBlockBytes = kIndexThreads * kIndexBytesPerThread;  // 4096

__device__ __forceinline__ unsigned match_mask16(const uint8_t *__restrict__ src, int64_t i0, int64_t n, uint8_t value) {
    unsigned m = 0;
    if (i0 + kIndexBytesPerThread <= n && (reinterpret_cast<uintptr_t>(src + i0) & 15) == 0) {
        const uint4 v = *reinterpret_cast<const uint4 *>(src + i0);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 16; ++k) m |= (((w[k >> 2] >> (8 * (k & 3))) & 0xFF) == value) << k;
    } else {
        for (int k = 0; k < kIndexBytesPerThread; ++k)
            if (i0 + k < n && src[i0 + k] == value) m |= 1u << k;
    }
    return m;
}

__global__ void __launch_bounds__(kIndexThreads) count_bytes_kernel(const uint8_t *__restrict__ src, int64_t n,
                                                                    uint8_t value, int64_t *__restrict__ block_counts) {
    __shared__ int s_warp[kIndexThreads / 32];
    const int64_t i0 = ((int64_t)blockIdx.x * kIndexThreads + threadIdx.x) * kIndexBytesPerThread;
    int c = __popc(match_mask16(src, i0, n, value));
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int i = 0; i < kIndexThreads / 32; ++i) t += s_warp[i];
        block_counts[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kIndexThreads) write_byte_index_kernel(
    const uint8_t *__restrict__ src, int64_t n, uint8_t value, const int64_t *__restrict__ block_offsets,
    int64_t *__restrict__ out, int64_t capacity) {
    __shared__ int s_warp[kIndexThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i0 = ((int64_t)blockIdx.x * kIndexThreads + threadIdx.x) * kIndexBytesPerThread;
    unsigned m = match_mask16(src, i0, n, value);
    const int c = __popc(m);
    int incl = c;  // inclusive warp scan
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int before = 0;
    for (int i = 0; i < warp; ++i) before += s_warp[i];
    int64_t o = block_offsets[blockIdx.x] + before + incl - c;
    while (m) {
        const int k = __ffs(m) - 1;
        m &= m - 1;
        if (o < capacity) out[o] = i0 + k;
        ++o;
    }
}

// ---- line parser --------------------------------------------------------------------------------

struct NameTable {
    const uint64_t *hash;      // FNV-1a 64 of every name, ascending
    const int32_t *id;         // id of the name at that rank
    const int64_t *name_off;   // [n + 1] byte offsets into names, by rank
    const uint8_t *names;
    int n;
};

struct BedColumns {
    int32_t *contig_id;
    int64_t *position;
    uint8_t *strand, *mod_type;
    int64_t *n_valid_cov;
    double *fraction_mod;
    uint16_t *percent_x100;
    int64_t *n_mod, *n_diff;  // may be null
};

__device__ __forceinline__ int lookup_name(const NameTable &t, uint64_t h, const uint8_t *s, int len) {
    int lo = 0, hi = t.n;  // first rank with hash >= h
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(t.hash + mid) < h) lo = mid + 1; else hi = mid;
    }
    for (; lo < t.n && __ldg(t.hash + lo) == h; ++lo) {
        const int64_t b = __ldg(t.name_off + lo), e = __ldg(t.name_off + lo + 1);
        if (e - b != len) continue;
        bool same = true;
        for (int i = 0; i < len && same; ++i) same = t.names[b + i] == s[i];
        if (same) return __ldg(t.id + lo);
    }
    return -1;
}

__constant__ double kPow10[16] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15};

// status counters: [0] malformed lines (fewer than 18 fields), [1] empty lines, [2] fields that are not
// plain numbers (NA / null / exponent notation / > 15 digits), [3] rows of unknown contigs
__global__ void __launch_bounds__(128) bed_parse_kernel(
    const uint8_t *__restrict__ text, int64_t n_bytes, const int64_t *__restrict__ newline_pos, int64_t n_lines,
    NameTable contigs, const uint64_t *__restrict__ modtype_keys, int n_modtypes, BedColumns out,
    int32_t *__restrict__ status) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_lines) return;
    int64_t p = r == 0 ? 0 : newline_pos[r - 1] + 1;
    const int64_t line_begin = p;

    uint64_t h = 0xcbf29ce484222325ull;  // field 1: FNV-1a of the contig name
    int name_len = 0;
    uint64_t mt_key = 0;                 // field 4: up to 8 bytes, first byte most significant
    int mt_len = 0;
    int strand_c = 0, strand_len = 0;    // field 6
    int64_t iv = 0;                      // running integer of the current numeric field
    int nd = 0, fd = 0;                  // digits seen, digits after the decimal point
    bool neg = false, point = false, notnum = false;
    int64_t position = -1, cov = -1, n_mod = -1, n_diff = -1;
    double percent = __longlong_as_double(0x7ff8000000000000ll);  // NaN until parsed
    int key = 0xFFFF;
    int n_notnum = 0;

    int field = 0;
    for (;; ++p) {
        const int c = p < n_bytes ? text[p] : '\n';
        if (c == '\t' || c == '\n' || c == '\r') {
            const bool ok = nd > 0 && !notnum;
            const int64_t v = neg ? -iv : iv;
            switch (field) {
                case 1: if (ok && !point) position = v; else ++n_notnum; break;
                case 9: if (ok && !point) cov = v; else ++n_notnum; break;
                case 11: if (ok && !point) n_mod = v; else if (out.n_mod) ++n_notnum; break;
                case 16: if (ok && !point) n_diff = v; else if (out.n_diff) ++n_notnum; break;
                case 10:
                    if (ok && nd <= 15) {
                        // sign applied to the double, not to iv: "-0.00" is -0.0 like the reference's reader
                        percent = (neg ? -(double)iv : (double)iv) / kPow10[fd];
                        if (!neg && fd <= 2) {
                            const int64_t k = iv * (fd == 0 ? 100 : fd == 1 ? 10 : 1);
                            if (k <= 10000) key = (int)k;
                        }
                    } else {
                        ++n_notnum;
                    }
                    break;
                default: break;
            }
            ++field;
            iv = 0; nd = 0; fd = 0; neg = false; point = false; notnum = false;
            if (c != '\t') break;
            continue;
        }
        switch (field) {
            case 0: h = (h ^ (uint64_t)c) * 0x100000001b3ull; ++name_len; break;
            case 3: if (mt_len < 8) mt_key = (mt_key << 8) | (uint64_t)c; ++mt_len; break;
            case 5: if (strand_len == 0) strand_c = c; ++strand_len; break;
            case 1: case 9: case 10: case 11: case 16:
                if (c >= '0' && c <= '9') {
                    if (nd < 18) iv = iv * 10 + (c - '0'); else notnum = true;
                    ++nd;
                    if (point) ++fd;
                } else if (c == '.' && field == 10 && !point) {
                    point = true;
                } else if (c == '-' && nd == 0 && !neg && !point) {
                    neg = true;
                } else {
                    notnum = true;
                }
                break;
            default: break;
        }
    }

    int cid = -2;  // line to drop
    if (field == 1 && name_len == 0) {
        atomicAdd(status + 1, 1);  // empty line
    } else if (field < 18) {
        atomicAdd(status + 0, 1);
    } else {
        cid = lookup_name(contigs, h, text + line_begin, name_len);
        if (cid < 0) atomicAdd(status + 3, 1);
        if (n_notnum) atomicAdd(status + 2, n_notnum);
    }
    int mt = 255;
    if (mt_len >= 1 && mt_len <= 8)
        for (int i = 0; i < n_modtypes; ++i)
            if (__ldg(modtype_keys + i) == mt_key) mt = i;
    out.contig_id[r] = cid;
    out.position[r] = position;
    out.strand[r] = strand_len == 1 ? (strand_c == '+' ? 0 : strand_c == '-' ? 1 : 2) : 2;
    out.mod_type[r] = (uint8_t)mt;
    out.n_valid_cov[r] = cov;
    out.fraction_mod[r] = percent / 100.0;  // dataload.py:85
    out.percent_x100[r] = (uint16_t)key;
    if (out.n_mod) out.n_mod[r] = n_mod;
    if (out.n_diff) out.n_diff[r] = n_diff;
}

// ---- FASTA text -> concatenated sequence bytes (nanomotif/fasta.py:35-49 load_fasta_fastx) ----
// Line r spans [begin, end) of the text (newline index as in bed_parse_kernel); leading / trailing blanks and '\r'
// are stripped like the host loader's line.strip().  kind[r] = 1 header ('>' first), 0 sequence; payload[r] = bytes
// this pass copies for the line: sequence bytes of sequence lines (want_headers = 0) or the header text after '>'
// of header lines (want_headers = 1).
__device__ __forceinline__ void fasta_line_span(const uint8_t *__restrict__ text, int64_t n_bytes,
                                                const int64_t *__restrict__ newline_pos, int64_t n_newlines, int64_t r,
                                                int64_t &b, int64_t &e) {
    b = r == 0 ? 0 : newline_pos[r - 1] + 1;
    e = r < n_newlines ? newline_pos[r] : n_bytes;
    while (e > b && (text[e - 1] == '\r' || text[e - 1] == ' ' || text[e - 1] == '\t')) --e;
    while (b < e && (text[b] == ' ' || text[b] == '\t')) ++b;
}

__global__ void __launch_bounds__(256) fasta_lines_kernel(const uint8_t *__restrict__ text, int64_t n_bytes,
                                                          const int64_t *__restrict__ newline_pos, int64_t n_newlines,
                                                          int64_t n_lines, int want_headers, uint8_t *__restrict__ kind,
                                                          int64_t *__restrict__ payload) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_lines) return;
    int64_t b, e;
    fasta_line_span(text, n_bytes, newline_pos, n_newlines, r, b, e);
    const bool header = e > b && text[b] == '>';
    kind[r] = header;
    payload[r] = want_headers ? (header ? e - b - 1 : 0) : (header ? 0 : e - b);
}

// One warp per line: copy its payload to out + out_off[r] (coalesced).
__global__ void __launch_bounds__(256) fasta_copy_kernel(const uint8_t *__restrict__ text, int64_t n_bytes,
                                                         const int64_t *__restrict__ newline_pos, int64_t n_newlines,
                                                         int64_t n_lines, int want_headers, const int64_t *__restrict__ out_off,
                                                         uint8_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_lines; r += warps) {
        int64_t b, e;
        fasta_line_span(text, n_bytes, newline_pos, n_newlines, r, b, e);
        const bool header = e > b && text[b] == '>';
        if (header != (want_headers != 0)) continue;
        if (header) ++b;
        uint8_t *dst = out + out_off[r];
        for (int64_t i = lane; i < e - b; i += 32) dst[i] = text[b + i];
    }
}

template <typename T>
__global__ void __launch_bounds__(256) gather_rows_kernel(const T *__restrict__ src, const int64_t *__restrict__ index,
                                                          int64_t n, T *__restrict__ dst) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[index[i]];
}


// ---- string columns of a table (Arrow utf8 / large_utf8 layout) -> ids -----------------------------
// Row r's string is data[off[r] .. off[r+1]); offsets are 32- or 64-bit.  One thread per row: FNV-1a of the
// bytes, binary search in the name table, byte compare.  Consecutive rows of a pileup mostly carry the same
// contig name, so the table probes hit the same cache lines across a warp.
template <typename OffT, typename OutT>
__global__ void __launch_bounds__(256) lookup_strings_kernel(const uint8_t *__restrict__ data,
                                                             const OffT *__restrict__ off, int64_t n_rows,
                                                             NameTable table, int missing,
                                                             OutT *__restrict__ out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int64_t b = off[r], e = off[r + 1];
    uint64_t h = 0xcbf29ce484222325ull;
    for (int64_t i = b; i < e; ++i) h = (h ^ data[i]) * 0x100000001b3ull;
    const int id = lookup_name(table, h, data + b, (int)(e - b));
    out[r] = (OutT)(id < 0 ? missing : id);
}

}  // namespace nmb

extern "C" {

int nmb_index_bytes(const uint8_t *src, int64_t n_bytes, int32_t value, int64_t *scratch, int64_t *out_index,
                    int64_t capacity, int64_t *n_out, void *stream) {
    NMB_REQUIRE(n_bytes >= 0 && value >= 0 && value <= 255 && capacity >= 0, "nmb_index_bytes: bad arguments");
    NMB_REQUIRE(n_out && scratch, "nmb_index_bytes: null argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (n_bytes == 0) {
        NMB_CUDA(cudaMemsetAsync(n_out, 0, sizeof(int64_t), s));
        return NMB_OK;
    }
    NMB_REQUIRE(src, "nmb_index_bytes: null source");
    const int64_t n_blocks = (n_bytes + nmb::kIndexBlockBytes - 1) / nmb::kIndexBlockBytes;
    NMB_REQUIRE(n_blocks < (1ll << 31), "nmb_index_bytes: buffer too large for one call");
    nmb::count_bytes_kernel<<<(unsigned)n_blocks, nmb::kIndexThreads, 0, s>>>(src, n_bytes, (uint8_t)value, scratch);
    NMB_CUDA(cudaGetLastError());
    nmb::scan_counts_kernel<1024><<<1, 1024, 0, s>>>(scratch, n_blocks, n_out);
    NMB_CUDA(cudaGetLastError());
    if (capacity > 0) {
        NMB_REQUIRE(out_index, "nmb_index_bytes: null output");
        nmb::write_byte_index_kernel<<<(unsigned)n_blocks, nmb::kIndexThreads, 0, s>>>(src, n_bytes, (uint8_t)value,
                                                                                     scratch, out_index, capacity);
        NMB_CUDA(cudaGetLastError());
    }
    return NMB_OK;
}

int nmb_bed_parse(const uint8_t *text, int64_t n_bytes, const int64_t *newline_pos, int64_t n_lines,
                  const uint64_t *contig_hash, const int32_t *contig_ids, const int64_t *contig_name_off,
                  const uint8_t *contig_names, int32_t n_contigs, const uint64_t *modtype_keys, int32_t n_modtypes,
                  int32_t *contig_id, int64_t *position, uint8_t *strand, uint8_t *mod_type, int64_t *n_valid_cov,
                  double *fraction_mod, uint16_t *percent_x100, int64_t *n_mod, int64_t *n_diff, int32_t *status,
                  void *stream) {
    NMB_REQUIRE(n_bytes >= 0 && n_lines >= 0 && n_contigs >= 0 && n_modtypes >= 0 && n_modtypes < 255,
                "nmb_bed_parse: bad sizes");
    NMB_REQUIRE(status, "nmb_bed_parse: null status");
    cudaStream_t s = (cudaStream_t)stream;
    NMB_CUDA(cudaMemsetAsync(status, 0, 4 * sizeof(int32_t), s));
    if (n_lines == 0) return NMB_OK;
    NMB_REQUIRE(text && (n_lines == 1 || newline_pos), "nmb_bed_parse: null input");
    NMB_REQUIRE(n_contigs == 0 || (contig_hash && contig_ids && contig_name_off && contig_names),
                "nmb_bed_parse: null contig table");
    NMB_REQUIRE(n_modtypes == 0 || modtype_keys, "nmb_bed_parse: null mod type table");
    NMB_REQUIRE(contig_id && position && strand && mod_type && n_valid_cov && fraction_mod && percent_x100,
                "nmb_bed_parse: null output column");
    nmb::NameTable t{contig_hash, contig_ids, contig_name_off, contig_names, n_contigs};
    nmb::BedColumns o{contig_id, position, strand, mod_type, n_valid_cov, fraction_mod, percent_x100, n_mod, n_diff};
    nmb::bed_parse_kernel<<<(unsigned)((n_lines + 127) / 128), 128, 0, s>>>(text, n_bytes, newline_pos, n_lines, t,
                                                                           modtype_keys, n_modtypes, o, status);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_fasta_lines(const uint8_t *text, int64_t n_bytes, const int64_t *newline_pos, int64_t n_newlines,
                    int64_t n_lines, int32_t want_headers, uint8_t *kind, int64_t *payload, void *stream) {
    NMB_REQUIRE(n_bytes >= 0 && n_lines >= 0 && n_newlines >= 0, "nmb_fasta_lines: bad sizes");
    if (n_lines == 0) return NMB_OK;
    NMB_REQUIRE(text && kind && payload && (n_newlines == 0 || newline_pos), "nmb_fasta_lines: null argument");
    nmb::fasta_lines_kernel<<<(unsigned)((n_lines + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        text, n_bytes, newline_pos, n_newlines, n_lines, want_headers, kind, payload);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_fasta_copy(const uint8_t *text, int64_t n_bytes, const int64_t *newline_pos, int64_t n_newlines,
                   int64_t n_lines, int32_t want_headers, const int64_t *out_off, uint8_t *out, void *stream) {
    NMB_REQUIRE(n_bytes >= 0 && n_lines >= 0 && n_newlines >= 0, "nmb_fasta_copy: bad sizes");
    if (n_lines == 0) return NMB_OK;
    NMB_REQUIRE(text && out_off && out && (n_newlines == 0 || newline_pos), "nmb_fasta_copy: null argument");
    int64_t blocks = (n_lines + 7) / 8;
    if (blocks > 148 * 32) blocks = 148 * 32;
    nmb::fasta_copy_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(text, n_bytes, newline_pos, n_newlines,
                                                                              n_lines, want_headers, out_off, out);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_exclusive_scan_i64(int64_t *values, int64_t n, int64_t *total, void *stream) {
    NMB_REQUIRE(values && total && n >= 0, "nmb_exclusive_scan_i64: bad argument");
    nmb::scan_counts_kernel<1024><<<1, 1024, 0, (cudaStream_t)stream>>>(values, n, total);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_gather_rows(const void *src, int32_t elem_bytes, const int64_t *index, int64_t n, void *dst, void *stream) {
    NMB_REQUIRE(n >= 0, "nmb_gather_rows: n=%lld", (long long)n);
    if (n == 0) return NMB_OK;
    NMB_REQUIRE(src && index && dst, "nmb_gather_rows: null argument");
    cudaStream_t s = (cudaStream_t)stream;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 32) blocks = 148 * 32;
    switch (elem_bytes) {
        case 1: nmb::gather_rows_kernel<uint8_t><<<(unsigned)blocks, 256, 0, s>>>((const uint8_t *)src, index, n, (uint8_t *)dst); break;
        case 2: nmb::gather_rows_kernel<uint16_t><<<(unsigned)blocks, 256, 0, s>>>((const uint16_t *)src, index, n, (uint16_t *)dst); break;
        case 4: nmb::gather_rows_kernel<uint32_t><<<(unsigned)blocks, 256, 0, s>>>((const uint32_t *)src, index, n, (uint32_t *)dst); break;
        case 8: nmb::gather_rows_kernel<uint64_t><<<(unsigned)blocks, 256, 0, s>>>((const uint64_t *)src, index, n, (uint64_t *)dst); break;
        default: NMB_FAIL(NMB_ERR_INVALID, "nmb_gather_rows: elem_bytes=%d not in {1,2,4,8}", elem_bytes);
    }
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

int nmb_lookup_strings(const uint8_t *data, const void *offsets, int32_t offset_bytes, int64_t n_rows,
                       const uint64_t *name_hash, const int32_t *name_ids, const int64_t *name_off,
                       const uint8_t *names, int32_t n_names, int32_t missing, void *out, int32_t out_bytes,
                       void *stream) {
    NMB_REQUIRE(n_rows >= 0 && n_names >= 0, "nmb_lookup_strings: bad sizes");
    NMB_REQUIRE((offset_bytes == 4 || offset_bytes == 8) && (out_bytes == 1 || out_bytes == 4),
                "nmb_lookup_strings: offsets must be 4 or 8 bytes wide, outputs 1 or 4");
    if (n_rows == 0) return NMB_OK;
    NMB_REQUIRE(offsets && out && (n_names == 0 || (name_hash && name_ids && name_off && names)),
                "nmb_lookup_strings: null argument");
    nmb::NameTable t = {name_hash, name_ids, name_off, names, n_names};
    const unsigned blocks = (unsigned)((n_rows + 255) / 256);
    cudaStream_t s = (cudaStream_t)stream;
    if (offset_bytes == 4 && out_bytes == 4)
        nmb::lookup_strings_kernel<int32_t, int32_t><<<blocks, 256, 0, s>>>(data, (const int32_t *)offsets, n_rows, t, missing, (int32_t *)out);
    else if (offset_bytes == 4)
        nmb::lookup_strings_kernel<int32_t, uint8_t><<<blocks, 256, 0, s>>>(data, (const int32_t *)offsets, n_rows, t, missing, (uint8_t *)out);
    else if (out_bytes == 4)
        nmb::lookup_strings_kernel<int64_t, int32_t><<<blocks, 256, 0, s>>>(data, (const int64_t *)offsets, n_rows, t, missing, (int32_t *)out);
    else
        nmb::lookup_strings_kernel<int64_t, uint8_t><<<blocks, 256, 0, s>>>(data, (const int64_t *)offsets, n_rows, t, missing, (uint8_t *)out);
    NMB_CUDA(cudaGetLastError());
    return NMB_OK;
}

}  // extern "C"
