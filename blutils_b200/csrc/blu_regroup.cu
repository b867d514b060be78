// blu_regroup.cu -- regrouping of a non-contiguous hit table by query id, on the GPU.
//
// The reference groups the joined rows through a HashMap<String, Vec<BlastResultRow>> (build_consensus_identities/mod.rs:145,192):
// the rows of one query need not be adjacent in the file; what the consensus of a query depends on is the file order of ITS
// rows.  The streaming pipeline (blu_kernels.cu) wants every query's rows adjacent, so a table in which a query id occurs in
// two separate runs (dup_kernel finds that) is first rewritten: queries in order of first appearance, rows of a query in
// file order, blank lines dropped, every row terminated by '\n'.  Pure data movement -- no field is parsed here:
//
//   row starts      two passes over the text (count per tile, exclusive scan, emit), 16 bytes per thread
//   row keys        one thread per row: length of the row, length and 64-bit hash of its first field
//   first row       open-addressing table keyed by the hash: slot.min_row = the first row with that id (atomicMin); every
//                   row then compares its id BYTES with that row's, so a hash collision is detected (the host path takes
//                   over), never silently merged
//   order           stable radix sort of the rows by "first row of my query" (blu_sort.cu)
//   copy            exclusive scan of the row lengths in the new order, one warp per row copies it to its place
//
// Everything stays in HBM; the regrouped text is handed to the normal device-resident pipeline.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <chrono>

#include <cub/device/device_scan.cuh>

#include "blu_sort.h"

// (declared in blu_kernels.h; that header pulls in the device core, which this file does not need)

namespace blu {
namespace {

constexpr int kRgThreads = 256;
constexpr int kRgItems = 4;                                // 16-byte units per thread
constexpr uint64_t kRgTile = (uint64_t)kRgThreads * kRgItems * 16;  // bytes per CTA

// Row starts among the 16 bytes [idx0, idx0 + 16) of the text (idx0 may be negative / run past n: the text pointer is aligned
// down to 16 bytes): bit k = byte idx0 + k is text, is not a newline, and the byte in front of it is a newline or nothing.
__device__ __forceinline__ uint32_t start_mask16(const uint8_t* base, long long idx0, uint64_t n, const uint8_t* text) {
    if (idx0 >= (long long)n || idx0 + 16 <= 0) return 0u;
    const uint4 v = *reinterpret_cast<const uint4*>(base);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    uint32_t nl = 0;
#pragma unroll
    for (int k = 0; k < 16; k++) nl |= (((w[k >> 2] >> ((k & 3) * 8)) & 0xFFu) == (uint32_t)'\n' ? 1u : 0u) << k;
    uint32_t valid = 0xFFFFu;
    if (idx0 < 0) valid &= 0xFFFFu << (int)(-idx0);
    if (idx0 + 16 > (long long)n) valid &= 0xFFFFu >> (int)(idx0 + 16 - (long long)n);
    const uint32_t prev_nl = idx0 <= 0 ? 1u : (text[idx0 - 1] == '\n' ? 1u : 0u);
    uint32_t before = ((nl << 1) | prev_nl) & 0xFFFFu;
    if (idx0 < 0) before |= 1u << (int)(-idx0);  // the first byte of the text follows "nothing"
    return ~nl & before & valid;
}

__global__ void __launch_bounds__(kRgThreads) rg_count_kernel(const uint8_t* text, uint64_t n, int mis, unsigned long long* tile_cnt) {
    const uint8_t* base0 = text - mis;
    const uint64_t unit0 = ((uint64_t)blockIdx.x * kRgThreads + threadIdx.x) * kRgItems;
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < kRgItems; i++) {
        const uint64_t u = unit0 + i;
        c += __popc(start_mask16(base0 + u * 16, (long long)(u * 16) - mis, n, text));
    }
    __shared__ uint32_t warp_sum[kRgThreads / 32];
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int i = 0; i < kRgThreads / 32; i++) t += warp_sum[i];
        tile_cnt[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(kRgThreads) rg_emit_kernel(const uint8_t* text, uint64_t n, int mis, const unsigned long long* tile_base, uint64_t* row_off) {
    const uint8_t* base0 = text - mis;
    const uint64_t unit0 = ((uint64_t)blockIdx.x * kRgThreads + threadIdx.x) * kRgItems;
    uint32_t m[kRgItems];
    uint32_t c = 0;
#pragma unroll
    for (int i = 0; i < kRgItems; i++) {
        const uint64_t u = unit0 + i;
        m[i] = start_mask16(base0 + u * 16, (long long)(u * 16) - mis, n, text);
        c += __popc(m[i]);
    }
    // exclusive scan of the thread counts over the CTA
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = c;
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    __shared__ uint32_t warp_tot[kRgThreads / 32];
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    uint32_t before = 0;
    for (int i = 0; i < warp; i++) before += warp_tot[i];
    uint64_t pos = tile_base[blockIdx.x] + (uint64_t)(before + inc - c);
#pragma unroll
    for (int i = 0; i < kRgItems; i++) {
        uint32_t mm = m[i];
        const long long idx0 = (long long)((unit0 + i) * 16) - mis;
        while (mm) {
            const int k = __ffs(mm) - 1;
            mm &= mm - 1;
            row_off[pos++] = (uint64_t)(idx0 + k);
        }
    }
}

__device__ __forceinline__ uint64_t fmix64(uint64_t h) {
    h ^= h >> 33;
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    h *= 0xc4ceb9fe1a85ec53ull;
    h ^= h >> 33;
    return h;
}

// one thread per row: its length (without the newline), the length and the hash of its first field
__global__ void rg_key_kernel(const uint8_t* text, uint64_t n, const uint64_t* row_off, uint32_t n_rows, uint64_t* hash, uint32_t* len, uint32_t* qlen,
                              int* too_long) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const uint64_t off = row_off[r];
    uint64_t e = r + 1 < n_rows ? row_off[r + 1] : n;
    while (e > off && text[e - 1] == '\n') e--;  // the row's own newline and blank lines behind it
    if (e - off > 0x7FFFFFFFull) {
        *too_long = 1;
        e = off + 0x7FFFFFFFull;
    }
    const uint32_t l = (uint32_t)(e - off);
    uint64_t h = 0xcbf29ce484222325ull;
    uint32_t q = 0;
    for (; q < l; q++) {
        const uint8_t c = text[off + q];
        if (c == '\t') break;
        h = (h ^ (uint64_t)c) * 0x100000001b3ull;
    }
    h = fmix64(h ^ ((uint64_t)q << 40));
    hash[r] = h ? h : 1ull;
    len[r] = l;
    qlen[r] = q;
}

__global__ void rg_insert_kernel(const uint64_t* hash, uint32_t n_rows, unsigned long long* tab_hash, uint32_t* tab_min, uint64_t mask) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const unsigned long long h = hash[r];
    for (uint64_t s = h & mask;; s = (s + 1) & mask) {
        const unsigned long long cur = atomicCAS(&tab_hash[s], 0ull, h);
        if (cur == 0ull || cur == h) {
            atomicMin(&tab_min[s], r);
            return;
        }
    }
}

// first[r] = first row with the id of row r; the ids are compared byte by byte (a hash collision raises the flag)
__global__ void rg_lookup_kernel(const uint8_t* text, const uint64_t* row_off, const uint64_t* hash, const uint32_t* qlen, uint32_t n_rows,
                                 const unsigned long long* tab_hash, const uint32_t* tab_min, uint64_t mask, uint32_t* first, uint32_t* iota, int* collided) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const unsigned long long h = hash[r];
    uint64_t s = h & mask;
    while (tab_hash[s] != h) s = (s + 1) & mask;
    const uint32_t f = tab_min[s];
    if (f != r) {
        const uint32_t q = qlen[r];
        bool same = qlen[f] == q;
        const uint8_t *a = text + row_off[r], *b = text + row_off[f];
        for (uint32_t i = 0; same && i < q; i++) same = a[i] == b[i];
        if (!same) *collided = 1;
    }
    first[r] = f;
    iota[r] = r;
}

__global__ void rg_len_kernel(const uint32_t* order, const uint32_t* len, uint32_t n_rows, uint64_t* slen) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_rows) slen[i] = (uint64_t)len[order[i]] + 1ull;
}

// one warp per row of the new order: copies the row and terminates it
__global__ void rg_copy_kernel(const uint8_t* text, const uint64_t* row_off, const uint32_t* len, const uint32_t* order, const uint64_t* dst, uint32_t n_rows,
                               uint8_t* out) {
    const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // (64-bit: 32 threads per row)
    const int lane = threadIdx.x & 31;
    if (i >= n_rows) return;
    const uint32_t r = order[i];
    const uint8_t* src = text + row_off[r];
    uint8_t* d = out + dst[i];
    const uint32_t l = len[r];
    for (uint32_t k = lane; k < l; k += 32) d[k] = src[k];
    if (lane == 0) d[l] = '\n';
}

// BLU_REGROUP_TRACE=1: wall time of every stage on stderr (the stream is synchronised at each mark: measurement only)
struct Trace {
    bool on;
    cudaStream_t s;
    std::chrono::steady_clock::time_point t0;
    explicit Trace(cudaStream_t st) : on(getenv("BLU_REGROUP_TRACE") != nullptr), s(st), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what) {
        if (!on) return;
        cudaStreamSynchronize(s);
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[blu regroup] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

struct Scratch {
    void* p[24];
    int n = 0;
    template <typename T>
    bool alloc(T** out, size_t count) {
        void* q = nullptr;
        if (cudaMalloc(&q, count * sizeof(T) + 256) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        p[n++] = q;
        *out = (T*)q;
        return true;
    }
    ~Scratch() {
        for (int i = 0; i < n; i++) cudaFree(p[i]);
    }
};

}  // namespace

// 0: done (*d_out = cudaMalloc'ed regrouped text, padded; the caller frees it); 1: not possible here (memory, 2^31 rows or
// more, a row of 2 GB, two ids with one hash) -- the caller regroups on the host; < 0: a CUDA error (cudaError_t negated).
int regroup_device(const uint8_t* d_text, uint64_t n, cudaStream_t s, uint8_t** d_out, uint64_t* out_n, uint64_t* n_rows_out) {
    *d_out = nullptr;
    *out_n = 0;
    if (n == 0) return 1;
#define RG_CK(x)                                 \
    do {                                         \
        cudaError_t e_ = (x);                    \
        if (e_ != cudaSuccess) return -(int)e_;  \
    } while (0)
    Scratch sc;
    Trace tr(s);
    const int mis = (int)((uintptr_t)d_text & 15);
    const uint64_t n_tiles64 = (n + (uint64_t)mis + kRgTile - 1) / kRgTile;
    if (n_tiles64 > 0x7FFFFFFFull) return 1;
    const uint32_t n_tiles = (uint32_t)n_tiles64;
    unsigned long long *tile_cnt, *tile_base;
    if (!sc.alloc(&tile_cnt, n_tiles + 1) || !sc.alloc(&tile_base, n_tiles + 1)) return 1;
    rg_count_kernel<<<n_tiles, kRgThreads, 0, s>>>(d_text, n, mis, tile_cnt);
    RG_CK(cudaGetLastError());
    // exclusive scan of the tile counts (n_tiles + 1 elements: the last one is the number of rows)
    RG_CK(cudaMemsetAsync(tile_cnt + n_tiles, 0, sizeof(unsigned long long), s));
    size_t tmp_bytes = 0;
    RG_CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, tile_cnt, tile_base, (int)(n_tiles + 1), s));
    uint8_t* tmp;
    if (!sc.alloc(&tmp, tmp_bytes)) return 1;
    RG_CK(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, tile_cnt, tile_base, (int)(n_tiles + 1), s));
    unsigned long long n_rows64 = 0;
    RG_CK(cudaMemcpyAsync(&n_rows64, tile_base + n_tiles, sizeof(n_rows64), cudaMemcpyDeviceToHost, s));
    RG_CK(cudaStreamSynchronize(s));
    tr.mark("count rows + scan");
    if (n_rows64 > 0x7FFFFFFFull) return 1;  // (row numbers are 32-bit here; larger tables take the host path)
    const uint32_t n_rows = (uint32_t)n_rows64;
    if (n_rows == 0) return 1;
    *n_rows_out = n_rows;

    // memory: ~60 bytes per row + the hash table + the output
    uint64_t cap = 1024;
    while (cap < 2ull * n_rows) cap <<= 1;
    {
        size_t free_b = 0, total_b = 0;
        RG_CK(cudaMemGetInfo(&free_b, &total_b));
        const uint64_t need = (uint64_t)n_rows * 72ull + cap * 12ull + n + (64ull << 20);
        if (need > (uint64_t)(free_b * 0.9)) return 1;
    }
    uint64_t *row_off, *hash, *slen, *dst;
    uint32_t *len, *qlen, *first, *first_sorted, *iota, *order, *tab_min;
    unsigned long long* tab_hash;
    int* flags;
    if (!sc.alloc(&row_off, (size_t)n_rows + 1) || !sc.alloc(&hash, n_rows) || !sc.alloc(&len, n_rows) || !sc.alloc(&qlen, n_rows) ||
        !sc.alloc(&first, n_rows) || !sc.alloc(&first_sorted, n_rows) || !sc.alloc(&iota, n_rows) || !sc.alloc(&order, n_rows) || !sc.alloc(&tab_hash, cap) ||
        !sc.alloc(&tab_min, cap) || !sc.alloc(&flags, 2))
        return 1;
    tr.mark("allocate");
    RG_CK(cudaMemsetAsync(flags, 0, 2 * sizeof(int), s));
    RG_CK(cudaMemsetAsync(tab_hash, 0, cap * sizeof(unsigned long long), s));
    RG_CK(cudaMemsetAsync(tab_min, 0xFF, cap * sizeof(uint32_t), s));
    tr.mark("clear table");
    rg_emit_kernel<<<n_tiles, kRgThreads, 0, s>>>(d_text, n, mis, tile_base, row_off);
    tr.mark("emit row starts");
    const uint32_t rb = (n_rows + 255) / 256;
    rg_key_kernel<<<rb, 256, 0, s>>>(d_text, n, row_off, n_rows, hash, len, qlen, flags + 1);
    tr.mark("row keys");
    rg_insert_kernel<<<rb, 256, 0, s>>>(hash, n_rows, tab_hash, tab_min, cap - 1);
    tr.mark("insert");
    rg_lookup_kernel<<<rb, 256, 0, s>>>(d_text, row_off, hash, qlen, n_rows, tab_hash, tab_min, cap - 1, first, iota, flags);
    RG_CK(cudaGetLastError());
    int h_flags[2] = {0, 0};
    RG_CK(cudaMemcpyAsync(h_flags, flags, sizeof(h_flags), cudaMemcpyDeviceToHost, s));
    RG_CK(cudaStreamSynchronize(s));
    tr.mark("lookup + verify");
    if (h_flags[0] || h_flags[1]) return 1;

    // stable sort of the rows by the first row of their query
    int bits = 1;
    while (bits < 32 && (1ull << bits) < (uint64_t)n_rows) bits++;
    uint8_t* sort_tmp;
    if (!sc.alloc(&sort_tmp, radix_sort_scratch_bytes(n_rows))) return 1;
    bool in_alt = false;
    RG_CK(radix_sort_pairs_u32(first, first_sorted, iota, order, n_rows, bits, sort_tmp, s, &in_alt));
    if (!in_alt) order = iota;
    tr.mark("sort");
    // where every row goes
    if (!sc.alloc(&slen, n_rows) || !sc.alloc(&dst, n_rows)) return 1;
    rg_len_kernel<<<rb, 256, 0, s>>>(order, len, n_rows, slen);
    size_t scan_bytes = 0;
    RG_CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, slen, dst, (int)n_rows, s));
    uint8_t* scan_tmp;
    if (!sc.alloc(&scan_tmp, scan_bytes)) return 1;
    RG_CK(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, slen, dst, (int)n_rows, s));
    uint64_t tail[2] = {0, 0};
    RG_CK(cudaMemcpyAsync(&tail[0], dst + (n_rows - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    RG_CK(cudaMemcpyAsync(&tail[1], slen + (n_rows - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
    RG_CK(cudaStreamSynchronize(s));
    tr.mark("destinations");
    const uint64_t total = tail[0] + tail[1];
    uint8_t* out = nullptr;
    if (cudaMalloc((void**)&out, total + 512) != cudaSuccess) {
        cudaGetLastError();
        return 1;
    }
    cudaError_t e = cudaMemsetAsync(out + total, 0, 512, s);
    if (e == cudaSuccess) {
        const uint64_t threads = (uint64_t)n_rows * 32ull;
        rg_copy_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(d_text, row_off, len, order, dst, n_rows, out);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {
        cudaFree(out);
        return -(int)e;
    }
    tr.mark("copy rows");
    *d_out = out;
    *out_n = total;
    return 0;
#undef RG_CK
}

}  // namespace blu
