// blu_sort.cu -- stable radix sort on the GPU, and the ordering of result records by query id built on it.
//
// Radix sort (LSD, 8-bit digits, one-sweep design):
//   histogram   one kernel counts the digits of every digit position of all keys at once; the host reads the counts, turns
//               them into the global offset of every digit and skips the positions at which every key has the same digit
//   pass        per digit position one kernel: a tile of 4096 keys takes its number from an atomic counter (tiles are then
//               started in number order, so the look-back below always makes progress), ranks its keys stably with
//               __match_any_sync per warp, publishes its digit counts and finds the counts of all tiles before it through a
//               decoupled look-back (one 64-bit status word per tile and digit: flag + value), then scatters
//
// Order of query ids (write_blutils_output.rs:111 sorts by `query`, bytewise):
//   an id is cut into 8-byte chunks, big-endian and zero-padded; chunk k carries a tag: the number of the id's bytes in it
//   (0..8) when the id ends there, 9 when it goes on.  (chunk, tag) compares like the bytes themselves, a prefix first.
//   level 0     every id is sorted by (chunk 0, tag 0)
//   level k     runs of equal (chunk, tag 9) are groups whose order is still open; their members are compacted (group
//               number = rank of the run) and sorted by (group, chunk k, tag k), and so on until no group is left.  Ids that
//               share long prefixes (read names, numbered ids) are the normal case: the members shrink level by level.
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "blu_sort.h"

namespace blu {
namespace {

constexpr int kThreads = 256;  // one thread per digit value in the look-back
constexpr int kWarps = kThreads / 32;
constexpr int kItems = 16;
constexpr uint32_t kTileItems = kThreads * kItems;
constexpr uint64_t kFlagAggregate = 1ull << 62, kFlagPrefix = 2ull << 62, kValueMask = (1ull << 62) - 1;
constexpr size_t kHistBytes = 8 * 256 * sizeof(uint32_t);
constexpr size_t kStatusOffset = 2 * kHistBytes + 256;  // histogram, global offsets, tile counter, then the status words

#define SK(x)                                   \
    do {                                        \
        const cudaError_t e_ = (x);             \
        if (e_ != cudaSuccess) return e_;       \
    } while (0)

__device__ __forceinline__ uint32_t lanemask_lt() { return (1u << (threadIdx.x & 31)) - 1u; }

template <class K>
__global__ void __launch_bounds__(kThreads) hist_kernel(const K* keys, uint32_t n, int n_pos, uint32_t* hist) {
    __shared__ uint32_t sh[8 * 256];
    for (int i = threadIdx.x; i < n_pos * 256; i += kThreads) sh[i] = 0;
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * kThreads;
    // warp-uniform loop: __match_any_sync needs every lane
    for (uint64_t i0 = (uint64_t)blockIdx.x * kThreads + (threadIdx.x & ~31u); i0 < n; i0 += stride) {
        const uint64_t i = i0 + (threadIdx.x & 31);
        const bool ok = i < n;
        const K k = ok ? keys[i] : (K)0;
        for (int p = 0; p < n_pos; p++) {
            const uint32_t d = ok ? (uint32_t)(k >> (8 * p)) & 0xFFu : 256u;
            const uint32_t peers = __match_any_sync(0xffffffffu, d);
            if (ok && (peers & lanemask_lt()) == 0) atomicAdd(&sh[p * 256 + d], (uint32_t)__popc(peers));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_pos * 256; i += kThreads)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// One digit position.  Warp w of a tile owns the keys [w * 32 * kItems, (w + 1) * 32 * kItems) of the tile, round j lane l the
// key j * 32 + l of that range: the rank of a key among the equal digits before it is the warp's count so far plus the equal
// lanes below it.
template <class K>
__global__ void __launch_bounds__(kThreads) pass_kernel(const K* kin, K* kout, const uint32_t* vin, uint32_t* vout, uint32_t n, int shift,
                                                        const uint32_t* gofs, uint32_t* tile_counter, uint64_t* status) {
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp[kWarps][256];
    __shared__ uint32_t s_base[256];
    if (threadIdx.x == 0) s_tile = atomicAdd(tile_counter, 1u);
    for (int i = threadIdx.x; i < kWarps * 256; i += kThreads) (&s_warp[0][0])[i] = 0;
    __syncthreads();
    const uint32_t tile = s_tile;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t first = (uint64_t)tile * kTileItems + (uint64_t)warp * 32 * kItems;
    K k[kItems];
    uint32_t v[kItems], rd[kItems];  // rd: rank in the warp's range | digit << 16 (digit 256: no key)
#pragma unroll
    for (int j = 0; j < kItems; j++) {
        const uint64_t i = first + (uint64_t)j * 32 + lane;
        const bool ok = i < n;
        k[j] = ok ? kin[i] : (K)0;
        v[j] = ok ? vin[i] : 0u;
        const uint32_t d = ok ? (uint32_t)(k[j] >> shift) & 0xFFu : 256u;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t before = ok ? s_warp[warp][d] : 0u;
        __syncwarp();
        if (ok && (peers & lanemask_lt()) == 0) s_warp[warp][d] = before + (uint32_t)__popc(peers);
        __syncwarp();
        rd[j] = (before + (uint32_t)__popc(peers & lanemask_lt())) | (d << 16);
    }
    __syncthreads();
    // thread d: digit d -- warp offsets inside the tile, the tile's count, then the counts of the tiles before it
    const uint32_t d = threadIdx.x;
    uint32_t cnt = 0;
    for (int w = 0; w < kWarps; w++) {
        const uint32_t c = s_warp[w][d];
        s_warp[w][d] = cnt;
        cnt += c;
    }
    volatile uint64_t* st = status;
    uint64_t excl = 0;
    if (tile > 0) {
        st[(uint64_t)tile * 256 + d] = kFlagAggregate | cnt;
        for (int64_t t = (int64_t)tile - 1; t >= 0;) {
            const uint64_t w = st[(uint64_t)t * 256 + d];
            if (w == 0) continue;  // tile t has not published yet
            excl += w & kValueMask;
            if (w & kFlagPrefix) break;
            t--;
        }
    }
    st[(uint64_t)tile * 256 + d] = kFlagPrefix | (excl + cnt);
    s_base[d] = gofs[d] + (uint32_t)excl;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kItems; j++) {
        const uint32_t dj = rd[j] >> 16;
        if (dj < 256) {
            const uint32_t pos = s_base[dj] + s_warp[warp][dj] + (rd[j] & 0xFFFFu);
            kout[pos] = k[j];
            vout[pos] = v[j];
        }
    }
}

uint32_t n_tiles(uint32_t n) { return n ? (uint32_t)(((uint64_t)n + kTileItems - 1) / kTileItems) : 1u; }

// Stable sort of (k[cur], v[cur]) by the low `bits` bits; `cur` names the buffer pair holding the result afterwards.
template <class K>
cudaError_t radix_stage(K* k[2], uint32_t* v[2], int& cur, uint32_t n, int bits, uint8_t* scratch, cudaStream_t s) {
    if (n <= 1) return cudaSuccess;
    int n_pos = (bits + 7) / 8;
    if (n_pos > (int)sizeof(K)) n_pos = (int)sizeof(K);
    uint32_t* hist = (uint32_t*)scratch;
    uint32_t* gofs = (uint32_t*)(scratch + kHistBytes);
    uint32_t* counter = (uint32_t*)(scratch + 2 * kHistBytes);
    uint64_t* status = (uint64_t*)(scratch + kStatusOffset);
    const uint32_t tiles = n_tiles(n);
    SK(cudaMemsetAsync(hist, 0, (size_t)n_pos * 256 * sizeof(uint32_t), s));
    int dev = 0, sms = 148;
    SK(cudaGetDevice(&dev));
    SK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const uint32_t hgrid = tiles < (uint32_t)sms * 8 ? tiles : (uint32_t)sms * 8;
    hist_kernel<K><<<hgrid, kThreads, 0, s>>>(k[cur], n, n_pos, hist);
    SK(cudaGetLastError());
    uint32_t h[8 * 256], go[8 * 256];
    SK(cudaMemcpyAsync(h, hist, (size_t)n_pos * 256 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    SK(cudaStreamSynchronize(s));
    bool active[8];
    for (int p = 0; p < n_pos; p++) {
        uint32_t sum = 0;
        active[p] = true;
        for (int d = 0; d < 256; d++) {
            if (h[p * 256 + d] == n) active[p] = false;  // every key has this digit: the pass would not move anything
            go[p * 256 + d] = sum;
            sum += h[p * 256 + d];
        }
    }
    // (pageable source: the copy is staged before the call returns)
    SK(cudaMemcpyAsync(gofs, go, (size_t)n_pos * 256 * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    for (int p = 0; p < n_pos; p++) {
        if (!active[p]) continue;
        SK(cudaMemsetAsync(counter, 0, kStatusOffset - 2 * kHistBytes + (size_t)tiles * 256 * sizeof(uint64_t), s));
        pass_kernel<K><<<tiles, kThreads, 0, s>>>(k[cur], k[cur ^ 1], v[cur], v[cur ^ 1], n, 8 * p, gofs + p * 256, counter, status);
        SK(cudaGetLastError());
        cur ^= 1;
    }
    return cudaSuccess;
}

// --- ids ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t id_tag(uint32_t len, uint32_t level) {
    const uint64_t b = (uint64_t)level * 8;
    const uint64_t rem = len > b ? len - b : 0;
    return rem <= 8 ? (uint32_t)rem : 9u;
}

__device__ __forceinline__ uint64_t id_chunk(const uint8_t* base, uint64_t off, uint32_t len, uint32_t level) {
    const uint64_t b = (uint64_t)level * 8;
    const uint64_t rem = len > b ? len - b : 0;
    const uint8_t* p = base + off + b;
    uint64_t c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) c = (c << 8) | (uint64_t)((uint64_t)i < rem ? p[i] : 0);
    return c;
}

// level 0: every id is a member, in index order, of group 0
__global__ void level0_kernel(uint32_t n, uint32_t* pos, uint32_t* rec, uint32_t* grp) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    pos[i] = rec[i] = (uint32_t)i;
    grp[i] = 0;
}

__global__ void key_tag_kernel(const uint32_t* m_rec, uint32_t m, const uint32_t* len, uint32_t level, uint64_t* keys, uint32_t* vals) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    keys[j] = id_tag(len[m_rec[j]], level);
    vals[j] = (uint32_t)j;
}

__global__ void key_chunk_kernel(const uint32_t* vals, const uint32_t* m_rec, uint32_t m, const uint8_t* base, const uint64_t* off, const uint32_t* len,
                                 uint32_t level, uint64_t* keys) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t r = m_rec[vals[j]];
    keys[j] = id_chunk(base, off[r], len[r], level);
}

__global__ void key_group_kernel(const uint32_t* vals, const uint32_t* m_g, uint32_t m, uint64_t* keys) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m) keys[j] = m_g[vals[j]];
}

// The members in their new order: the j-th goes to position m_pos[j] (the members of a group hold consecutive positions and
// the groups are numbered in position order).  Their (group, chunk, tag) are kept for the next level's groups.
__global__ void emit_kernel(const uint32_t* vals, uint32_t m, const uint32_t* m_pos, const uint32_t* m_rec, const uint32_t* m_g, const uint8_t* base,
                            const uint64_t* off, const uint32_t* len, uint32_t level, uint32_t* perm, uint32_t* t_rec, uint32_t* t_g, uint64_t* t_ck,
                            uint8_t* t_tag) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const uint32_t mi = vals[j];
    const uint32_t r = m_rec[mi];
    perm[m_pos[j]] = r;
    t_rec[j] = r;
    t_g[j] = m_g[mi];
    t_ck[j] = id_chunk(base, off[r], len[r], level);
    t_tag[j] = (uint8_t)id_tag(len[r], level);
}

// bit 0: member j is in a group of the next level; bit 32: it starts that group
__device__ __forceinline__ uint64_t member_bits(const uint32_t* g, const uint64_t* ck, const uint8_t* tag, uint32_t m, uint32_t j) {
    if (tag[j] != 9) return 0;
    const bool prev = j > 0 && tag[j - 1] == 9 && ck[j - 1] == ck[j] && g[j - 1] == g[j];
    const bool next = j + 1 < m && tag[j + 1] == 9 && ck[j + 1] == ck[j] && g[j + 1] == g[j];
    if (!prev && !next) return 0;
    return 1ull | ((uint64_t)!prev << 32);
}

constexpr int kScanItems = 16;
constexpr uint32_t kScanTile = kThreads * kScanItems;

__device__ uint64_t block_exclusive_scan(uint64_t x, uint64_t* total) {
    __shared__ uint64_t wsum[kWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t inc = x;
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    uint64_t before = 0, tot = 0;
    for (int w = 0; w < kWarps; w++) {
        if (w < warp) before += wsum[w];
        tot += wsum[w];
    }
    __syncthreads();
    *total = tot;
    return before + inc - x;
}

__global__ void __launch_bounds__(kThreads) scan_sums_kernel(const uint32_t* g, const uint64_t* ck, const uint8_t* tag, uint32_t m, uint64_t* bsum) {
    const uint64_t j0 = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    uint64_t x = 0;
    for (int i = 0; i < kScanItems; i++)
        if (j0 + i < m) x += member_bits(g, ck, tag, m, (uint32_t)(j0 + i));
    uint64_t tot;
    block_exclusive_scan(x, &tot);
    if (threadIdx.x == 0) bsum[blockIdx.x] = tot;
}

// exclusive scan of the tile sums in place; *total = members | groups << 32 of the next level
__global__ void __launch_bounds__(kThreads) scan_tiles_kernel(uint64_t* bsum, uint32_t nb, uint64_t* total) {
    uint64_t carry = 0;
    for (uint32_t b0 = 0; b0 < nb; b0 += kThreads) {
        const uint32_t b = b0 + threadIdx.x;
        const uint64_t x = b < nb ? bsum[b] : 0;
        uint64_t tot;
        const uint64_t e = block_exclusive_scan(x, &tot);
        if (b < nb) bsum[b] = carry + e;
        carry += tot;
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(kThreads) compact_kernel(const uint32_t* m_pos, const uint32_t* t_rec, const uint32_t* t_g, const uint64_t* t_ck,
                                                           const uint8_t* t_tag, uint32_t m, const uint64_t* bofs, uint32_t* n_pos, uint32_t* n_rec,
                                                           uint32_t* n_g) {
    const uint64_t j0 = (uint64_t)blockIdx.x * kScanTile + (uint64_t)threadIdx.x * kScanItems;
    uint64_t bits[kScanItems];
    uint64_t x = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; i++) {
        bits[i] = j0 + i < m ? member_bits(t_g, t_ck, t_tag, m, (uint32_t)(j0 + i)) : 0;
        x += bits[i];
    }
    uint64_t tot;
    uint64_t run = bofs[blockIdx.x] + block_exclusive_scan(x, &tot);
#pragma unroll
    for (int i = 0; i < kScanItems; i++) {
        run += bits[i];  // (inclusive: the group number counts this member's own group start)
        if (bits[i] & 1) {
            const uint32_t o = (uint32_t)run - 1u;
            const uint64_t j = j0 + i;
            n_pos[o] = m_pos[j];
            n_rec[o] = t_rec[j];
            n_g[o] = (uint32_t)(run >> 32) - 1u;
        }
    }
}

__global__ void record_ids_kernel(const blu_record* rec, uint32_t n, uint64_t* off, uint32_t* len) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    off[i] = rec[i].query_off;
    len[i] = rec[i].query_len;
}

// four threads per 64-byte record
__global__ void gather_records_kernel(const blu_record* in, const uint32_t* perm, uint32_t n, blu_record* out) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t i = t >> 2;
    if (i >= n) return;
    const uint4* src = reinterpret_cast<const uint4*>(in + perm[i]);
    uint4* dst = reinterpret_cast<uint4*>(out + i);
    dst[t & 3] = src[t & 3];
}

unsigned blocks_for(uint64_t n, unsigned per_block) { return (unsigned)((n + per_block - 1) / per_block); }

struct IdScratch {
    uint64_t* keys[2];
    uint32_t* vals[2];
    uint32_t *pos[2], *rec[2], *grp[2];
    uint32_t *t_rec, *t_g;
    uint64_t* t_ck;
    uint8_t* t_tag;
    uint64_t *bsum, *total;
    uint8_t* radix;
};

// the layout of sort_ids_device's scratch; base == nullptr only sizes it
uint64_t carve(uint8_t* base, uint64_t n, IdScratch* s) {
    uint64_t at = 0;
    auto take = [&](auto** p, uint64_t count) {
        at = (at + 255) & ~255ull;
        *p = base ? (std::remove_reference_t<decltype(**p)>*)(base + at) : nullptr;
        at += count * sizeof(**p);
    };
    for (int i = 0; i < 2; i++) {
        take(&s->keys[i], n);
        take(&s->vals[i], n);
        take(&s->pos[i], n);
        take(&s->rec[i], n);
        take(&s->grp[i], n);
    }
    take(&s->t_rec, n);
    take(&s->t_g, n);
    take(&s->t_ck, n);
    take(&s->t_tag, n);
    take(&s->bsum, n / kScanTile + 2);
    take(&s->total, 1);
    take(&s->radix, radix_sort_scratch_bytes((uint32_t)n));
    return at + 256;
}

cudaError_t sort_ids_levels(const uint8_t* base, const uint64_t* off, const uint32_t* len, uint32_t n, uint32_t* perm, const IdScratch& S, cudaStream_t s) {
    level0_kernel<<<blocks_for(n, 256), 256, 0, s>>>(n, S.pos[0], S.rec[0], S.grp[0]);
    SK(cudaGetLastError());
    uint64_t* keys[2] = {S.keys[0], S.keys[1]};
    uint32_t* vals[2] = {S.vals[0], S.vals[1]};
    uint32_t m = n;
    int ms = 0;
    for (uint32_t level = 0; m > 0; level++, ms ^= 1) {
        const unsigned mb = blocks_for(m, 256);
        int cur = 0;
        key_tag_kernel<<<mb, 256, 0, s>>>(S.rec[ms], m, len, level, keys[0], vals[0]);
        SK(cudaGetLastError());
        SK(radix_stage<uint64_t>(keys, vals, cur, m, 4, S.radix, s));
        key_chunk_kernel<<<mb, 256, 0, s>>>(vals[cur], S.rec[ms], m, base, off, len, level, keys[cur]);
        SK(cudaGetLastError());
        SK(radix_stage<uint64_t>(keys, vals, cur, m, 64, S.radix, s));
        if (level > 0) {  // (level 0: one group)
            key_group_kernel<<<mb, 256, 0, s>>>(vals[cur], S.grp[ms], m, keys[cur]);
            SK(cudaGetLastError());
            SK(radix_stage<uint64_t>(keys, vals, cur, m, 32, S.radix, s));
        }
        emit_kernel<<<mb, 256, 0, s>>>(vals[cur], m, S.pos[ms], S.rec[ms], S.grp[ms], base, off, len, level, perm, S.t_rec, S.t_g, S.t_ck, S.t_tag);
        SK(cudaGetLastError());
        const uint32_t nb = (uint32_t)(((uint64_t)m + kScanTile - 1) / kScanTile);
        scan_sums_kernel<<<nb, kThreads, 0, s>>>(S.t_g, S.t_ck, S.t_tag, m, S.bsum);
        scan_tiles_kernel<<<1, kThreads, 0, s>>>(S.bsum, nb, S.total);
        compact_kernel<<<nb, kThreads, 0, s>>>(S.pos[ms], S.t_rec, S.t_g, S.t_ck, S.t_tag, m, S.bsum, S.pos[ms ^ 1], S.rec[ms ^ 1], S.grp[ms ^ 1]);
        SK(cudaGetLastError());
        uint64_t total = 0;
        SK(cudaMemcpyAsync(&total, S.total, sizeof total, cudaMemcpyDeviceToHost, s));
        SK(cudaStreamSynchronize(s));
        m = (uint32_t)total;
    }
    return cudaSuccess;
}

}  // namespace

size_t radix_sort_scratch_bytes(uint32_t n) { return kStatusOffset + (size_t)n_tiles(n) * 256 * sizeof(uint64_t); }

cudaError_t radix_sort_pairs_u32(uint32_t* keys, uint32_t* keys_alt, uint32_t* vals, uint32_t* vals_alt, uint32_t n, int bits, void* scratch,
                                 cudaStream_t s, bool* in_alt) {
    uint32_t* k[2] = {keys, keys_alt};
    uint32_t* v[2] = {vals, vals_alt};
    int cur = 0;
    const cudaError_t e = radix_stage<uint32_t>(k, v, cur, n, bits, (uint8_t*)scratch, s);
    *in_alt = cur == 1;
    return e;
}

uint64_t sort_ids_device_bytes(uint64_t n) {
    IdScratch S;
    return carve(nullptr, n, &S);
}

int sort_ids_device(const uint8_t* base, const uint64_t* off, const uint32_t* len, uint32_t n, uint32_t* perm, cudaStream_t s) {
    if (n == 0) return 0;
    IdScratch S;
    const uint64_t bytes = carve(nullptr, n, &S);
    uint8_t* mem = nullptr;
    if (cudaMalloc((void**)&mem, bytes) != cudaSuccess) {
        cudaGetLastError();
        return 1;
    }
    carve(mem, n, &S);
    cudaError_t e = sort_ids_levels(base, off, len, n, perm, S, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    cudaFree(mem);
    return e == cudaSuccess ? 0 : -(int)e;
}

cudaError_t launch_record_ids(const blu_record* rec, uint32_t n, uint64_t* off, uint32_t* len, cudaStream_t s) {
    if (!n) return cudaSuccess;
    record_ids_kernel<<<blocks_for(n, 256), 256, 0, s>>>(rec, n, off, len);
    return cudaGetLastError();
}

cudaError_t launch_gather_records(const blu_record* in, const uint32_t* perm, uint32_t n, blu_record* out, cudaStream_t s) {
    if (!n) return cudaSuccess;
    gather_records_kernel<<<blocks_for((uint64_t)n * 4, 256), 256, 0, s>>>(in, perm, n, out);
    return cudaGetLastError();
}

#undef SK

}  // namespace blu
