// blu_kernels.cu -- hand-written sm_100a kernels of the consensus-identity path.
//
//   tile_kernel    : the dominant kernel (streaming).  Every CTA walks one contiguous segment of the outfmt-6 text in
//                    32 KB windows staged by TMA bulk copies (cp.async.bulk + mbarrier, double-buffered), classifies
//                    the bytes with SIMD-in-register tests (newline / tab / digit bitmasks, dp4a packing), indexes
//                    the rows, validates / parses every row, finds query runs and their top bit-score group --
//                    carrying the unfinished query from window to window -- and emits one record header plus the
//                    parsed top rows per query.  Text is read from HBM once; nothing per-row is written back.
//   consensus_kernel: one warp per query: taxid join, multi-taxa consensus, cutoffs (reads the tile kernel's output).
//   longrun_kernel : block-per-query path for the few queries the tile kernel hands over (top group of more than 32
//                    rows, bit score beyond int32, first row without a predecessor in its window).
//   gather_kernel  : copies query ids and accessions of finished queries into the result's string pool.
//   dup_kernel     : detects a query id that occurs in two separate runs (non-contiguous input).
//   fanout_kernel  : several configurations in one pass: copies the tile kernel's record headers and text cursors from the
//                    first configuration to the others.
//
// Reference semantics: see blu_core.cuh.  Geometry and roofline accounting: DESIGN.md.
#include <cuda_runtime.h>

#include <climits>
#include <cstdio>

#include "blu_kernels.h"

namespace blu {

namespace {

constexpr int kRowCap = kWin / 26 + 16;   // a valid row is >= 26 bytes (13 one-byte fields, 12 tabs, '\n')
constexpr int kLongThreads = 512;
constexpr int kLongWarps = kLongThreads / 32;

// ---------------------------------------------------------------------------------------------------------------
// small PTX wrappers (TMA 1-D bulk copy + mbarrier)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// One shared-memory atomic add, as written: atomicAdd() on shared memory is expanded by the compiler into a warp-aggregated
// sequence (vote, leader election, popc, shuffle: ~12 instructions), which is pure overhead where a single lane -- or a lane
// or two of a diverged warp -- executes it, as everywhere in the tile kernel.
__device__ __forceinline__ uint32_t atoms_add(void* addr, uint32_t v) {
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(addr)), "r"(v) : "memory");
    return old;
}

__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned long long* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// asks the TMA unit to pull [src, src+bytes) into L2 (no destination): the tile after the current one
__device__ __forceinline__ void tma_prefetch_l2(const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

// grammar-class errors (a malformed row, a limit of this implementation hit while scanning): fatal wherever the row sits
__device__ __forceinline__ void report(Counters* ctr, uint32_t err, unsigned long long off) {
    if (atomicCAS(&ctr->err_code, 0u, err) == 0u) ctr->err_off = off;
}
// consensus-class errors (join miss, unparsable lineage, root-level disagreement, empty adjusted taxonomy, a top row's number
// outside the exactly-parsed range): what the reference only meets on the rows of a query's TOP group -- fatal once the
// table is known to be contiguous (a fragment of a scattered query may have a different top group than the merged query)
__device__ __forceinline__ void report_soft(Counters* ctr, uint32_t err, unsigned long long off) {
    if (atomicCAS(&ctr->soft_code, 0u, err) == 0u) ctr->soft_off = off;
}

// ---------------------------------------------------------------------------------------------------------------
// shared-memory window + row index (used by both kernels)
// ---------------------------------------------------------------------------------------------------------------
constexpr int kChunks = (kWin + 128) / 16;  // 16-byte chunks of the window (incl. the spare tail)

struct WindowIndex {
    alignas(128) uint8_t win[kWin + 128];
    // byte-class bitmasks, one bit per window byte (u16 per 16-byte chunk; read back as 64-bit words)
    alignas(8) uint16_t tabm[kChunks + 8];
    alignas(8) uint16_t digm[kChunks + 8];
    // row starts / row ends per chunk (pass 1 of the row scan -> pass 2).  Dead once the row table exists: the tile
    // kernel re-uses the space for the per-row bit scores.
    alignas(8) uint16_t startm[kChunks + 8];
    uint16_t endm[kChunks + 8];
    uint16_t row_s[kRowCap];
    uint16_t row_e[kRowCap + 1];
    int n_starts, n_ends;
    int bad_byte;  // window offset of the first '"' / '\r' byte inside [qlo, qhi), or INT_MAX
    int warp_cnt[32];
};

struct WinGeom {
    unsigned long long lo;  // absolute offset of win[0]
    int vb;                 // first valid byte of the window (everything before it is not text / not loaded)
    int rb;                 // == vb when a row is known to start there (virtual newline in front), else -1
    int re;                 // end - lo   (may exceed the window)
    int loaded;             // bytes staged
    int L;                  // bytes scanned (text end + optional virtual newline)
    bool covers_eof;        // the window contains the end of the text
    int qlo, qhi;           // window range in which a '"' / '\r' byte is this CTA's to report
};

// Stage [lo, lo+bytes) of the text into the window with TMA bulk copies.  All threads call; returns when the
// bytes are visible.  `phase` is the barrier parity, flipped by the caller after every use.
__device__ __forceinline__ void load_window(WindowIndex& W, unsigned long long* mbar, const uint8_t* text, unsigned long long lo, int bytes,
                                            uint32_t& phase, bool synced = false) {
    if (!synced) __syncthreads();  // everyone is done with the previous contents
    if (threadIdx.x == 0) {
        fence_proxy_async();
        mbar_expect_tx(mbar, (uint32_t)bytes);
        for (int o = 0; o < bytes; o += 16384) {
            int n = bytes - o < 16384 ? bytes - o : 16384;
            tma_bulk_g2s(W.win + o, text + lo + o, (uint32_t)n, mbar);
        }
    }
    while (!mbar_try_wait(mbar, phase)) {
    }
    phase ^= 1;
}

// Window geometry for text [begin, end) seen through a window starting at `lo` of at most `max_bytes`.
__device__ __forceinline__ WinGeom make_geom(unsigned long long lo, int max_bytes, unsigned long long begin, unsigned long long end) {
    WinGeom g;
    g.lo = lo;
    unsigned long long up = (end + 15ull) & ~15ull;
    unsigned long long hi = lo + (unsigned long long)max_bytes;
    if (hi > up) hi = up;
    g.loaded = hi > lo ? (int)(hi - lo) : 0;
    g.rb = begin >= lo ? (int)((begin - lo) > 0x7fffffffull ? 0x7fffffff : (begin - lo)) : -1;
    g.vb = g.rb < 0 ? 0 : g.rb;
    long long re = (long long)end - (long long)lo;
    g.re = re > (long long)kWin + 64 ? kWin + 64 : (int)re;
    g.covers_eof = end <= lo + (unsigned long long)g.loaded;
    g.L = g.re < g.loaded ? g.re : g.loaded;
    g.qlo = g.vb;
    g.qhi = g.L;
    return g;
}

// SIMD-in-register byte classification: 0x80 in every byte of the result where the predicate holds
__device__ __forceinline__ uint32_t bytes_eq(uint32_t x, uint32_t c4) {
    uint32_t t = x ^ c4;  // zero byte <=> equal
    return ~(((t & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | t) & 0x80808080u;
}
__device__ __forceinline__ uint32_t bytes_digit(uint32_t x) {
    uint32_t t = x ^ 0x30303030u;  // '0'..'9' -> 0..9
    return ~(((t & 0x7F7F7F7Fu) + 0x76767676u) | t) & 0x80808080u;
}
// bytes below 0x23 ('#'): control characters, space, '!' and '"'.  In clean BLAST text only tab and newline are.
__device__ __forceinline__ uint32_t bytes_below_23(uint32_t x) {
    uint32_t t = (x | 0x80808080u) - 0x23232323u;  // no borrow between bytes; bit 7 survives iff (x & 0x7f) >= 0x23
    return ~t & ~x & 0x80808080u;
}
// Gathers the sixteen 0x80 flags of four words into a 16-bit mask with four dot products:
// a flag byte is 0x80 = 128, so dp4a(flags, weights) = 128 * (sum of the weights of the set bytes).
__device__ __forceinline__ uint32_t pack16(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    const uint32_t lo = __dp4a(a, 0x08040201u, __dp4a(b, 0x80402010u, 0u));
    const uint32_t hi = __dp4a(c, 0x08040201u, __dp4a(d, 0x80402010u, 0u));
    return (lo >> 7) | (hi << 1);
}

__device__ __forceinline__ uint32_t range_mask16(int pos0, int lo, int hi) {  // bits k with lo <= pos0+k < hi
    int a = lo - pos0, b = hi - pos0;
    a = a < 0 ? 0 : (a > 16 ? 16 : a);
    b = b < 0 ? 0 : (b > 16 ? 16 : b);
    if (b <= a) return 0;
    return ((1u << b) - 1u) & ~((1u << a) - 1u);
}

// Rare path of the row scan: some byte below 0x23 is neither tab nor newline -- look for '"' / '\r' exactly.
__device__ __noinline__ void quote_check(WindowIndex& W, const WinGeom& g, const uint4 v, int pos0) {
    const uint32_t qm = pack16(bytes_eq(v.x, 0x22222222u) | bytes_eq(v.x, 0x0D0D0D0Du), bytes_eq(v.y, 0x22222222u) | bytes_eq(v.y, 0x0D0D0D0Du),
                               bytes_eq(v.z, 0x22222222u) | bytes_eq(v.z, 0x0D0D0D0Du), bytes_eq(v.w, 0x22222222u) | bytes_eq(v.w, 0x0D0D0D0Du)) &
                        range_mask16(pos0, g.qlo, g.qhi);
    if (qm) atomicMin(&W.bad_byte, pos0 + __ffs(qm) - 1);
}

// Row scan, pass 1: classifies one 16-byte chunk (newline / tab / digit / quote-or-CR) with SIMD-in-register byte
// tests, publishes the tab and digit masks, and derives the row-start / row-end masks of the chunk
// (DESIGN.md "row index").  `carry` = the byte in front of the chunk is a newline.
__device__ __forceinline__ void classify_chunk(WindowIndex& W, const WinGeom& g, int c, uint32_t carry, uint32_t& nl_out, uint32_t& start,
                                               uint32_t& end) {
    const int pos0 = c << 4;
    const uint4 v = *reinterpret_cast<const uint4*>(W.win + pos0);
    const int rb = g.vb;
    const int tend = g.re < g.loaded ? g.re : g.loaded;  // end of the text inside the window
    const uint32_t nx = bytes_eq(v.x, 0x0A0A0A0Au), ny = bytes_eq(v.y, 0x0A0A0A0Au), nz = bytes_eq(v.z, 0x0A0A0A0Au), nw = bytes_eq(v.w, 0x0A0A0A0Au);
    const uint32_t tx = bytes_eq(v.x, 0x09090909u), ty = bytes_eq(v.y, 0x09090909u), tz = bytes_eq(v.z, 0x09090909u), tw = bytes_eq(v.w, 0x09090909u);
    uint32_t nl = pack16(nx, ny, nz, nw);
    W.tabm[c] = (uint16_t)pack16(tx, ty, tz, tw);
    W.digm[c] = (uint16_t)pack16(bytes_digit(v.x), bytes_digit(v.y), bytes_digit(v.z), bytes_digit(v.w));
    // any byte below 0x23 that is neither tab nor newline is suspicious; only then look for '"' / '\r' exactly
    const uint32_t sus = (bytes_below_23(v.x) & ~(nx | tx)) | (bytes_below_23(v.y) & ~(ny | ty)) | (bytes_below_23(v.z) & ~(nz | tz)) |
                         (bytes_below_23(v.w) & ~(nw | tw));
    if (__builtin_expect(sus != 0, 0)) quote_check(W, g, v, pos0);
    if (__builtin_expect(pos0 <= rb || pos0 + 16 > tend, 0)) {
        // chunk on an edge of the text (the first / last chunk of the whole text only)
        nl &= range_mask16(pos0, rb, g.L);
        const uint32_t tmask = range_mask16(pos0, rb, tend);
        if (g.rb >= 0 && pos0 == g.rb) carry = 1;  // virtual newline in front of the text
        if (pos0 < rb) carry = 0;
        uint32_t prev = ((nl << 1) | carry) & 0xFFFFu;
        if (g.rb > pos0 && g.rb < pos0 + 16) prev |= 1u << (g.rb - pos0);
        start = prev & ~nl & tmask;
        end = nl & ~prev;
    } else {
        const uint32_t prev = ((nl << 1) | carry) & 0xFFFFu;
        start = prev & ~nl;
        end = nl & ~prev;
    }
    nl_out = nl;
}

// Builds row_s / row_e for the staged window.  Returns false (uniformly) when the row table would overflow,
// which can only happen when some row is shorter than 26 bytes, i.e. malformed.
template <int NWARPS>
__device__ bool scan_rows(WindowIndex& W, const WinGeom& g) {
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int cbeg = g.vb >> 4;  // chunks in front of the first valid byte are not scanned
    const int nchunks = (g.L + 15) >> 4;
    const int cpw = ((((nchunks - cbeg) + NWARPS - 1) / NWARPS) + 31) & ~31;  // chunks per warp, whole 32-lane rounds
    const int c0 = cbeg + w * cpw;
    const int c1 = c0 + cpw < nchunks ? c0 + cpw : nchunks;
    const int rb = g.vb;
    // ---- pass 1: classify; every warp compacts the row starts / ends of its chunk range ------------------------------
    // A valid row is >= 26 bytes, so a 16-byte chunk holds at most one row start and one row end; a chunk with more
    // proves a malformed (too short) row and is reported as such.  So a warp's k-th row start can be parked at index
    // c0 + k of the (chunk-indexed) scratch array: it never overtakes the chunk it came from.
    const uint32_t lt = (1u << lane) - 1u;
    int ns = 0, ne = 0;
    bool crowded = false;
    uint32_t carry_in = 0;
    if (c0 < c1 && (c0 << 4) > rb) carry_in = W.win[(c0 << 4) - 1] == '\n';
    for (int base = c0; base < c1; base += 32) {
        const int c = base + lane;
        uint32_t nl = 0, s = 0, e = 0;
        const bool live = c < c1;
        if (live) classify_chunk(W, g, c, 0u, nl, s, e);  // provisional carry 0, bit 0 is patched below
        const uint32_t up = __shfl_up_sync(0xffffffffu, nl, 1);
        const uint32_t carry = lane == 0 ? carry_in : (up >> 15) & 1u;
        carry_in = (__shfl_sync(0xffffffffu, nl, 31) >> 15) & 1u;
        const int pos0 = c << 4;
        if (live && carry && pos0 >= rb && !(g.rb >= 0 && pos0 == g.rb)) {
            // byte 0 of the chunk follows a newline: it starts a row unless it is a newline itself, and a newline
            // there does not end a row (empty line)
            const int tend = g.re < g.loaded ? g.re : g.loaded;
            if (!(nl & 1u) && pos0 < tend) s |= 1u;
            e &= ~1u;
        }
        crowded |= (s & (s - 1)) != 0 || (e & (e - 1)) != 0;
        const uint32_t bs = __ballot_sync(0xffffffffu, s != 0), be = __ballot_sync(0xffffffffu, e != 0);
        // (all chunks of this round are classified before anything is parked: the parking slots c0+ns.. lie at or
        // below the chunks of this round, whose own masks are not needed any more)
        if (s) W.startm[c0 + ns + __popc(bs & lt)] = (uint16_t)(pos0 + __ffs(s) - 1);
        if (e) W.endm[c0 + ne + __popc(be & lt)] = (uint16_t)(pos0 + __ffs(e) - 1);
        ns += __popc(bs);
        ne += __popc(be);
    }
    crowded = __any_sync(0xffffffffu, crowded);
    if (lane == 0) W.warp_cnt[w] = ns | (ne << 16) | (crowded ? 0x80000000 : 0);
    __syncthreads();
    int so = 0, eo = 0, ts = 0, te = 0;
    bool any_crowded = false;
#pragma unroll
    for (int i = 0; i < NWARPS; i++) {
        const int v = W.warp_cnt[i];
        any_crowded |= v < 0;
        if (i < w) {
            so += v & 0xFFFF;
            eo += (v >> 16) & 0x7FFF;
        }
        ts += v & 0xFFFF;
        te += (v >> 16) & 0x7FFF;
    }
    if (tid == 0) {
        W.n_starts = ts;
        W.n_ends = te;
    }
    if (any_crowded || ts > kRowCap || te > kRowCap) {
        __syncthreads();
        return false;
    }
    // ---- pass 2: move every warp's compacted positions to their place in the row table -------------------------------
    for (int i = lane; i < ns; i += 32) W.row_s[so + i] = W.startm[c0 + i];
    for (int i = lane; i < ne; i += 32) W.row_e[eo + i] = W.endm[c0 + i];
    __syncthreads();
    return true;
}

// Writes the virtual newline that terminates an unterminated last row (final chunk only) and fixes g.L.
__device__ __forceinline__ void finish_geom(WindowIndex& W, WinGeom& g, bool final_chunk) {
    if (final_chunk && g.covers_eof && g.re > 0 && g.re <= g.loaded) {
        bool needs = (g.re - 1 >= 0) && W.win[g.re - 1] != '\n' && g.re - 1 >= g.vb;
        if (needs) {
            __syncthreads();
            if (threadIdx.x == 0) W.win[g.re] = '\n';  // win has 128 spare bytes
            g.L = g.re + 1;
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// tile kernel (streaming)
//
// The text [begin, end) is cut into gridDim.x contiguous segments; CTA c owns every query run whose first row starts
// inside segment c.  It walks its segment in windows of kTile bytes, staged into shared memory by TMA bulk copies
// into two alternating buffers (the copy of window k+1 runs under the row / run phases of window k).  A window
// starts 16-byte aligned just in front of the last complete row of the previous window (that row is the
// "look-behind" row: it is only there so that the first new row can be compared with its predecessor), so no row
// and no query ever has to fit a window: the unfinished query is carried in shared memory (row count, best bit
// score, its top rows so far) from window to window, and a CTA keeps walking past the end of its segment until the
// query it has open ends.  Phases of one window (three CTA-wide barriers):
//   B  classify   every lane owns 32 bytes: SIMD-in-register byte tests (ASCII fast path) -> newline / tab / digit
//                 bitmasks (dp4a packing); row starts compacted per 1 KB round with two ballots; the last warp out
//                 computes the prefix over the rounds' row counts
//   D  rows       one thread per row (global row index -> round by a shuffle search): validation + truncated bit score
//                 (parse_row_lean, falling back to the full grammar), packed field positions, head flag (query id
//                 differs from the previous row's); meanwhile the last warp of the CTA finds the last newline and
//                 requests the next window's bytes
//   E  runs       one warp per query run (static assignment): extent, best bit score, top rows (ballot compaction);
//                 the warp decides the run's fate (finished / still open / block path), merges it with the carried
//                 query, takes top-row slots from the CTA's slab and a place in the record buffer (shared-memory
//                 atomics), folds its top rows' digits (top_row_from_info) and writes them to HBM / the carry
//      then       thread 0: a new slot slab when the current one runs low, record flush (one global atomic per >= 128
//                 headers), where the CTA goes next
// ---------------------------------------------------------------------------------------------------------------
constexpr int kSWarps = kTileThreads / 32;
constexpr int kUnits = kTile / 32 + 1;       // 32-byte units of a window (+1: the unit that can hold a virtual final newline)
#ifndef BLU_ROUND_UNITS
#define BLU_ROUND_UNITS 32
#endif
constexpr int kRoundUnits = BLU_ROUND_UNITS;  // phase B works in rounds of this many 32-byte units per warp (32: 1 KB, 64: 2 KB -- half as
                                              // many rounds, so half the per-round bookkeeping); the extra unit of a virtual final
                                              // newline goes to the last round
constexpr int kRounds = kTile / (32 * kRoundUnits);
constexpr int kSegCap = kRoundUnits * 2 + 4;  // row starts one round can find (<= 1 per 16 bytes, else malformed)
constexpr int kSRowCap = kTile / 26 + 8;     // a valid row is >= 26 bytes
constexpr int kRecFlush = 128;                // buffered record headers that trigger a flush (one global atomic)
constexpr int kRecBuf = 176;                  // capacity of the record buffer (beyond: the run reserves its record itself)
#ifndef BLU_TOPQ
#define BLU_TOPQ 160
#endif
constexpr int kTopQCap = BLU_TOPQ;            // top rows of a window whose field parse is deferred to the next window (0: parse in the run phase)
constexpr uint16_t kTopQEmpty = 0xFFFFu;      // TopQ::where of a slot a failed reservation left unfilled
constexpr uint32_t kSlotSlab = 1024;          // top-row slots a CTA reserves at a time (one global atomic)
constexpr uint32_t kSlotLow = 64;             // a new slab is fetched at the end of a window that leaves fewer free slots
constexpr int kCarryTop = 32;                 // top rows of the open query kept in shared memory (beyond: block path)

static_assert(kSRowCap < 0x8000, "row indices are 15-bit");
static_assert(kTile % 32 == 0 && kTile + 128 < 65536, "window offsets are 16-bit");
static_assert(kRoundUnits % 32 == 0 && kTile % (32 * kRoundUnits) == 0 && kRounds <= 32 && kRounds >= 1, "per-round tables are read by one warp");

enum : uint32_t { RK_EMIT = 1, RK_DEFER = 2, RK_PSEUDO = 4, RK_OPEN = 8, RK_NEWCARRY = 16 };

struct CarryRun {
    unsigned long long head_abs;  // offset of the open query's first row
    uint32_t qlen;
    uint32_t nrows;
    int32_t mx;        // best truncated bit score so far
    int32_t g;         // top rows so far (kept in tops[])
    int32_t open;
    int32_t deferred;  // the query goes to the block path when it ends (top group too large / bit score beyond int32)
    TopRowRaw tops[kCarryTop];  // its top rows so far
};

struct StagedRec {
    unsigned long long abs;
    uint32_t qlen, nrows;
    int32_t mx;
    uint32_t slot;  // first top-row slot
    uint32_t gtot;
    uint32_t pad;
};

// A top row found by the run phase, to be split and parsed later: one warp does it for ALL runs of a window with full lanes
// (next window, by the warp that has no rows) instead of every run's warp doing it for its own two or three rows.
struct TopQ {
    uint32_t dst;    // HBM: top-row slot; carry: index into its tops[]
    uint32_t info;   // packed field positions of the row (parse_row_lean), 0: unknown
    uint16_t s, e;   // the row in its window
    uint16_t where;  // 0: p.toprows, 1 / 2: carry[0] / carry[1]
    uint16_t pad;
};

struct WinDesc {  // what a window covers; written one window ahead, together with the request for its bytes
    unsigned long long lo;  // text offset of win[0] (16-byte aligned)
    int loaded, tend, vb;   // bytes staged; end / begin of the text inside the window
    int flags;              // 1: the window reaches the end of the text, 2: it contains the first byte of the text
};

struct WinGeo {  // row geometry of a window; written by the last warp that leaves phase B
    unsigned long long next_lo;
    int n_starts, n_complete, last_nl, may_continue, crowded;
    int inc[32], nfirst[32], plast[32];  // per warp share: rows up to and including it; first row start behind / last before it
};

struct StreamSmem {
    alignas(128) uint8_t win[2][kTile + 128];
    // byte-class bitmasks, bit i of word u = byte 32u+i of the window (read by the row parsers as 32/64-bit words)
    alignas(8) uint32_t tabm[kUnits + 7];
    alignas(8) uint32_t digm[kUnits + 7];
    alignas(8) uint32_t nlm[kUnits + 7];
    uint16_t seg[kRounds][kSegCap];  // row starts found in round i, in order
    uint16_t row_s[kSRowCap + 2];    // all row starts of the window (written by phase D)
    int32_t bits[kSRowCap];
    uint8_t flags[kSRowCap];         // bit1: bit score does not fit int32
    uint32_t rowinfo[kSRowCap];      // packed tab positions of the row (parse_row_lean), 0: unknown
    uint32_t headw[(kSRowCap + kTileThreads) / 32 + 2];  // head flags, one bit per row (the row loop writes whole rounds)
    uint32_t runs[kSRowCap + 1];     // head rows in arrival order: row | id length << 16 (bit 15: continuation of the carried query)
    StagedRec rec_buf[kRecBuf];  // record headers of finished queries, waiting for the next flush
    TopQ tq[kTopQCap > 0 ? kTopQCap : 1];
    unsigned long long tq_lo;    // text offset of the window the queued rows belong to
    int tq_cnt;
    uint16_t stage[kSWarps][32];
    CarryRun carry[2];
    alignas(8) unsigned long long mbar[2];
    int warp_cnt[32], warp_first[32], warp_last[32];  // per round of phase B: row starts, the first and the last one
    WinDesc wd[2];
    WinGeo geo;
    int b_done;  // warps that have finished phase B of the current window
    int bad_byte, has_blank, crowded;
    int n_runs, next_run, n_skip, term, new_open;
    unsigned long long rec_base;
    uint32_t slot_cur, slot_end;  // the CTA's current slab of top-row slots: [slot_cur, slot_end) is free
    int rec_cnt;                  // record headers in rec_buf
    uint32_t slots_taken;         // slots this CTA has reserved in slabs so far (sizes the next slab)
    int out_ok;                   // 0: an output capacity was exceeded (the host grows the arrays and reruns)
};

static_assert((sizeof(StreamSmem) + 1024) * kTileCtasPerSm <= 227 * 1024, "tile CTAs must fit one SM");

__device__ __forceinline__ void push_defer(const RunParams& p, unsigned long long off, unsigned check_prev) {
    unsigned i = atomicAdd(&p.ctr->n_defer, 1u);
    if (i < p.defer_cap)
        p.defer[i] = (off << 1) | check_prev;
    else
        p.ctr->cap_overflow = 1;
}

__device__ __forceinline__ void stream_issue_load(StreamSmem& S, int buf, const uint8_t* text, unsigned long long lo, int bytes) {
    fence_proxy_async();
    mbar_expect_tx(&S.mbar[buf], (uint32_t)bytes);
    for (int o = 0; o < bytes; o += 16384) {
        const int n = bytes - o < 16384 ? bytes - o : 16384;
        tma_bulk_g2s(S.win[buf] + o, text + lo + o, (uint32_t)n, &S.mbar[buf]);
    }
}

// dp4a gathers the 0x80 flags of two words into 128 * (8-bit mask)
__device__ __forceinline__ uint32_t pack8(uint32_t a, uint32_t b) { return __dp4a(a, 0x08040201u, __dp4a(b, 0x80402010u, 0u)); }
__device__ __forceinline__ uint32_t pack32(const uint32_t (&f)[8]) {
    const uint32_t b0 = pack8(f[0], f[1]) + (pack8(f[2], f[3]) << 8);  // 128 * 16-bit mask
    const uint32_t b1 = pack8(f[4], f[5]) + (pack8(f[6], f[7]) << 8);
    return __funnelshift_r(b0 + (b1 << 16), b1 >> 16, 7);
}

// Exact byte-wise classification of one 32-byte unit: text edges (bytes outside [vb, tend) are not text), units with
// non-ASCII bytes, and the exact '"' / '\r' search behind the cheap "suspicious byte" test.  Publishes the unit's tab /
// digit / newline masks when `publish` is set and returns the newline mask.
__device__ __noinline__ uint32_t classify_unit_slow(StreamSmem& S, const uint8_t* w, int pos0, int vb, int tend, int virt_nl_at, bool publish) {
    uint32_t nl = 0, tab = 0, dig = 0;
    int bad = INT_MAX;
    for (int k = 0; k < 32; k++) {
        const int pos = pos0 + k;
        if (pos < vb || pos >= tend) continue;
        const uint32_t c = w[pos];
        if (c == '\n') nl |= 1u << k;
        if (c == '\t') tab |= 1u << k;
        if (c - '0' <= 9u) dig |= 1u << k;
        if ((c == '"' || c == '\r') && pos < bad) bad = pos;
    }
    if (bad != INT_MAX) atomicMin(&S.bad_byte, bad);
    if (virt_nl_at >= pos0 && virt_nl_at < pos0 + 32) nl |= 1u << (virt_nl_at - pos0);
    if (publish) {
        const int u = pos0 >> 5;
        S.tabm[u] = tab;
        S.digm[u] = dig;
        S.nlm[u] = nl;
    }
    return nl;
}

// first head row at index >= from, or -1 (whole warp)
__device__ __forceinline__ int next_head(const StreamSmem& S, int from, int n_rows, int lane) {
    const int nwords = (n_rows + 31) >> 5;
    for (int k0 = from >> 5; k0 < nwords; k0 += 32) {
        const int k = k0 + lane;
        uint32_t w = k < nwords ? S.headw[k] : 0u;
        if (k == (from >> 5)) w &= ~0u << (from & 31);
        const unsigned bal = __ballot_sync(0xffffffffu, w != 0);
        if (bal) {
            const int src = __ffs(bal) - 1;
            const uint32_t wv = __shfl_sync(0xffffffffu, w, src);
            return ((k0 + src) << 5) + __ffs(wv) - 1;
        }
    }
    return -1;
}

// end (position of the newline) of the row that starts at window offset s, through the newline mask
__device__ __noinline__ int row_end_search(const StreamSmem& S, int s, int limit) {
    for (int u = s >> 5; (u << 5) <= limit; u++) {
        uint32_t w = S.nlm[u];
        if (u == (s >> 5)) w &= ~0u << (s & 31);
        if (w) return (u << 5) + __ffs(w) - 1;
    }
    return limit;
}

// Phase B for one round: units [u0, u1) of the window (32 of them; the last round may have one more).  kInterior: every
// unit is whole text (no edge of the input in the window), so the per-unit edge tests are compiled out.
template <bool kInterior>
__device__ __forceinline__ void classify_round(StreamSmem& S, const uint8_t* win, int round, int u0, int u1, int vb, int tend, bool has_begin,
                                               bool virt_nl, int lane) {
    const unsigned FULL = 0xffffffffu;
    const uint32_t lt = (1u << lane) - 1u;
    int cnt = 0;
    uint32_t crowd = 0, blank = 0;
    uint32_t carry_in = 0;
    if (u0 < u1 && u0 > 0 && (u0 << 5) - 1 >= vb) carry_in = win[(u0 << 5) - 1] == '\n';
    uint16_t* const seg = S.seg[round];
    for (int base = u0; base < u1; base += 32) {
        const int u = base + lane;
        const int pos0 = u << 5;
        uint32_t nl = 0;
        const bool live = kInterior || u < u1;
        const bool edge = !kInterior && ((has_begin && pos0 <= vb) || pos0 + 32 > tend);  // first / last bytes of the text
        if (live) {
            const uint4 v0 = *reinterpret_cast<const uint4*>(win + pos0);
            const uint4 v1 = *reinterpret_cast<const uint4*>(win + pos0 + 16);
            const uint32_t x[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
            const uint32_t hi = (x[0] | x[1] | x[2] | x[3] | x[4] | x[5] | x[6] | x[7]) & 0x80808080u;
            if (__builtin_expect(edge || hi != 0, 0)) {
                nl = classify_unit_slow(S, win, pos0, vb, tend, virt_nl ? tend : -1, true);
            } else {
                // ASCII bytes: per-byte sums stay below 0x100, so plain 32-bit adds classify four bytes at once
                uint32_t fn[8], ft[8], fd[8], sus = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    uint32_t tu = (x[k] ^ 0x09090909u) + 0x7F7F7F7Fu;  // bit 7 clear <=> tab
                    uint32_t nu = (x[k] ^ 0x0A0A0A0Au) + 0x7F7F7F7Fu;  // bit 7 clear <=> newline
                    // (opaque to the optimiser: it would otherwise re-derive ~tu / ~nu with a second add per word)
                    asm("" : "+r"(tu));
                    asm("" : "+r"(nu));
                    const uint32_t ge30 = x[k] + 0x50505050u, ge3a = x[k] + 0x46464646u, ge23 = x[k] + 0x5D5D5D5Du;
                    ft[k] = ~tu & 0x80808080u;
                    fn[k] = ~nu & 0x80808080u;
                    fd[k] = ge30 & ~ge3a & 0x80808080u;
                    sus |= ~ge23 & tu & nu;  // below '#' and neither tab nor newline: look closer
                }
                nl = pack32(fn);
                S.tabm[u] = pack32(ft);
                S.digm[u] = pack32(fd);
                S.nlm[u] = nl;
                if (__builtin_expect((sus & 0x80808080u) != 0, 0)) classify_unit_slow(S, win, pos0, vb, tend, -1, false);  // exact '"' / '\r' search
            }
        }
        // row starts: a non-newline byte behind a newline (or behind the virtual newline in front of the text)
        const uint32_t upv = __shfl_up_sync(FULL, nl, 1);
        const uint32_t carry = lane == 0 ? carry_in : (upv >> 31);
        carry_in = __shfl_sync(FULL, nl, 31) >> 31;
        uint32_t prev = (nl << 1) | carry;
        uint32_t st;
        if (__builtin_expect(edge, 0)) {
            const uint32_t valid_lo = pos0 >= vb ? ~0u : (vb - pos0 >= 32 ? 0u : ~0u << (vb - pos0));
            const uint32_t valid_hi = pos0 + 32 <= tend ? ~0u : (tend <= pos0 ? 0u : ~0u >> (32 - (tend - pos0)));
            if (pos0 <= vb) prev &= valid_lo;  // the byte in front of vb is not text
            if (has_begin && vb >= pos0 && vb < pos0 + 32) prev |= 1u << (vb - pos0);
            st = prev & ~nl & valid_lo & valid_hi;
        } else
            st = prev & ~nl;
        blank |= nl & prev;
        // a valid row is >= 26 bytes: at most one start per 16 bytes, compacted with one ballot per half
        const uint32_t sl = st & 0xFFFFu, sh = st >> 16;
        crowd |= (sl & (sl - 1u)) | (sh & (sh - 1u));
        const unsigned bl = __ballot_sync(FULL, sl != 0), bh = __ballot_sync(FULL, sh != 0);
        int idx = cnt + __popc(bl & lt) + __popc(bh & lt);
        if (sl) seg[idx++] = (uint16_t)(pos0 + __ffs(sl) - 1);
        if (sh) seg[idx] = (uint16_t)(pos0 + 16 + __ffs(sh) - 1);
        cnt += __popc(bl) + __popc(bh);
    }
    if (__any_sync(FULL, (blank | crowd) != 0)) {  // (one vote on the common path)
        if (__any_sync(FULL, blank != 0) && lane == 0) S.has_blank = 1;
        if (__any_sync(FULL, crowd != 0) && lane == 0) S.crowded = 1;
    }
    __syncwarp();
    if (lane == 0) {
        S.warp_cnt[round] = cnt;
        S.warp_first[round] = cnt ? (int)seg[0] : -1;
        S.warp_last[round] = cnt ? (int)seg[cnt - 1] : -1;
    }
}

// Splits and parses the queued top rows of the window whose bytes are in `win` (fields 1..4 through the tab positions the row
// phase found: digit folds only; a row of any other shape leaves unparsed -- offset + length -- and is split by the consensus
// kernel's full parser) and writes them where the run phase said.  Entries [first, n) in steps of `stride`.
__device__ __forceinline__ void drain_topq(const RunParams& p, StreamSmem& S, const uint8_t* win, int first, int stride) {
    const int n = S.tq_cnt < kTopQCap ? S.tq_cnt : kTopQCap;
    const unsigned long long lo = S.tq_lo;
    const bool ok = S.out_ok != 0;
    for (int i = first; i < n; i += stride) {
        const TopQ d = S.tq[i];
        if (d.where == kTopQEmpty) continue;
        TopRowRaw ref;
        if (!top_row_from_info(win, (int)d.s, d.info, lo, ref)) {
            ref.acc_off = lo + (unsigned long long)d.s;
            ref.acc_len = (uint32_t)((int)d.e - (int)d.s);
            ref.taxid = 0, ref.alnlen = 0, ref.pident = 0.0;
            ref.dec_frac = kTopRowUnparsed;
        }
        if (d.where == 0) {
            if (ok) p.toprows[d.dst] = ref;
        } else
            S.carry[d.where - 1].tops[d.dst] = ref;
    }
}

__device__ __forceinline__ void write_record(blu_record* dst, const StagedRec& sr) {
    blu_record rec;
    rec.query_off = sr.abs;
    rec.query_len = sr.qlen;
    rec.n_rows = sr.nrows;
    rec.keep_mask = 0;
    rec.perc_identity = 0.0;
    rec.bit_score = (int64_t)sr.mx;
    rec.ref_lineage = 0;
    rec.bean_base = sr.slot;     // first top-row slot / size of the top group until the consensus kernel has run
    rec.n_beans = sr.gtot;
    rec.acc_base = 0;
    rec.status = 2;              // waiting for the consensus kernel
    rec.single_match = 0;
    rec.mutated = 0;
    rec.reached_pos = 0;
    rec.allowed_pos = -1;
    rec.bean_level = 0;
    rec.pad[0] = rec.pad[1] = 0;
    *dst = rec;
}

// Flushes the buffered record headers: ONE global atomic reserves their (dense) place in the record array, then every
// thread writes headers.  All threads of the CTA call; two barriers.
__device__ __forceinline__ void flush_records(const RunParams& p, StreamSmem& S, int tid) {
    const int n = S.rec_cnt < kRecBuf ? S.rec_cnt : kRecBuf;
    if (n == 0) return;
    if (tid == 0) {
        const unsigned long long rec_base = atomicAdd(&p.ctr->rec_count, (unsigned long long)n);
        S.rec_base = rec_base;
        if (rec_base + (unsigned long long)n > p.rec_cap) {
            S.out_ok = 0;
            p.ctr->cap_overflow = 1;
        }
    }
    __syncthreads();
    if (S.out_ok) {
        const unsigned long long rec_base = S.rec_base;
        for (int i = tid; i < n; i += kTileThreads) write_record(p.records + rec_base + i, S.rec_buf[i]);
    }
    __syncthreads();
    if (tid == 0) S.rec_cnt = 0;
}

// One thread: describes the window that starts at `lo` in S.wd[buf] and asks the TMA unit for its bytes.
__device__ __forceinline__ void describe_and_load(StreamSmem& S, int buf, const RunParams& p, unsigned long long p_begin, unsigned long long lo,
                                                  unsigned long long up) {
    const int loaded = (int)(up - lo < (unsigned long long)kTile ? up - lo : (unsigned long long)kTile);
    WinDesc d;
    d.lo = lo;
    d.loaded = loaded;
    d.tend = (int)(p.end - lo < (unsigned long long)loaded ? p.end - lo : (unsigned long long)loaded);
    const bool has_begin = lo <= p_begin;
    d.vb = has_begin ? (int)(p_begin - lo) : 0;
    d.flags = (p.end <= lo + (unsigned long long)loaded ? 1 : 0) | (has_begin ? 2 : 0);
    S.wd[buf] = d;
    stream_issue_load(S, buf, p.text, lo, loaded);
}

#ifdef BLU_PHASE_CLOCKS
#define PCLK(i)                                  \
    {                                            \
        long long _t;                            \
        (void)*(volatile int*)&S.n_runs; /* a shared-memory access: the warp really is past the barrier */ \
        asm volatile("mov.u64 %0, %%clock64;" : "=l"(_t)::"memory"); \
        pc[i] += _t - pt;                        \
        pt = _t;                                 \
    }
#define RCLK(i)                                  \
    {                                            \
        long long _t;                            \
        asm volatile("mov.u64 %0, %%clock64;" : "=l"(_t)::"memory"); \
        rc[i] += _t - rt;                        \
        rt = _t;                                 \
    }
#else
#define PCLK(i)
#define RCLK(i)
#endif

// One segment [seg_lo, seg_hi) of the text, walked by the whole CTA.  ph0 / ph1: parities of the two window barriers (they
// live across the segments a CTA processes).
__device__ __forceinline__ void tile_segment(const RunParams& p, StreamSmem& S, const unsigned long long p_begin, const unsigned long long seg_lo,
                                             const unsigned long long seg_hi, uint32_t& ph0, uint32_t& ph1) {
#ifdef BLU_PHASE_CLOCKS
    long long pc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    long long pt = clock64();
    int n_win = 0;
    long long rc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long rt = 0;
#endif
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned FULL = 0xffffffffu;
    const unsigned long long b16 = p_begin & ~15ull;
    const unsigned long long up = (p.end + 15ull) & ~15ull;

    if (tid == 0) {
        S.carry[0].open = S.carry[1].open = 0;
        S.bad_byte = INT_MAX;
        S.has_blank = S.crowded = 0;
        S.n_runs = S.next_run = S.n_skip = S.term = S.new_open = 0;
        S.b_done = 0;
        S.tq_cnt = 0;
        {
            // the CTA's first slab of top-row slots (about 40 per window of the segment, at most kSlotSlab)
            const unsigned long long est = ((seg_hi - seg_lo) / (unsigned long long)kTile + 1ull) * 40ull + (unsigned long long)kSlotLow;
            const uint32_t slab = est < (unsigned long long)kSlotSlab ? (uint32_t)est : kSlotSlab;
            const unsigned long long rs = atomicAdd(&p.ctr->slot_count, (unsigned long long)slab);
            S.slot_cur = (uint32_t)rs;
            S.slot_end = (uint32_t)rs + slab;
            S.slots_taken = slab;
            S.rec_cnt = 0;
            S.out_ok = 1;
            if (rs + (unsigned long long)slab > p.slot_cap) {  // (slot_cap < 2^32: slot numbers fit the 32-bit fields)
                S.out_ok = 0;
                p.ctr->cap_overflow = 1;
            }
        }
    }
    for (int i = tid; i < 7; i += kTileThreads) S.tabm[kUnits + i] = S.digm[kUnits + i] = S.nlm[kUnits + i] = 0u;
    __syncthreads();
    int cur = 0;  // which carry buffer holds the open query
    int win_idx = 1;  // number of the window (epoch of S.new_open)
    unsigned long long own_from = seg_lo;  // rows that start at or after this offset have not been processed yet
    int buf = 0;
    if (tid == 0) {
        unsigned long long lo0 = seg_lo > p_begin + kBack ? (seg_lo - kBack) & ~15ull : b16;
        if (lo0 < b16) lo0 = b16;
        describe_and_load(S, 0, p, p_begin, lo0, up);
    }
    __syncthreads();

    while (true) {
        const uint8_t* const win = S.win[buf];
        const unsigned long long lo = S.wd[buf].lo;
        const int tend = S.wd[buf].tend, vb = S.wd[buf].vb;
        const bool covers_eof = (S.wd[buf].flags & 1) != 0, has_begin = (S.wd[buf].flags & 2) != 0;
        if (tid == 32) {
            // the window after the next one: start moving it from HBM to L2
            const unsigned long long nb = lo + 2ull * kTile - 512ull;
            if (nb < up && (nb < seg_hi + kTile)) {
                const unsigned long long n = up - nb < (unsigned long long)kTile ? up - nb : (unsigned long long)kTile;
                tma_prefetch_l2(p.text + nb, (uint32_t)n);
            }
        }
        // wait for this window's bytes
        {
            uint32_t& ph = buf ? ph1 : ph0;
            while (!mbar_try_wait(&S.mbar[buf], ph)) {
            }
            ph ^= 1;
        }
        PCLK(0)
        // an unterminated last row of the input is closed by a virtual newline at `tend`
        const bool virt_nl = p.final_chunk && covers_eof && tend > vb && win[tend - 1] != '\n';
        const int scan_len = tend + (virt_nl ? 1 : 0);
        const int n_units = (scan_len + 31) >> 5;

        // ---- phase B: classify + row starts, 1 KB rounds ------------------------------------------------------------------
        {
            const bool interior = !has_begin && tend == kTile && !virt_nl;
            for (int rd = warp; rd < kRounds; rd += kSWarps) {
                const int u0 = rd * kRoundUnits;
                if (interior)
                    classify_round<true>(S, win, rd, u0, u0 + kRoundUnits, 0, tend, false, false, lane);
                else {
                    const int u1 = (rd == kRounds - 1 || u0 + kRoundUnits > n_units) ? n_units : u0 + kRoundUnits;
                    classify_round<false>(S, win, rd, u0, u1 > u0 ? u1 : u0, vb, tend, has_begin, virt_nl, lane);
                }
            }
        }
        PCLK(1)
        // ---- row tables of the window: the prefix over the rounds is computed ONCE, by the last warp that leaves
        //      phase B; everything else (last newline, next window) is worked out behind the barrier by the last warp of the
        //      CTA, which normally has no rows in phase D, while the others already parse rows
        {
            int ticket = 0;
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                ticket = (int)atoms_add(&S.b_done, 1u);
            }
            ticket = __shfl_sync(FULL, ticket, 0);
            if (ticket == kSWarps - 1) {
                __threadfence_block();
                // lane i < kRounds holds the tables of round i
                const int c_i = lane < kRounds ? S.warp_cnt[lane] : 0;
                int inc_i = c_i;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int t = __shfl_up_sync(FULL, inc_i, d);
                    if (lane >= d) inc_i += t;
                }
                const int n_starts = __shfl_sync(FULL, inc_i, 31);
                const unsigned ne = __ballot_sync(FULL, c_i > 0);
                const unsigned below = ne & ((1u << lane) - 1u), above = lane >= 31 ? 0u : (ne & (~0u << (lane + 1)));
                const int wl = lane < kRounds ? S.warp_last[lane] : -1, wf = lane < kRounds ? S.warp_first[lane] : -1;
                int plast_i = __shfl_sync(FULL, wl, below ? 31 - __clz(below) : 0);
                if (!below) plast_i = -1;
                int nfirst_i = __shfl_sync(FULL, wf, above ? __ffs(above) - 1 : 0);
                if (!above) nfirst_i = -1;
                if (lane < kRounds) {
                    S.geo.inc[lane] = inc_i;
                    S.geo.nfirst[lane] = nfirst_i;
                    S.geo.plast[lane] = plast_i;
                }
                if (lane < 4) S.tabm[n_units + lane] = S.digm[n_units + lane] = S.nlm[n_units + lane] = 0u;
                if (lane == 0) {
                    S.geo.n_starts = n_starts;
                    S.geo.crowded = (S.crowded != 0 || n_starts > kSRowCap) ? 1 : 0;
                    S.b_done = 0;
                }
            }
        }
        __syncthreads();
        PCLK(2)
        const int n_starts = S.geo.n_starts;
        const bool blank = S.has_blank != 0;
        if (S.geo.crowded) {
            // a row shorter than 16 bytes / more rows than 26-byte rows fit: malformed input
            if (tid == 0) report(p.ctr, DE_BAD_FIELD_COUNT, lo);
            break;  // (no copy in flight: the next window has not been requested)
        }
        if (tid == 0 && S.bad_byte != INT_MAX) report(p.ctr, DE_QUOTE_OR_CR, lo + (unsigned)S.bad_byte);
        const int c_i = lane < kRounds ? S.warp_cnt[lane] : 0;
        const int inc_i = lane < kRounds ? S.geo.inc[lane] : n_starts;
        const int nfirst_i = lane < kRounds ? S.geo.nfirst[lane] : -1, plast_i = lane < kRounds ? S.geo.plast[lane] : -1;
        if (warp == kSWarps - 1) {
            if (kTopQCap > 0 && S.tq_cnt > 0) {
                // the previous window's top rows: its bytes are still in the other buffer (the copy into it is requested below)
                drain_topq(p, S, S.win[buf ^ 1], lane, 32);
                __syncwarp();
                if (lane == 0) S.tq_cnt = 0;
                __syncwarp();
            }
            // ---- last newline, last complete row, the next window (its bytes are requested now) ---------------------------
            const unsigned ne = __ballot_sync(FULL, c_i > 0);
            int last_start = __shfl_sync(FULL, lane < kRounds ? S.warp_last[lane] : -1, ne ? 31 - __clz(ne) : 0);
            if (!ne) last_start = -1;
            int last_nl = -1;
            for (int ub = n_units - 1; ub >= 0 && last_nl < 0; ub -= 32) {
                const int u = ub - lane;
                const uint32_t w = u >= 0 ? S.nlm[u] : 0u;
                const unsigned bal = __ballot_sync(FULL, w != 0);
                if (bal) {
                    const int src = __ffs(bal) - 1;
                    const uint32_t wv = __shfl_sync(FULL, w, src);
                    last_nl = ((ub - src) << 5) + 31 - __clz(wv);
                }
            }
            const int n_complete = (n_starts > 0 && last_start > last_nl) ? n_starts - 1 : n_starts;
            // the last complete row: the look-behind row of the next window
            int lc = last_start;
            if (n_complete != n_starts) {
                const int wlast = 31 - __clz(ne);  // (ne != 0: n_starts > 0)
                const int cl = __shfl_sync(FULL, c_i, wlast);
                const unsigned rest = ne & ~(1u << wlast);
                const int w2 = rest ? 31 - __clz(rest) : 0;
                const int c2 = __shfl_sync(FULL, c_i, w2);
                lc = cl >= 2 ? (int)S.seg[wlast][cl - 2] : (rest ? (int)S.seg[w2][c2 - 1] : -1);
            }
            if (lane == 0) {
                const bool progress = lc >= 0 && lo + (unsigned long long)lc >= own_from;  // a complete row this CTA had not seen yet
                unsigned long long next_lo = lo;
                if (progress) {
                    const unsigned long long la = lo + (unsigned long long)lc;
                    next_lo = la > p_begin ? (la - 1) & ~15ull : b16;
                    if (next_lo < b16) next_lo = b16;
                }
                const bool may_continue = progress && !covers_eof && next_lo > lo;
                S.geo.n_complete = n_complete;
                S.geo.last_nl = last_nl;
                S.geo.may_continue = may_continue ? 1 : 0;
                if (n_complete == n_starts) S.row_s[n_starts] = (uint16_t)(last_nl + 1);  // sentinel: end of the last row
                if (may_continue) describe_and_load(S, buf ^ 1, p, p_begin, next_lo, up);
            }
        }
        const uint64_t* tabw = reinterpret_cast<const uint64_t*>(S.tabm);
        const uint64_t* digw = reinterpret_cast<const uint64_t*>(S.digm);
        PCLK(3)
        // ---- phase D: one thread per row -------------------------------------------------------------------------------
        for (int rb = 0; rb < n_starts; rb += kTileThreads) {
            const int r = rb + tid;
            const bool live = r < n_starts;
            const int rr = live ? r : n_starts - 1;
            // which round found row rr: number of rounds that end at or before it
            int w = 0;
#pragma unroll
            for (int step = 16; step; step >>= 1) {
                const int cand = w + step;
                const int v = __shfl_sync(FULL, inc_i, (cand - 1) & 31);
                if (cand <= kRounds && v <= rr) w = cand;
            }
            const int cw = __shfl_sync(FULL, c_i, w);
            const int k = rr - (__shfl_sync(FULL, inc_i, w) - cw);
            const int nf = __shfl_sync(FULL, nfirst_i, w), pl = __shfl_sync(FULL, plast_i, w);
            bool head = false, skip = false;
            // part 1: validate + parse the row (the lanes of a warp part ways here: evalue shapes, the rare full-grammar path)
            bool parsed = false;
            int s = 0, ql = 0, prv = -1;
            unsigned long long abs = 0;
            if (live) {
                const uint16_t* const seg_w = S.seg[w];
                s = seg_w[k];
                S.row_s[r] = (uint16_t)s;
                abs = lo + (unsigned long long)s;
                if (abs < own_from)
                    skip = true;  // look-behind rows: seen by the previous window / owned by the previous segment
                else {
                    // the row's newline: in front of the next row start; the window's last start (and any row of a window
                    // with blank lines) looks it up in the newline mask -- none: an unterminated row, left to the next window
                    const int nxt = k + 1 < cw ? (int)seg_w[k + 1] : nf;
                    const int e = (nxt < 0 || blank) ? row_end_search(S, s, scan_len) : nxt - 1;
                    if (e < scan_len) {
                        int64_t bits;
                        uint32_t info;
                        if (!parse_row_lean(win, S.tabm, S.digm, s, e, bits, ql, info)) {
                            const LightRow lr = parse_row_masked(win, tabw, digw, s, e);
                            if (lr.err) report(p.ctr, lr.err, abs);
                            bits = lr.bits;
                            ql = lr.q_len;
                            info = 0;
                        }
                        S.rowinfo[r] = info;
                        const int32_t b32 = (int32_t)bits;
                        S.flags[r] = ((int64_t)b32 != bits) ? 2 : 0;
                        S.bits[r] = b32;
                        prv = k > 0 ? (int)seg_w[k - 1] : pl;
                        parsed = true;
                    }
                }
            }
            // part 2, with the warp back together (without this the two halves of a warp that took different branches above run
            // the compare one after the other): head flag = the query id differs from the previous row's
            __syncwarp();
            if (parsed) {
                if (prv < 0) {
                    head = has_begin;  // first row of the text; else: predecessor not in the window
                    if (!head) push_defer(p, abs, 1);  // the block path decides whether it starts a query
                } else
                    head = !same_qid_lean(win, S.tabm, s, ql, prv);
                if (head) {
                    if (abs < seg_hi) {
                        const int i = (int)atoms_add(&S.n_runs, 1u);
                        S.runs[i] = (uint32_t)r | ((uint32_t)(ql > 0xFFFF ? 0xFFFF : ql) << 16);
                    } else
                        S.term = 1;  // a query of the next segment starts here: this CTA ends with this window
                }
            }
            const unsigned hb = __ballot_sync(FULL, head);
            if (lane == 0) S.headw[r >> 5] = hb;
            const unsigned sb = __ballot_sync(FULL, skip);
            if (sb && lane == 0) atoms_add(&S.n_skip, (uint32_t)__popc(sb));
        }
        PCLK(4)
        __syncthreads();
        PCLK(5)
        // ---- phase E: one warp per query run (static assignment) -----------------------------------------------------------
        //   extent, best bit score, top rows (ballot compaction); the warp decides the run's fate (finished / still open /
        //   block path), merges it with the carried query, reserves its output and splits + parses its own top rows
        const int n_complete = S.geo.n_complete, last_nl = S.geo.last_nl;
        const bool may_continue = S.geo.may_continue != 0;
        const int n_runs = S.n_runs;
        const int r0 = S.n_skip;  // first row of this window the CTA had not seen
        const bool term = S.term != 0;
        const bool closes = covers_eof && p.final_chunk;  // the end of this window ends the open query
        PCLK(6)
#ifdef BLU_PHASE_CLOCKS
        rt = clock64();
#endif
        for (int j = warp; j < n_runs; j += kSWarps) {
            RCLK(0)
            const uint32_t entry = S.runs[j];
            const bool pseudo = (entry & 0x8000u) != 0;
            const int h = pseudo ? r0 : (int)(entry & 0x7FFFu);
            int e = next_head(S, pseudo ? h : h + 1, n_complete, lane);
            const bool open = e < 0;
            if (open) e = n_complete;
            if (e < h) e = h;
            RCLK(1)
            int mx = INT32_MIN;
            bool ovf = false;
            int g = 0;
            if (e - h <= 64) {
                // the usual case: the run's bit scores in two registers per lane, one pass over shared memory
                const int ra = h + lane, rb2 = ra + 32;
                int ba = INT32_MIN, bb = INT32_MIN;
                if (ra < e) {
                    ba = S.bits[ra];
                    ovf = (S.flags[ra] & 2) != 0;
                }
                if (rb2 < e) {
                    bb = S.bits[rb2];
                    ovf |= (S.flags[rb2] & 2) != 0;
                }
                mx = __reduce_max_sync(FULL, ba > bb ? ba : bb);
                ovf = __any_sync(FULL, ovf);
                const bool ta = ra < e && ba == mx, tb = rb2 < e && bb == mx;
                const unsigned bala = __ballot_sync(FULL, ta), balb = __ballot_sync(FULL, tb);
                const unsigned lt = (1u << lane) - 1u;
                const int na = __popc(bala);
                const int pa = __popc(bala & lt), pb = na + __popc(balb & lt);
                if (ta && pa < 32) S.stage[warp][pa] = (uint16_t)ra;
                if (tb && pb < 32) S.stage[warp][pb] = (uint16_t)rb2;
                g = na + __popc(balb);
            } else {
                for (int r = h + lane; r < e; r += 32) {
                    const int b = S.bits[r];
                    mx = b > mx ? b : mx;
                    ovf |= (S.flags[r] & 2) != 0;
                }
                mx = __reduce_max_sync(FULL, mx);
                ovf = __any_sync(FULL, ovf);
                for (int b = h; b < e; b += 32) {
                    const int r = b + lane;
                    const bool top = r < e && S.bits[r] == mx;
                    const unsigned bal = __ballot_sync(FULL, top);
                    const int pos = g + __popc(bal & ((1u << lane) - 1u));
                    if (top && pos < 32) S.stage[warp][pos] = (uint16_t)r;
                    g += __popc(bal);
                }
            }
            __syncwarp();
            if (g > 32) ovf = true;
            RCLK(2)
            // ---- lane 0: what happens to the run ------------------------------------------------------------------------
            uint32_t kind = 0, slot = 0;
            int g_part = 0, dst = 0, n_old = 0;
            if (lane == 0) {
                const int rows_t = e - h;
                g_part = ovf ? 0 : g;
                int g_tot = 0;
                kind = pseudo ? RK_PSEUDO : 0;
                unsigned long long abs;
                uint32_t qlen, nrows;
                if (pseudo) {
                    CarryRun& C = S.carry[cur];
                    if (ovf) C.deferred = 1;
                    if (rows_t > 0 && !C.deferred) {
                        if (mx > C.mx) {
                            C.mx = mx;
                            C.g = 0;
                        } else if (mx < C.mx)
                            g_part = 0;
                        if (C.g + g_part > kCarryTop) C.deferred = 1;
                    }
                    if (C.deferred || rows_t == 0) g_part = 0;
                    abs = C.head_abs, qlen = C.qlen, nrows = C.nrows + (uint32_t)rows_t;
                    mx = C.mx;
                    if (!open || closes) {
                        kind |= C.deferred ? RK_DEFER : RK_EMIT;
                        g_tot = C.g + g_part;
                        dst = C.g;
                        n_old = C.deferred ? 0 : C.g;
                        C.open = 0;
                    } else if (covers_eof) {
                        // the input continues in the next chunk: the whole query is carried over by the host
                        atomicMin(&p.ctr->tail_start, C.head_abs);
                        g_part = 0;
                        C.open = 0;
                    } else {
                        kind |= RK_OPEN;
                        C.nrows = nrows;
                        dst = -1 - C.g;
                        C.g += g_part;
                    }
                } else {
                    const int s = S.row_s[h];
                    qlen = entry >> 16;
                    if (qlen == 0xFFFFu) {
                        const int re = blank ? row_end_search(S, s, last_nl) : (int)S.row_s[h + 1] - 1;
                        qlen = (uint32_t)(next_tab(tabw, s, re) - s);
                    }
                    abs = lo + (unsigned long long)s;
                    nrows = (uint32_t)rows_t;
                    if (!open || closes) {
                        kind |= ovf ? RK_DEFER : RK_EMIT;
                        g_tot = g_part;
                    } else if (covers_eof) {
                        atomicMin(&p.ctr->tail_start, abs);
                        g_part = 0;
                    } else {
                        // a query that starts in this window and does not end in it: it becomes the carried query
                        CarryRun& C = S.carry[cur ^ 1];
                        kind |= RK_OPEN | RK_NEWCARRY;
                        C.open = 1;
                        C.deferred = ovf ? 1 : 0;
                        C.head_abs = abs;
                        C.qlen = qlen;
                        C.nrows = nrows;
                        C.mx = mx;
                        C.g = g_part;
                        dst = -1;
                        S.new_open = win_idx;
                    }
                }
                if (kind & RK_EMIT) {
                    // top-row slots from the CTA's slab (or, when it is exhausted, straight from the global counter)
                    if (g_tot > 0) {
                        slot = atoms_add(&S.slot_cur, (uint32_t)g_tot);
                        if (slot + (uint32_t)g_tot > S.slot_end || slot + (uint32_t)g_tot < slot) {
                            const unsigned long long rs = atomicAdd(&p.ctr->slot_count, (unsigned long long)g_tot);
                            slot = (uint32_t)rs;
                            if (rs + (unsigned long long)g_tot > p.slot_cap) {
                                S.out_ok = 0;
                                p.ctr->cap_overflow = 1;
                            }
                        }
                    }
                    StagedRec sr;
                    sr.abs = abs, sr.qlen = qlen, sr.nrows = nrows, sr.mx = mx, sr.gtot = (uint32_t)g_tot, sr.slot = slot, sr.pad = 0;
                    const int ri = (int)atoms_add(&S.rec_cnt, 1u);
                    if (ri < kRecBuf)
                        S.rec_buf[ri] = sr;
                    else {
                        // record buffer full (a window of very short queries): this record is reserved on its own
                        const unsigned long long ri2 = atomicAdd(&p.ctr->rec_count, 1ull);
                        if (ri2 < p.rec_cap)
                            write_record(p.records + ri2, sr);
                        else
                            p.ctr->cap_overflow = 1;
                    }
                }
                if (kind & RK_DEFER) push_defer(p, abs, 0);
            }
            RCLK(3)
            kind = __shfl_sync(FULL, kind, 0);
            slot = __shfl_sync(FULL, slot, 0);
            g_part = __shfl_sync(FULL, g_part, 0);
            dst = __shfl_sync(FULL, dst, 0);
            n_old = __shfl_sync(FULL, n_old, 0);
            const bool ok = S.out_ok != 0;
            // ---- the run's top rows of this window: queued for the warp that parses all of the window's top rows at once ------------
            if (g_part > 0 && (kind & (RK_EMIT | RK_OPEN))) {
                int qbase = -1;
                if (kTopQCap > 0) {
                    if (lane == 0) {
                        // no undo when the queue is full (an undo could land after another warp's successful reservation and take
                        // that warp's entries out of the count): the count stays above the capacity until the queue is drained,
                        // every later run of this window parses its rows itself, and the slots this reservation left unfilled
                        // are marked empty below
                        qbase = (int)atoms_add(&S.tq_cnt, (uint32_t)g_part);
                        if (qbase + g_part <= kTopQCap) S.tq_lo = lo;
                    }
                    qbase = __shfl_sync(FULL, qbase, 0);
                    if (qbase + g_part > kTopQCap) {
                        if (lane < g_part && qbase + lane < kTopQCap) S.tq[qbase + lane].where = kTopQEmpty;
                        qbase = -1;
                    }
                }
                if (lane < g_part) {
                    const int r = S.stage[warp][lane];
                    const int s = S.row_s[r];
                    const int re = blank ? row_end_search(S, s, last_nl) : (int)S.row_s[r + 1] - 1;
                    const int carry_buf = (kind & RK_NEWCARRY) ? (cur ^ 1) : cur;
                    if (qbase >= 0) {
                        TopQ d;
                        d.info = S.rowinfo[r];
                        d.s = (uint16_t)s, d.e = (uint16_t)re;
                        d.pad = 0;
                        if (kind & RK_EMIT)
                            d.where = 0, d.dst = slot + (uint32_t)(dst + lane);
                        else
                            d.where = (uint16_t)(1 + carry_buf), d.dst = (uint32_t)(-1 - dst + lane);
                        S.tq[qbase + lane] = d;
                    } else {
                        TopRowRaw ref;
                        if (!top_row_from_info(win, s, S.rowinfo[r], lo, ref)) {
                            ref.acc_off = lo + (unsigned long long)s;
                            ref.acc_len = (uint32_t)(re - s);
                            ref.taxid = 0, ref.alnlen = 0, ref.pident = 0.0;
                            ref.dec_frac = kTopRowUnparsed;
                        }
                        if (kind & RK_EMIT) {
                            if (ok) p.toprows[slot + (uint32_t)(dst + lane)] = ref;
                        } else
                            S.carry[carry_buf].tops[-1 - dst + lane] = ref;
                    }
                }
            }
            RCLK(4)
            // a carried query that ends here: its earlier top rows go in front of this window's
            if (lane < n_old && ok) p.toprows[slot + lane] = S.carry[cur].tops[lane];
            __syncwarp();
            RCLK(5)
        }
        PCLK(7)
        __syncthreads();
        PCLK(8)
        const bool new_open = S.new_open == win_idx;  // (an epoch, not a flag: nothing to reset)
        const bool need_flush = S.rec_cnt >= kRecFlush;
        if (tid == 0) {
            // a new slab of slots when this one runs low (one global atomic every few dozen windows)
            if (S.slot_end - S.slot_cur < kSlotLow || S.slot_cur > S.slot_end) {
                // sized by what the rest of the segment is likely to need (slots used per window so far x windows left), so that
                // the unused tail of a CTA's last slab -- a hole in slot space that is downloaded with the results -- stays small
                const unsigned long long left = seg_hi > lo ? (seg_hi - lo) / (unsigned long long)kTile + 1ull : 1ull;
                const unsigned long long est = (unsigned long long)(S.slots_taken / (uint32_t)win_idx + 8u) * left + (unsigned long long)kSlotLow;
                const uint32_t slab = est < (unsigned long long)kSlotSlab ? (uint32_t)est : kSlotSlab;
                S.slots_taken += slab;
                const unsigned long long rs = atomicAdd(&p.ctr->slot_count, (unsigned long long)slab);
                S.slot_cur = (uint32_t)rs;
                S.slot_end = (uint32_t)rs + slab;
                if (rs + (unsigned long long)slab > p.slot_cap) {
                    S.out_ok = 0;
                    p.ctr->cap_overflow = 1;
                }
            }
        }
        if (need_flush) flush_records(p, S, tid);
        PCLK(9)
        // ---- where next? -----------------------------------------------------------------------------------------------
        // The CTA is done when the window reached the end of the text, when a query that belongs to the next segment
        // started in it, or when nothing is open and the segment is exhausted.
        if (new_open) cur ^= 1;
        const bool open_now = S.carry[cur].open != 0;
        bool done = covers_eof || term;
        if (!done && !open_now && lo + (unsigned long long)(last_nl + 1) >= seg_hi) done = true;
        if (!done && !may_continue) {
            // no complete new row in a whole window: a row longer than this kernel stages
            if (tid == 0) report(p.ctr, DE_CARRY_TOO_BIG, own_from);
            done = true;
        }
        if (done) {
            if (may_continue) {
                // a copy into the other buffer is in flight: it must land before the CTA leaves the segment
                uint32_t& ph = (buf ^ 1) ? ph1 : ph0;
                while (!mbar_try_wait(&S.mbar[buf ^ 1], ph)) {
                }
                ph ^= 1;
            }
            break;
        }
#ifdef BLU_PHASE_CLOCKS
        n_win++;
#endif
        own_from = lo + (unsigned long long)(last_nl + 1);
        buf ^= 1;
        win_idx++;
        // reset the per-window state (published by the barrier behind phase B of the next window)
        if (tid == 0) {
            S.bad_byte = INT_MAX;
            S.has_blank = 0;
            S.n_skip = 0;
            S.term = 0;
            S.n_runs = open_now ? 1 : 0;
            S.runs[0] = 0x8000;  // the carried query continues (or ends) at the first new row
        }
    }
#ifdef BLU_PHASE_CLOCKS
    if ((blockIdx.x == 7 || blockIdx.x == 200) && (lane == 0))
        printf("cta %d warp %d windows %d | tma %lld B %lld bar1 %lld geom %lld D %lld bar2 %lld flush %lld E %lld bar3 %lld F %lld bar4 %lld\n", blockIdx.x, warp, n_win, pc[0] / (n_win + 1),
               pc[1] / (n_win + 1), pc[2] / (n_win + 1), pc[3] / (n_win + 1), pc[4] / (n_win + 1), pc[5] / (n_win + 1), pc[6] / (n_win + 1), pc[7] / (n_win + 1), pc[8] / (n_win + 1),
               pc[9] / (n_win + 1), pc[10] / (n_win + 1));
    if ((blockIdx.x == 7) && (lane == 0))
        printf("rcl %d warp %d windows %d | queue %lld head %lld stats %lld decide %lld parse %lld old %lld\n", blockIdx.x, warp, n_win, rc[0] / (n_win + 1), rc[1] / (n_win + 1),
               rc[2] / (n_win + 1), rc[3] / (n_win + 1), rc[4] / (n_win + 1), rc[5] / (n_win + 1));
#endif
    // ---- the last window's queued top rows (its bytes are still in `buf`), the record headers still in the buffer -----------
    __syncthreads();
    if (kTopQCap > 0) {
        drain_topq(p, S, S.win[buf], tid, kTileThreads);
        __syncthreads();
        if (tid == 0) S.tq_cnt = 0;
    }
    flush_records(p, S, tid);
    __syncthreads();
}

__global__ void __launch_bounds__(kTileThreads, kTileCtasPerSm) tile_kernel(const __grid_constant__ RunParams p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    StreamSmem& S = *reinterpret_cast<StreamSmem*>(smem_raw);
    // a later range of a resident table starts where the previous one stopped (its open last query): no host round trip
    const unsigned long long p_begin = p.begin == kBeginFromCounters ? p.ctr->next_begin : p.begin;
    if (p.end <= p_begin) return;
    // the text [begin, end) is cut into gridDim.x segments, one per CTA
    const unsigned long long total = p.end - p_begin;
    unsigned long long seg = (total + gridDim.x - 1) / gridDim.x;
    if (seg < 4ull * kTile) seg = 4ull * kTile;
    const unsigned long long seg_lo = p_begin + (unsigned long long)blockIdx.x * seg;
    if (seg_lo >= p.end) return;
    const unsigned long long seg_hi = (seg_lo + seg < p.end) ? seg_lo + seg : p.end;
    if (threadIdx.x == 0) {
        mbar_init(&S.mbar[0], 1);
        mbar_init(&S.mbar[1], 1);
    }
    __syncthreads();
    uint32_t ph0 = 0, ph1 = 0;
    tile_segment(p, S, p_begin, seg_lo, seg_hi, ph0, ph1);
}

// ---------------------------------------------------------------------------------------------------------------
// long-run kernel: one CTA per deferred run
// ---------------------------------------------------------------------------------------------------------------
constexpr int kQidCache = 256;  // bytes of the run's query id kept in shared memory

// Sort-phase arrays of the block-parallel consensus (the window and its row tables are dead by then): all indices are
// 16-bit (a top group holds at most kLongTopCap <= 65535 rows)
struct LongSort {
    uint16_t order[kLongTopCap];  // S: row numbers in the order of find_multi_taxa_consensus.rs:39-54
    uint16_t bord[kLongTopCap];   // positions of S sorted by (bean key, position): one segment per bean, S order inside
    uint16_t hb[kLongTopCap + 1]; // inclusive count of segment heads: bean number + 1
    uint16_t kp[kLongTopCap + 1]; // exclusive count of kept accessions (Vec::dedup)
    uint16_t st[kLongTopCap + 1]; // first position of every bean's segment
    uint16_t bsort[kLongTopCap];  // beans in output order (occurrences desc, identifier asc)
    uint16_t abeg[kLongTopCap];   // first accession of every bean, relative to the record's acc_base
    uint16_t tmp[kLongTopCap + 1];
    uint32_t key[kLongTopCap];    // bean key of every position of S
};

struct LongScanState {
    WindowIndex W;
    long long bits[kRowCap];
    uint8_t same[kRowCap];
};

struct LongSmem {
    union {
        LongScanState scan;
        LongSort sort;
    };
    alignas(8) unsigned long long mbar;  // (outside the union: its phase lives across runs)
    uint8_t qid[kQidCache];  // first field (+ its tab) of the run's first row
    long long red_max[kLongWarps];
    int red_cnt[kLongWarps];
    int red_first[kLongWarps];
    int scan_tot[kLongWarps];
    int bcast[8];
    unsigned long long bcast64[4];
};

static_assert(sizeof(LongSmem) <= 227 * 1024, "long-run CTA exceeds shared memory");

// first field of window row `a` == the run's query id (`qid` holds the id and its terminating tab, qn bytes)
__device__ __forceinline__ bool same_query_cached(const uint8_t* a, int alen, const uint8_t* qid, int qn) {
    if (alen < qn) return false;
    for (int i = 0; i < qn; i++)
        if (a[i] != qid[i]) return false;
    return true;
}

__device__ __forceinline__ bool same_query(const uint8_t* a, int alen, const uint8_t* text, unsigned long long s, unsigned long long end) {
    // compares the first field of row `a` (window) with the first field of the row at absolute offset s (global)
    for (int i = 0; i < alen; i++) {
        if (s + i >= end) return false;
        uint8_t b = text[s + i];
        if (a[i] != b) return false;
        if (b == '\t') return true;
    }
    return false;
}

struct LongScan {
    int ncomplete, eskip, d;     // d = first row that does not belong to the run (== ncomplete when none)
    unsigned long long next;     // where the next window starts
    bool at_end;                 // no more text after this window
    bool giant;                  // a row does not fit the window
};

// Stages the window that starts at `cur`, indexes and parses its rows, and marks which rows belong to the run
// whose first row starts at absolute offset `s`.
__device__ LongScan long_scan(LongSmem& S, const RunParams& p, unsigned long long s, unsigned long long cur, uint32_t& phase, int qn) {
    WindowIndex& W = S.scan.W;
    LongScan r;
    const unsigned long long lo = cur & ~15ull;
    WinGeom g = make_geom(lo, kWin, cur, p.end);
    __syncthreads();
    if (threadIdx.x == 0) W.bad_byte = INT_MAX;
    load_window(W, &S.mbar, p.text, lo, g.loaded, phase, true);
    if (threadIdx.x == 32) {
        // a long run continues right behind this window: pull the next one into L2 meanwhile
        const unsigned long long nb = lo + (unsigned long long)g.loaded;
        const unsigned long long up = (p.end + 15ull) & ~15ull;
        if (nb < up) tma_prefetch_l2(p.text + nb, (uint32_t)(up - nb < (unsigned long long)kWin ? up - nb : (unsigned long long)kWin));
    }
    finish_geom(W, g, p.final_chunk != 0);
    r.giant = false;
    if (!scan_rows<kLongWarps>(W, g)) {
        if (threadIdx.x == 0) report(p.ctr, DE_BAD_FIELD_COUNT, lo);
        r.ncomplete = 0, r.eskip = 0, r.d = 0, r.next = p.end, r.at_end = true;
        return r;
    }
    const int n_starts = W.n_starts, n_ends = W.n_ends;
    r.eskip = (n_ends > 0 && (n_starts == 0 || W.row_e[0] < W.row_s[0])) ? 1 : 0;
    r.ncomplete = n_starts < n_ends - r.eskip ? n_starts : n_ends - r.eskip;
    int first_other = r.ncomplete;
    for (int i = threadIdx.x; i < r.ncomplete; i += kLongThreads) {
        const int st = W.row_s[i];
        const int len = (int)W.row_e[i + r.eskip] - st;
        LightRow lr;
        {
            int64_t fb;
            int fq;
            if (parse_row_fast(W.win, reinterpret_cast<const uint32_t*>(W.tabm), reinterpret_cast<const uint32_t*>(W.digm), st, st + len, fb, fq)) {
                lr.bits = fb, lr.q_len = (uint16_t)fq, lr.err = DE_NONE;
            } else
                lr = parse_row_masked(W.win, reinterpret_cast<const uint64_t*>(W.tabm), reinterpret_cast<const uint64_t*>(W.digm), st, st + len);
        }
        const bool sm = qn > 0 ? same_query_cached(W.win + st, len, S.qid, qn) : same_query(W.win + st, len, p.text, s, p.end);
        if (lr.err && sm) report(p.ctr, lr.err, lo + st);
        S.scan.bits[i] = lr.bits;
        S.scan.same[i] = sm;
        if (!sm && i < first_other) first_other = i;
    }
#pragma unroll
    for (int dd = 16; dd > 0; dd >>= 1) {
        int o = __shfl_xor_sync(0xffffffffu, first_other, dd);
        first_other = o < first_other ? o : first_other;
    }
    if ((threadIdx.x & 31) == 0) S.red_first[threadIdx.x >> 5] = first_other;
    __syncthreads();
    int d = r.ncomplete;
    for (int i = 0; i < kLongWarps; i++) d = S.red_first[i] < d ? S.red_first[i] : d;
    r.d = d;
    if (W.bad_byte != INT_MAX && threadIdx.x == 0) {
        // only bytes of this run's rows are ours to report
        const int run_end = d < r.ncomplete ? (int)W.row_s[d] : (n_starts > r.ncomplete ? (int)W.row_s[r.ncomplete] : g.L);
        if (W.bad_byte < run_end) report(p.ctr, DE_QUOTE_OR_CR, lo + (unsigned)W.bad_byte);
    }
    if (n_starts > r.ncomplete) {
        r.next = lo + W.row_s[r.ncomplete];
        r.at_end = false;
        if (r.ncomplete == 0) r.giant = !g.covers_eof || !p.final_chunk;  // partial row only: too long, or chunk tail
        if (g.covers_eof) r.at_end = true;
    } else {
        r.next = r.ncomplete > 0 ? lo + W.row_e[r.ncomplete - 1 + r.eskip] + 1 : p.end;
        r.at_end = g.covers_eof || r.next >= p.end;
    }
    __syncthreads();
    return r;
}

// ---- block-wide primitives of the long-run kernel's consensus ----------------------------------------------------------
// Bitonic sort of the 16-bit indices idx[0, n2) (n2 a power of two; the padding entries hold 0xFFFF and sort last) by a
// strict total order `less`.  All threads of the CTA call.
template <class Less>
__device__ __forceinline__ void block_bitonic_u16(uint16_t* idx, int n2, Less less) {
    for (int k = 2; k <= n2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = threadIdx.x; t < (n2 >> 1); t += kLongThreads) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int l = i | j;
                const uint16_t x = idx[i], y = idx[l];
                const bool up = (i & k) == 0;
                // lt(u, v): u sorts in front of v
                const uint16_t u = up ? y : x, v = up ? x : y;
                const bool sw = u != 0xFFFFu && (v == 0xFFFFu || less((int)u, (int)v));
                if (sw) {
                    idx[i] = y;
                    idx[l] = x;
                }
            }
            __syncthreads();
        }
}

// out[i] = f(0) + ... + f(i-1) for i in [0, n], out[n] = total (16-bit: totals stay below 65536).  All threads call.
template <class F>
__device__ __forceinline__ int block_excl_scan_u16(uint16_t* out, int n, F f, int* warp_tot) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + kLongThreads - 1) / kLongThreads;
    const int b = tid * per < n ? tid * per : n, e = b + per < n ? b + per : n;
    int sum = 0;
    for (int i = b; i < e; i++) sum += f(i);
    int inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    int base = 0, total = 0;
    for (int k = 0; k < kLongWarps; k++) {
        if (k < warp) base += warp_tot[k];
        total += warp_tot[k];
    }
    int run = base + inc - sum;
    for (int i = b; i < e; i++) {
        out[i] = (uint16_t)run;
        run += f(i);
    }
    if (tid == 0) out[n] = (uint16_t)total;
    __syncthreads();
    return total;
}

__device__ __forceinline__ bool acc_equal(const TopRow& a, const TopRow& b, const uint8_t* text) {
    return a.acc_len == b.acc_len && bytes_cmp(text + a.acc_off, a.acc_len, text + b.acc_off, b.acc_len) == 0;
}

// Block-parallel multi-taxa consensus of a top group of g >= 2 joined rows (file order, global scratch): the same result
// as the serial consensus_multi() of blu_core.cuh (find_multi_taxa_consensus.rs:22-217, build_blast_consensus_identity.rs,
// consensus_result.rs:65-88), computed with block-wide sorts and scans so that a group of thousands of rows (BASELINE
// config C4 allows 5000 hits per query) costs a few hundred microseconds instead of a serial quadratic walk.
// Returns the soft error (uniform), or DE_NONE after the record, its beans and accession references have been written.
__device__ uint32_t long_consensus(LongSmem& S, const RunParams& p, const TopRow* rows, int g, unsigned long long s, uint32_t qlen,
                                   unsigned long long nrows, long long mx) {
    LongSort& Q = S.sort;
    const LinTables& T = p.T;
    const int tid = threadIdx.x, lane = tid & 31;
    int n2 = 2;
    while (n2 < g) n2 <<= 1;
    // ---- S = the top group sorted by (lineage length, pident, align length, accession; file order)   fmtc.rs:39-54 ----
    for (int i = tid; i < n2; i += kLongThreads) Q.order[i] = i < g ? (uint16_t)i : (uint16_t)0xFFFFu;
    if (tid == 0) {
        S.bcast[5] = INT_MAX;
        S.bcast64[0] = 0ull;
    }
    __syncthreads();
    block_bitonic_u16(Q.order, n2, [&](int a, int b) { return row_less(rows, p.text, a, b); });
    const TopRow ref = rows[p.strategy == BLU_STRATEGY_CAUTIOUS ? Q.order[0] : Q.order[g - 1]];  // fmtc.rs:60-63
    const int m = rows[Q.order[0]].lin_len;  // shortest lineage: levels >= m are never looked at
    // ---- level walk (fmtc.rs:137-214): first level at which the level keys disagree; max pident folded from 0.0 ----------
    {
        const uint32_t lin0 = rows[0].lin;
        const uint32_t o0 = T.lin_off[lin0];
        int myd = INT_MAX;
        double mypid = 0.0;
        for (int r = tid; r < g; r += kLongThreads) {
            const TopRow x = rows[r];
            if (x.pident > mypid) mypid = x.pident;
            if (x.lin != lin0) {
                const uint32_t o = T.lin_off[x.lin];
                for (int i = 0; i < m && i < myd; i++)
                    if (T.lvl_key[o + i] != T.lvl_key[o0 + i]) {
                        myd = i;
                        break;
                    }
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const int od = __shfl_xor_sync(0xffffffffu, myd, d);
            const double op = __shfl_xor_sync(0xffffffffu, mypid, d);
            myd = od < myd ? od : myd;
            mypid = op > mypid ? op : mypid;
        }
        if (lane == 0) {
            if (myd != INT_MAX) atomicMin(&S.bcast[5], myd);
            if (mypid > 0.0) atomicMax(&S.bcast64[0], (unsigned long long)__double_as_longlong(mypid));  // positive doubles order like their bits
        }
        __syncthreads();
    }
    const int diverge = S.bcast[5] == INT_MAX ? -1 : S.bcast[5];
    if (diverge == 0) return DE_ROOT_DISAGREE;
    double identity;
    int idx, level;
    bool single;
    if (diverge > 0) {
        identity = __longlong_as_double((long long)S.bcast64[0]), idx = diverge - 1, level = diverge, single = false;
    } else {
        identity = ref.pident, idx = m - 1, level = m - 1, single = true;
    }
    // ---- bean folding at `level` in S order (consensus_result.rs:65-88) ----------------------------------------------
    for (int i = tid; i < n2; i += kLongThreads) {
        Q.bord[i] = i < g ? (uint16_t)i : (uint16_t)0xFFFFu;
        if (i < g) Q.key[i] = T.bean_key[T.lin_off[rows[Q.order[i]].lin] + level];
    }
    __syncthreads();
    block_bitonic_u16(Q.bord, n2, [&](int a, int b) { return Q.key[a] != Q.key[b] ? Q.key[a] < Q.key[b] : a < b; });
    // flags per position of `bord`: bit 0 = first of its bean, bit 1 = accession kept (Vec::dedup drops an accession equal
    // to its predecessor in the bean's S-ordered list)
    for (int i = tid; i < g; i += kLongThreads) {
        const bool head = i == 0 || Q.key[Q.bord[i]] != Q.key[Q.bord[i - 1]];
        const bool kept = head || !acc_equal(rows[Q.order[Q.bord[i]]], rows[Q.order[Q.bord[i - 1]]], p.text);
        Q.tmp[i] = (uint16_t)((head ? 1 : 0) | (kept ? 2 : 0));
    }
    __syncthreads();
    const int nb = block_excl_scan_u16(Q.hb, g, [&](int i) { return (int)(Q.tmp[i] & 1u); }, S.scan_tot);
    const int nkept = block_excl_scan_u16(Q.kp, g, [&](int i) { return (int)((Q.tmp[i] >> 1) & 1u); }, S.scan_tot);
    for (int i = tid; i < g; i += kLongThreads) {
        const bool head = (Q.tmp[i] & 1u) != 0;
        if (head) Q.st[Q.hb[i]] = (uint16_t)i;  // (hb is exclusive here: the bean's number)
    }
    if (tid == 0) Q.st[nb] = (uint16_t)g;
    __syncthreads();
    for (int i = tid; i < g; i += kLongThreads) Q.hb[i] = (uint16_t)(Q.hb[i] + (Q.tmp[i] & 1u));  // inclusive: bean number + 1
    // ---- beans in output order: occurrences desc, identifier asc (bbci.rs:50-60), ties on the key id ----------------------
    int nb2 = 2;
    while (nb2 < nb) nb2 <<= 1;
    for (int j = tid; j < nb2; j += kLongThreads) Q.bsort[j] = j < nb ? (uint16_t)j : (uint16_t)0xFFFFu;
    __syncthreads();
    block_bitonic_u16(Q.bsort, nb2, [&](int a, int b) {
        const int oa = (int)Q.st[a + 1] - (int)Q.st[a], ob = (int)Q.st[b + 1] - (int)Q.st[b];
        if (oa != ob) return oa > ob;
        const uint32_t pa = T.lin_off[rows[Q.order[Q.bord[Q.st[a]]]].lin] + (uint32_t)level, pb = T.lin_off[rows[Q.order[Q.bord[Q.st[b]]]].lin] + (uint32_t)level;
        const uint32_t ia = T.ident_rank[pa], ib = T.ident_rank[pb];
        if (ia != ib) return ia < ib;
        return Q.key[Q.bord[Q.st[a]]] < Q.key[Q.bord[Q.st[b]]];
    });
    // first accession of every bean: exclusive scan of the kept counts in output order, scattered back to bean numbers
    block_excl_scan_u16(Q.tmp, nb, [&](int j) { const int bb = Q.bsort[j]; return (int)Q.kp[Q.st[bb + 1]] - (int)Q.kp[Q.st[bb]]; }, S.scan_tot);
    for (int j = tid; j < nb; j += kLongThreads) Q.abeg[Q.bsort[j]] = Q.tmp[j];
    // ---- output: one record, nb beans, nkept accession references, all compact --------------------------------------------
    if (tid == 0) {
        const unsigned long long ri = atomicAdd(&p.ctr->rec_count, 1ull);
        const unsigned long long bb = atomicAdd(&p.ctr->bean_used, (unsigned long long)nb);
        const unsigned long long ab = atomicAdd(&p.ctr->acc_used, (unsigned long long)nkept);
        S.bcast64[1] = ri, S.bcast64[2] = bb, S.bcast64[3] = ab;
        if (ri >= p.rec_cap || bb + (unsigned long long)nb > p.bean_cap || ab + (unsigned long long)nkept > p.acc_cap) {
            p.ctr->cap_overflow = 1;
            S.bcast64[1] = ~0ull;
        }
    }
    __syncthreads();
    if (S.bcast64[1] == ~0ull) return DE_NONE;  // the host grows the arrays and reruns
    const unsigned long long ri = S.bcast64[1], bean_base = S.bcast64[2], acc_base = S.bcast64[3];
    for (int j = tid; j < nb; j += kLongThreads) {
        const int bb = Q.bsort[j];
        blu_bean bn;
        bn.first_lineage = rows[Q.order[Q.bord[Q.st[bb]]]].lin;
        bn.occurrences = (uint32_t)((int)Q.st[bb + 1] - (int)Q.st[bb]);
        bn.acc_begin = Q.abeg[bb];
        bn.n_acc = (uint32_t)((int)Q.kp[Q.st[bb + 1]] - (int)Q.kp[Q.st[bb]]);
        p.beans[bean_base + j] = bn;
    }
    for (int i = tid; i < g; i += kLongThreads)
        if (Q.kp[i + 1] != Q.kp[i]) {
            const int bb = (int)Q.hb[i] - 1;
            const TopRow& x = rows[Q.order[Q.bord[i]]];
            p.accs[acc_base + Q.abeg[bb] + (Q.kp[i] - Q.kp[Q.st[bb]])].ref = (x.acc_off << 16) | (unsigned long long)x.acc_len;
        }
    if (tid == 0) {
        blu_record* rec = p.records + ri;
        rec->query_off = s;
        rec->query_len = qlen;
        rec->n_rows = (uint32_t)nrows;
        rec->bit_score = mx;
        rec->perc_identity = ref.pident;
        rec->ref_lineage = ref.lin;
        rec->bean_base = (uint32_t)bean_base;
        rec->n_beans = (uint32_t)nb;
        rec->acc_base = (uint32_t)acc_base;
        rec->status = 1;
        rec->single_match = 0;
        rec->bean_level = (int8_t)level;
        rec->pad[0] = rec->pad[1] = 0;
        apply_cutoffs(T, ref.lin, identity, single && nb == 1, idx, rec);
    }
    return DE_NONE;
}

__global__ void __launch_bounds__(kLongThreads, 1) longrun_kernel(const __grid_constant__ RunParams p) {
    // (launched behind every tile kernel without a host round trip in between: nothing deferred -> nothing to do)
    if (p.ctr->n_defer == 0) return;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    LongSmem& S = *reinterpret_cast<LongSmem*>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned long long p_begin = p.begin == kBeginFromCounters ? p.ctr->next_begin : p.begin;
    if (tid == 0) mbar_init(&S.mbar, 1);
    __syncthreads();
    uint32_t phase = 0;
    const unsigned n_defer = p.ctr->n_defer < p.defer_cap ? p.ctr->n_defer : p.defer_cap;
    TopRow* const rows = p.big_rows + (size_t)blockIdx.x * kLongTopCap;
    unsigned long long* const cand = p.big_cand + (size_t)blockIdx.x * kLongTopCap;

    while (true) {
        __syncthreads();
        if (tid == 0) S.bcast[0] = (int)atomicAdd(&p.ctr->work_ticket, 1u);
        __syncthreads();
        const unsigned wi = (unsigned)S.bcast[0];
        if (wi >= n_defer) break;
        const unsigned long long entry = p.defer[wi];
        const unsigned long long s = entry >> 1;
        // ---- is it really the first row of a run? ------------------------------------------------------------
        if (entry & 1) {
            if (tid == 0) {
                int head = 1;
                if (s > p_begin) {
                    long long q = (long long)s - 1;
                    while (q >= (long long)p_begin && p.text[q] == '\n') q--;  // skip the newline(s) before s
                    if (q >= (long long)p_begin) {
                        long long st = q;
                        while (st > (long long)p_begin && p.text[st - 1] != '\n') st--;
                        // compare first fields of rows at st and s
                        head = 0;
                        for (unsigned long long i = 0;; i++) {
                            if (s + i >= p.end || (unsigned long long)st + i > (unsigned long long)q) {
                                head = 1;
                                break;
                            }
                            uint8_t a = p.text[st + i], b = p.text[s + i];
                            if (a != b) {
                                head = 1;
                                break;
                            }
                            if (a == '\t') break;
                        }
                    }
                }
                S.bcast[1] = head;
            }
            __syncthreads();
            if (!S.bcast[1]) continue;
        }
        // ---- the run's query id (with its tab) is compared against every row: keep it in shared memory ---------------
        if (tid == 0) {
            int qn = 0;
            while (qn < kQidCache && s + qn < p.end) {
                const uint8_t b = p.text[s + qn];
                S.qid[qn++] = b;
                if (b == '\t') break;
            }
            S.bcast[4] = (qn > 0 && S.qid[qn - 1] == '\t') ? qn : 0;  // 0: id longer than the cache -> compare in global memory
        }
        __syncthreads();
        const int qn = S.bcast[4];
        // ---- single pass: extent, max bit score, and the rows that carry it (candidate list reset on a new maximum) --
        long long mx = LLONG_MIN;
        long long cnt = 0, nrows = 0;
        unsigned long long cur = s;
        bool ended = false, hit_end = false, fail = false;
        while (true) {
            LongScan sc = long_scan(S, p, s, cur, phase, qn);
            if (sc.giant && sc.d == 0 && sc.ncomplete == 0) {
                // an unterminated row: either the chunk tail (carried over) or a row longer than the window
                if (!sc.at_end || p.final_chunk) {
                    if (tid == 0) report(p.ctr, DE_CARRY_TOO_BIG, cur);
                    fail = true;
                }
                hit_end = true;
                break;
            }
            const unsigned long long lo = cur & ~15ull;
            // maximum of this window's rows of the run
            long long lm = LLONG_MIN;
            for (int i = tid; i < sc.d; i += kLongThreads) {
                const long long b = S.scan.bits[i];
                lm = b > lm ? b : lm;
            }
#pragma unroll
            for (int dd = 16; dd > 0; dd >>= 1) {
                const long long om = __shfl_xor_sync(0xffffffffu, lm, dd);
                lm = om > lm ? om : lm;
            }
            if (lane == 0) S.red_max[warp] = lm;
            __syncthreads();
            long long wm = LLONG_MIN;
            for (int i = 0; i < kLongWarps; i++) wm = S.red_max[i] > wm ? S.red_max[i] : wm;
            if (sc.d > 0 && wm > mx) {
                mx = wm;
                cnt = 0;  // earlier candidates are beaten
            }
            // append this window's rows with bits == mx, in file order
            for (int b0 = 0; b0 < sc.d; b0 += kLongThreads) {
                const int i = b0 + tid;
                const bool top = i < sc.d && S.scan.bits[i] == mx;
                const unsigned bal = __ballot_sync(0xffffffffu, top);
                if (lane == 0) S.red_cnt[warp] = __popc(bal);
                __syncthreads();
                long long before = cnt;
                int total = 0;
                for (int k = 0; k < kLongWarps; k++) {
                    if (k < warp) before += S.red_cnt[k];
                    total += S.red_cnt[k];
                }
                if (top) {
                    const long long pos = before + __popc(bal & ((1u << lane) - 1u));
                    if (pos < kLongTopCap)
                        cand[pos] = ((lo + S.scan.W.row_s[i]) << 16) |
                                    (unsigned long long)(uint32_t)((int)S.scan.W.row_e[i + sc.eskip] - (int)S.scan.W.row_s[i]);  // (a row fits the window: < 65536 bytes)
                }
                cnt += total;
                __syncthreads();
            }
            nrows += sc.d;
            if (sc.d < sc.ncomplete) {
                ended = true;
                break;
            }
            if (sc.at_end) {
                hit_end = true;
                break;
            }
            cur = sc.next;
        }
        if (fail) continue;
        if (!ended && hit_end && !p.final_chunk) {
            if (tid == 0) atomicMin(&p.ctr->tail_start, s);  // carried into the next chunk
            continue;
        }
        if (nrows == 0) continue;
        if (cnt > kLongTopCap) {
            if (tid == 0) report(p.ctr, DE_TOPGROUP_TOO_BIG, s);
            continue;
        }
        const int gcount = (int)cnt;
        // ---- join the top rows (read back from the text; they are few) -----------------------------------------------
        uint32_t my_err = 0;
        unsigned long long my_off = 0;
        for (int i = tid; i < gcount; i += kLongThreads) {
            const unsigned long long off = cand[i] >> 16;
            const uint32_t err = heavy_parse_row(p.text + off, (int)(cand[i] & 0xFFFFull), off, p.T, rows[i]);
            if (err && !my_err) my_err = err, my_off = off;
        }
        if (my_err) report_soft(p.ctr, my_err, my_off);
        uint32_t soft = __syncthreads_or(my_err != 0) ? 1u : 0u;
        uint32_t ql = 0;
        if (qn > 0)
            ql = (uint32_t)(qn - 1);
        else
            while (s + ql < p.end && p.text[s + ql] != '\t') ql++;
        if (!soft && gcount > 1) {
            const uint32_t ce = long_consensus(S, p, rows, gcount, s, ql, (unsigned long long)nrows, mx);
            if (ce) {
                if (tid == 0) report_soft(p.ctr, ce, s);
                soft = 1;
            }
        }
        if (tid == 0 && (soft || gcount == 1)) {
            // a single top row, or a query whose consensus failed: the record is written here.  A failed query still leaves
            // a record (status 0) so that the duplicate-id check sees its id: a fragment of a scattered query may fail
            // although the merged query would not, and then the table is regrouped and run again.
            const unsigned long long ri = atomicAdd(&p.ctr->rec_count, 1ull);
            unsigned long long bb = 0, ab = 0;
            if (!soft) {
                bb = atomicAdd(&p.ctr->bean_used, 1ull);
                ab = atomicAdd(&p.ctr->acc_used, 1ull);
            }
            if (ri >= p.rec_cap || bb + 1 > p.bean_cap || ab + 1 > p.acc_cap)
                p.ctr->cap_overflow = 1;
            else {
                blu_record* rec = p.records + ri;
                rec->query_off = s;
                rec->query_len = ql;
                rec->n_rows = (uint32_t)nrows;
                rec->keep_mask = 0;
                rec->perc_identity = 0.0;
                rec->bit_score = mx;
                rec->ref_lineage = 0;
                rec->bean_base = (uint32_t)bb;
                rec->n_beans = 0;
                rec->acc_base = (uint32_t)ab;
                rec->status = 0;
                rec->single_match = rec->mutated = 0;
                rec->reached_pos = 0, rec->allowed_pos = -1, rec->bean_level = 0;
                rec->pad[0] = rec->pad[1] = 0;
                if (!soft) {
                    QueryOut out{rec, p.beans + bb, p.accs + ab};
                    const uint32_t ce = consensus_single(rows[0], p.T, out);
                    if (ce) {
                        report_soft(p.ctr, ce, s);
                        rec->status = 0, rec->n_beans = 0;
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// consensus kernel: W lanes per query (W = 8: four queries per warp; W = 32 for top groups of 9..32 rows), lanes = rows
// of the top bit-score group
//   find_multi_taxa_consensus.rs:39-214 + build_blast_consensus_identity.rs:9-105 + consensus_result.rs:65-88
//   (same semantics as the serial consensus_multi() in blu_core.cuh, which the host tests use, and as long_consensus())
// Everything is written so that the four queries of a warp walk through the SAME instructions (loop bounds are the
// warp-wide maxima, a query that is done is merely predicated off): top groups hold 1..8 rows in practice, so one
// query per warp leaves most lanes idle (round 1: 928 warp-instructions per query at 15 active lanes).
// Output is compact: a CTA adds up the beans / accession references of its 32 queries and reserves them with one atomic
// each, so nothing but what the results need is ever downloaded.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int cmp_u64(unsigned long long a, unsigned long long b) { return a < b ? -1 : (a > b ? 1 : 0); }

// bytewise comparison of two accessions given their first 16 bytes as big-endian keys (zero padded)
__device__ __forceinline__ int cmp_acc(unsigned long long a0, unsigned long long a1, unsigned alen, unsigned long long aoff, unsigned long long b0,
                                       unsigned long long b1, unsigned blen, unsigned long long boff, const uint8_t* text) {
    int c = cmp_u64(a0, b0);
    if (c) return c;
    c = cmp_u64(a1, b1);
    if (c) return c;
    if (alen > 16 && blen > 16) {
        const unsigned n = alen < blen ? alen : blen;
        for (unsigned i = 16; i < n; i++) {
            int d = (int)text[aoff + i] - (int)text[boff + i];
            if (d) return d;
        }
    }
    return (int)alen - (int)blen;
}

constexpr int kConsThreads = 128;

// What a lane holds once its query's consensus is computed; written out after the output space has been reserved.
struct ConsLane {
    // lane 0 of the group: the record
    unsigned long long keep_mask;
    double perc_identity;
    uint32_t ref_lineage;
    int nb, nkept;         // beans / kept accession references of the query (0: the query failed or is not this pass's)
    int reached, allowed, level;
    bool mutated, single, ok;
    // every lane: its bean (leaders) and its accession reference (kept rows)
    bool leader, keeps;
    blu_bean bean;
    int bean_idx, acc_idx;
    unsigned long long acc_ref;
};

// `valid`: this group has a record to process in this pass; g = size of its top group (1..W), slot = its first top row.
template <int W>
__device__ __forceinline__ ConsLane cons_compute(const PostParams& p, bool valid, int g, unsigned long long slot, unsigned long long query_off, int lane) {
    const unsigned FULL = 0xffffffffu;
    const LinTables& T = p.T;
    const int sl = lane & (W - 1);
    const int gsh = lane & ~(W - 1);  // first lane of the group
    const unsigned WM = W == 32 ? FULL : ((1u << (W & 31)) - 1u);
    auto seg = [&](unsigned b) { return W == 32 ? b : ((b >> gsh) & WM); };
    const unsigned ltm = (1u << sl) - 1u;
    ConsLane o;
    o.keep_mask = 0, o.perc_identity = 0.0, o.ref_lineage = 0, o.nb = 0, o.nkept = 0, o.reached = 0, o.allowed = -1, o.level = 0;
    o.mutated = false, o.single = false, o.ok = false, o.leader = false, o.keeps = false, o.bean_idx = 0, o.acc_idx = 0, o.acc_ref = 0;
    o.bean.first_lineage = 0, o.bean.occurrences = 0, o.bean.acc_begin = 0, o.bean.n_acc = 0;
    const bool on = valid && sl < g;
    // ---- the rows as the tile kernel left them: the join (left_join on subject_taxid == taxid, mod.rs:72-76) ------------
    TopRow r;
    r.pident = 0.0, r.alnlen = 0, r.acc_off = 0, r.lin = 0, r.acc_len = 0, r.lin_len = 0;
    uint32_t pos0 = 0, jerr = 0;
    if (on) {
        const TopRowRaw raw = p.toprows[slot + sl];
        const unsigned long long off = raw.acc_off;
        if (raw.dec_frac == kTopRowUnparsed)  // a row of unusual shape: split and parsed here by the full parser (acc_off / acc_len are the ROW's)
            jerr = off + (unsigned long long)raw.acc_len <= p.text_end ? heavy_parse_row(p.text + off, (int)raw.acc_len, off, T, r) : (uint32_t)DE_INTERNAL;
        else
            jerr = join_top_row(raw, T, r);
        if (jerr)
            report_soft(p.ctr, jerr, off);
        else
            pos0 = T.lin_off[r.lin];
    }
    bool failed = seg(__ballot_sync(FULL, jerr != 0)) != 0;
    const bool live = valid && !failed;
    // ---- first 16 accession bytes as big-endian keys ---------------------------------------------------------------
    unsigned long long k0 = 0, k1 = 0;
    if (on && !failed && g > 1) {
        // five aligned words cover the 16 bytes at any alignment (the row goes on for >= 20 bytes behind saccver, so the
        // reads stay inside the text); realigned by funnel shifts, byte-swapped to big-endian, bytes beyond the accession zeroed
        const unsigned n = r.acc_len;
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(p.text + (r.acc_off & ~3ull));
        const uint32_t sh8 = (uint32_t)(r.acc_off & 3ull) * 8u;
        const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = wp[4];
        const uint32_t q0 = __byte_perm(__funnelshift_r(w0, w1, sh8), 0u, 0x0123), q1 = __byte_perm(__funnelshift_r(w1, w2, sh8), 0u, 0x0123),
                       q2 = __byte_perm(__funnelshift_r(w2, w3, sh8), 0u, 0x0123), q3 = __byte_perm(__funnelshift_r(w3, w4, sh8), 0u, 0x0123);
        k0 = ((unsigned long long)q0 << 32) | (unsigned long long)q1;
        k1 = ((unsigned long long)q2 << 32) | (unsigned long long)q3;
        if (n < 16) k1 = n > 8 ? (k1 & (~0ull << (8u * (16u - n)))) : 0ull;
        if (n < 8) k0 = n > 0 ? (k0 & (~0ull << (8u * (8u - n)))) : 0ull;
    }
    // ---- S = stable sort by (lineage length, pident, align length, accession)   fmtc.rs:39-54 ----------------------
    int gmax = live ? g : 0;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const int t = __shfl_xor_sync(FULL, gmax, d);
        gmax = t > gmax ? t : gmax;
    }
    if (gmax > 1) {
        int rank = 0;
        for (int j = 0; j < gmax; j++) {
            const int len_j = __shfl_sync(FULL, (int)r.lin_len, j, W);
            const double pid_j = __shfl_sync(FULL, r.pident, j, W);
            const long long aln_j = __shfl_sync(FULL, (long long)r.alnlen, j, W);
            const unsigned long long k0_j = __shfl_sync(FULL, k0, j, W), k1_j = __shfl_sync(FULL, k1, j, W);
            const unsigned alen_j = __shfl_sync(FULL, (unsigned)r.acc_len, j, W);
            const unsigned long long off_j = __shfl_sync(FULL, (unsigned long long)r.acc_off, j, W);
            if (on && live && j < g && j != sl) {
                bool lt;
                if (len_j != (int)r.lin_len)
                    lt = len_j < (int)r.lin_len;
                else if (pid_j < r.pident)
                    lt = true;
                else if (pid_j > r.pident)
                    lt = false;
                else if (aln_j != (long long)r.alnlen)
                    lt = aln_j < (long long)r.alnlen;
                else {
                    const int c = cmp_acc(k0_j, k1_j, alen_j, off_j, k0, k1, r.acc_len, r.acc_off, p.text);
                    lt = c < 0 || (c == 0 && j < sl);
                }
                if (lt) rank++;
            }
        }
        // move the row of rank s into lane s
        int src = sl;
        for (int j = 0; j < gmax; j++) {
            const int rj = __shfl_sync(FULL, rank, j, W);
            if (on && live && j < g && rj == sl) src = j;
        }
        r.pident = __shfl_sync(FULL, r.pident, src, W);
        r.alnlen = __shfl_sync(FULL, (long long)r.alnlen, src, W);
        r.acc_off = __shfl_sync(FULL, (unsigned long long)r.acc_off, src, W);
        r.lin = __shfl_sync(FULL, r.lin, src, W);
        r.acc_len = (uint16_t)__shfl_sync(FULL, (unsigned)r.acc_len, src, W);
        r.lin_len = (uint16_t)__shfl_sync(FULL, (unsigned)r.lin_len, src, W);
        pos0 = __shfl_sync(FULL, pos0, src, W);
        k0 = __shfl_sync(FULL, k0, src, W);
        k1 = __shfl_sync(FULL, k1, src, W);
    }
    // ---- reference row + level walk (fmtc.rs:60-63,137-214) ----------------------------------------------------------
    const int ref_lane = p.strategy == BLU_STRATEGY_CAUTIOUS ? 0 : (g > 0 ? g - 1 : 0);
    const int m = __shfl_sync(FULL, (int)r.lin_len, 0, W);  // shortest lineage
    const uint32_t lin0 = __shfl_sync(FULL, r.lin, 0, W);
    const unsigned dm = seg(__ballot_sync(FULL, on && r.lin != lin0));
    const bool differ = live && g > 1 && dm != 0;
    int diverge = -1;
    {
        int mmax = differ ? m : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const int t = __shfl_xor_sync(FULL, mmax, d);
            mmax = t > mmax ? t : mmax;
        }
        for (int i0 = 0; i0 < mmax; i0 += 4) {
            // four levels at a time: the loads go out together, then the votes
            uint32_t key[4];
#pragma unroll
            for (int u = 0; u < 4; u++) key[u] = (on && differ && diverge < 0 && i0 + u < m) ? T.lvl_key[pos0 + i0 + u] : 0u;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint32_t key0 = __shfl_sync(FULL, key[u], 0, W);
                const bool mism = on && differ && i0 + u < m && key[u] != key0;
                const unsigned bm = seg(__ballot_sync(FULL, mism));
                if (bm && diverge < 0) diverge = i0 + u;
            }
            if (__all_sync(FULL, !differ || diverge >= 0)) break;
        }
    }
    if (live && diverge == 0) {
        if (sl == 0) report_soft(p.ctr, DE_ROOT_DISAGREE, query_off);
        failed = true;
    }
    double identity;
    int idx, level;
    bool single;
    const double ref_pid = __shfl_sync(FULL, r.pident, ref_lane, W);
    double mxp = on ? r.pident : 0.0;  // max pident of the group, folded from 0.0 (fmtc.rs:182-185)
    if (!(mxp > 0.0)) mxp = 0.0;
#pragma unroll
    for (int d = W / 2; d > 0; d >>= 1) {
        const double t = __shfl_xor_sync(FULL, mxp, d);
        mxp = t > mxp ? t : mxp;
    }
    if (diverge > 0)
        identity = mxp, idx = diverge - 1, level = diverge, single = false;
    else
        identity = ref_pid, idx = m - 1, level = m - 1, single = true;
    const bool go = valid && !failed;
    // ---- fold beans at `level` in S order (consensus_result.rs:65-88) -----------------------------------------------
    unsigned long long mkey = 0x8000000000000000ull | (unsigned long long)lane;  // lanes without a row match nobody
    uint32_t bkey = 0, irank = 0;
    if (on && go) {
        bkey = T.bean_key[pos0 + level];
        irank = T.ident_rank[pos0 + level];
        mkey = ((unsigned long long)(gsh + 1) << 32) | (unsigned long long)bkey;
    }
    const unsigned grp = seg(__match_any_sync(FULL, mkey));  // (relative to the group's first lane)
    const unsigned below = grp & ltm;
    const bool leader = on && go && below == 0;
    const int occ = __popc(grp);
    // Vec::dedup: an accession equal to its predecessor in the bean's S-ordered list is dropped
    const int pl = below ? 31 - __clz(below) : sl;
    const unsigned long long pk0 = __shfl_sync(FULL, k0, pl, W), pk1 = __shfl_sync(FULL, k1, pl, W);
    const unsigned plen = __shfl_sync(FULL, (unsigned)r.acc_len, pl, W);
    const unsigned long long poff = __shfl_sync(FULL, (unsigned long long)r.acc_off, pl, W);
    bool dropped = false;
    if (on && go && below) dropped = plen == r.acc_len && cmp_acc(pk0, pk1, plen, poff, k0, k1, r.acc_len, r.acc_off, p.text) == 0;
    const unsigned kept = seg(__ballot_sync(FULL, on && go && !dropped));
    const int nacc_bean = __popc(grp & kept);
    const int my_idx = __popc(grp & kept & ltm);
    // sort beans: occurrences desc, identifier asc (bbci.rs:50-60); deterministic tie-break on the key id
    const unsigned lm = seg(__ballot_sync(FULL, leader));
    int brank = 0, acc_begin = 0;
    {
        int jmax = go ? g : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const int t = __shfl_xor_sync(FULL, jmax, d);
            jmax = t > jmax ? t : jmax;
        }
        for (int j = 0; j < jmax; j++) {
            const int occ_j = __shfl_sync(FULL, occ, j, W);
            const uint32_t ir_j = __shfl_sync(FULL, irank, j, W), bk_j = __shfl_sync(FULL, bkey, j, W);
            const int na_j = __shfl_sync(FULL, nacc_bean, j, W);
            if (leader && ((lm >> j) & 1u) && j != sl) {
                const bool better = occ_j != occ ? occ_j > occ : (ir_j != irank ? ir_j < irank : bk_j < bkey);
                if (better) {
                    brank++;
                    acc_begin += na_j;
                }
            }
        }
    }
    const int my_begin = __shfl_sync(FULL, acc_begin, grp ? __ffs(grp) - 1 : 0, W);
    const int nb = __popc(lm);
    // ---- rank selection on the reference lineage (bbci.rs:22-37,66-95; single match: fsqc.rs:74-150), lanes = positions --
    const uint32_t ref_lin = __shfl_sync(FULL, r.lin, ref_lane, W);
    const uint32_t ref_o = __shfl_sync(FULL, pos0, ref_lane, W);
    const int ref_k = __shfl_sync(FULL, (int)r.lin_len, ref_lane, W);
    unsigned long long ge = 0, notgt = 0;
    {
        int kmax = go ? ref_k : 0;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const int t = __shfl_xor_sync(FULL, kmax, d);
            kmax = t > kmax ? t : kmax;
        }
        for (int j0 = 0; j0 < kmax; j0 += W) {
            const int j = j0 + sl;
            const bool in = go && j < ref_k;
            double c = 0.0;
            if (in) c = T.cut[ref_o + j];
            const unsigned b_ge = seg(__ballot_sync(FULL, in && identity >= c));    // linnaean_ranks.rs:208
            const unsigned b_ng = seg(__ballot_sync(FULL, in && !(identity > c)));  // linnaean_ranks.rs:188
            ge |= (unsigned long long)b_ge << j0;
            notgt |= (unsigned long long)b_ng << j0;
        }
    }
    if (go && g == 1 && !ge) {
        if (sl == 0) report_soft(p.ctr, DE_EMPTY_ADJUSTED, query_off);
        failed = true;
    }
    o.ok = valid && !failed;
    if (!o.ok) return o;
    o.leader = leader;
    o.keeps = on && !dropped;
    o.bean.first_lineage = r.lin, o.bean.occurrences = (uint32_t)occ, o.bean.acc_begin = (uint32_t)acc_begin, o.bean.n_acc = (uint32_t)nacc_bean;
    o.bean_idx = brank;
    o.acc_idx = my_begin + my_idx;
    o.acc_ref = (r.acc_off << 16) | (unsigned long long)r.acc_len;
    o.nb = nb;
    o.nkept = __popc(kept);
    o.ref_lineage = ref_lin;
    o.level = level;
    if (g == 1) {
        const int last = 63 - __clzll((long long)ge);
        o.keep_mask = ge, o.perc_identity = ref_pid, o.single = true, o.mutated = false, o.reached = last, o.allowed = -1, o.level = last;
    } else {
        const int allowed = notgt ? (__ffsll((long long)notgt) - 1) : -1;
        unsigned long long mask = ge;
        if (!(single && nb == 1)) {
            // keep the first idx+1 survivors: enumerate AFTER the filter, take_while(index <= bean_index)
            unsigned long long mk = 0, rest = ge;
            for (int n = 0; n <= idx && rest; n++) {
                const unsigned long long low = rest & (~rest + 1);
                mk |= low;
                rest ^= low;
            }
            mask = mk;
        }
        const int last = mask ? 63 - __clzll((long long)mask) : -1;
        o.keep_mask = mask, o.perc_identity = ref_pid, o.single = false, o.allowed = allowed, o.reached = last >= 0 ? last : idx;
        o.mutated = sl == 0 && allowed >= 0 && T.rank_cls[ref_o + idx] != T.allowed_cls[ref_o + allowed];
    }
    return o;
}

// the record fields the consensus decides (everything but where its beans / accession references end up)
__device__ __forceinline__ void cons_write_record(blu_record* rec, const ConsLane& o) {
    if (o.ok) {
        rec->keep_mask = o.keep_mask;
        rec->perc_identity = o.perc_identity;
        rec->ref_lineage = o.ref_lineage;
        rec->n_beans = (uint32_t)o.nb;
        rec->single_match = o.single ? 1 : 0;
        rec->mutated = o.mutated ? 1 : 0;
        rec->reached_pos = (int8_t)o.reached;
        rec->allowed_pos = (int8_t)o.allowed;
        rec->bean_level = (int8_t)o.level;
        rec->status = 1;
    } else {
        // a failed query keeps its id (the duplicate-id check must see it) and owns no beans / accession references
        rec->bean_base = 0, rec->n_beans = 0, rec->acc_base = 0;
        rec->status = 0;
    }
}

constexpr int kConsWarps = kConsThreads / 32;
constexpr int kConsBatch = 32;  // queries a warp finishes between two reservations of output space

// per-warp staging of one batch's beans / accession references (a narrow query has at most 8 of each)
struct ConsStage {
    blu_bean beans[kConsBatch][8];
    unsigned long long accs[kConsBatch][8];
    int nb[kConsBatch], na[kConsBatch];
    uint8_t list[kConsBatch];  // the batch's narrow queries (top groups of 1..8 rows) in the order of their top-group size
};

#ifndef BLU_CONS_SORTED
#define BLU_CONS_SORTED 1
#endif

// (64 registers, 8 CTAs = 32 warps per SM: the kernel waits on memory, occupancy decides -- measured per million queries:
// 106 registers 0.92 ms, 95: 0.87, 80: 0.71, 72: 0.68, 64 (a few spills): 0.615)
#ifndef BLU_CONS_MINB
#define BLU_CONS_MINB 8
#endif
__global__ void __launch_bounds__(kConsThreads, BLU_CONS_MINB) consensus_kernel(const __grid_constant__ PostParams p) {
    __shared__ ConsStage stage_all[kConsWarps];
    const unsigned FULL = 0xffffffffu;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    const int sub = lane >> 3, sl8 = lane & 7;
    ConsStage& St = stage_all[warp];
    if (p.ctr->cap_overflow) return;  // the tile kernel ran out of space: the host grows the arrays and reruns
    const unsigned long long rb = p.ctr->post_done;
    unsigned long long re = p.ctr->rec_count;
    if (re > p.rec_cap) re = p.rec_cap;
    unsigned long long rows_sum = 0;
    const unsigned long long gw = (unsigned long long)blockIdx.x * kConsWarps + (unsigned long long)warp;
    const unsigned long long wstride = (unsigned long long)gridDim.x * kConsWarps * kConsBatch;
    // A warp finishes 32 queries at a time: lane = query for the headers (all 32 records are requested at once), then rounds of
    // four queries, 8 lanes per query, taken in the order of their top-group size -- the loops of a round run to the largest
    // top group among its four queries, and half of all queries are single matches: sorted, they share rounds whose loops
    // all collapse (0.615 instead of 0.646 ms per million queries).  Beans / accession references are staged in shared memory, their output space is reserved with one
    // atomic per array and batch, and they are copied out compactly: no CTA-wide barrier anywhere.
    for (unsigned long long base = rb + gw * kConsBatch; base < re; base += wstride) {
        // ---- headers: lane = query ----------------------------------------------------------------------------------------------
        const unsigned long long qi = base + (unsigned long long)lane;
        blu_record* rec = p.records + qi;
        int g = 0, cls = 0;  // cls 1: 1..8 rows, 2: 9..32 rows, 3: more (cannot come from the tile kernel)
        unsigned long long slot = 0, qoff = 0;
        if (qi < re) {
            rows_sum += rec->n_rows;
            if (rec->status == 2) {
                g = (int)rec->n_beans;
                slot = rec->bean_base;
                qoff = rec->query_off;
                if (g >= 1 && slot + (unsigned long long)g <= p.slot_cap) cls = g <= 8 ? 1 : (g <= 32 ? 2 : 3);  // (else: cannot happen without cap_overflow)
            }
        }
        St.nb[lane] = 0, St.na[lane] = 0;
        if (cls == 3) {
            report(p.ctr, DE_INTERNAL, qoff);  // (the tile kernel hands top groups of more than 32 rows to the long-run kernel)
            rec->status = 0, rec->n_beans = 0;
        }
        // ---- the narrow queries, listed by top-group size ------------------------------------------------------------------------
        int n8 = 0;
        {
            int pos = 0;
#pragma unroll
            for (int k = 1; k <= 8; k++) {
                const unsigned mk = __ballot_sync(FULL, cls == 1 && (BLU_CONS_SORTED ? g == k : k == 1));
                if (BLU_CONS_SORTED ? k < g : false) pos += __popc(mk);
                if (BLU_CONS_SORTED ? k == g : k == 1) pos += __popc(mk & lt);
                n8 += __popc(mk);
            }
            if (cls == 1) St.list[pos] = (uint8_t)lane;
        }
        unsigned m32 = __ballot_sync(FULL, cls == 2);
        __syncwarp();
        for (int t = 0; t * 4 < n8; t++) {
            const int at = t * 4 + sub;
            const bool valid = at < n8;
            const int q = valid ? (int)St.list[at] : 0;  // the query's place in the batch == the lane that holds its header
            const int gq = __shfl_sync(FULL, g, q);
            const unsigned long long slotq = __shfl_sync(FULL, slot, q), qoffq = __shfl_sync(FULL, qoff, q);
            const ConsLane o = cons_compute<8>(p, valid, gq, slotq, qoffq, lane);
            if (o.ok && o.leader) St.beans[q][o.bean_idx] = o.bean;
            if (o.ok && o.keeps) St.accs[q][o.acc_idx] = o.acc_ref;
            if (valid && sl8 == 0) {
                St.nb[q] = o.ok ? o.nb : 0;
                St.na[q] = o.ok ? o.nkept : 0;
                cons_write_record(p.records + base + (unsigned long long)q, o);
            }
        }
        __syncwarp();
        // ---- output space for the batch: lane = query -------------------------------------------------------------------------
        const int vb = St.nb[lane], va = St.na[lane];
        int ib = vb, ia = va;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int tb = __shfl_up_sync(FULL, ib, d), ta = __shfl_up_sync(FULL, ia, d);
            if (lane >= d) ib += tb, ia += ta;
        }
        const int tot_b = __shfl_sync(FULL, ib, 31), tot_a = __shfl_sync(FULL, ia, 31);
        unsigned long long bb = 0, ab = 0;
        if (lane == 0) {
            if (tot_b) bb = atomicAdd(&p.ctr->bean_used, (unsigned long long)tot_b);
            if (tot_a) ab = atomicAdd(&p.ctr->acc_used, (unsigned long long)tot_a);
        }
        bb = __shfl_sync(FULL, bb, 0), ab = __shfl_sync(FULL, ab, 0);
        const bool fits = bb + (unsigned long long)tot_b <= p.bean_cap && ab + (unsigned long long)tot_a <= p.acc_cap;
        if (!fits && lane == 0) p.ctr->cap_overflow = 1;
        const unsigned long long my_b = bb + (unsigned long long)(ib - vb), my_a = ab + (unsigned long long)(ia - va);
        if (fits) {
            if (vb > 0) {
                rec->bean_base = (uint32_t)my_b;
                rec->acc_base = (uint32_t)my_a;
            }
            // copy out: 8 lanes per query, four queries per step
            for (int t = 0; t < kConsBatch / 4; t++) {
                const int qslot = t * 4 + sub;
                const unsigned long long qb = __shfl_sync(FULL, my_b, qslot), qa = __shfl_sync(FULL, my_a, qslot);
                const int nbq = __shfl_sync(FULL, vb, qslot), naq = __shfl_sync(FULL, va, qslot);
                if (sl8 < nbq) p.beans[qb + sl8] = St.beans[qslot][sl8];
                if (sl8 < naq) p.accs[qa + sl8].ref = St.accs[qslot][sl8];
            }
        }
        __syncwarp();
        // ---- top groups of 9..32 rows: one query per warp, its own reservation ------------------------------------------------
        while (m32) {
            const int q = __ffs(m32) - 1;
            m32 &= m32 - 1;
            const int gw2 = __shfl_sync(FULL, g, q);
            const unsigned long long slotw = __shfl_sync(FULL, slot, q), qoffw = __shfl_sync(FULL, qoff, q);
            blu_record* recw = p.records + base + (unsigned long long)q;
            const ConsLane ow = cons_compute<32>(p, true, gw2, slotw, qoffw, lane);
            unsigned long long wb = 0, wa = 0;
            int wfits = 1;
            if (lane == 0 && ow.ok) {
                wb = atomicAdd(&p.ctr->bean_used, (unsigned long long)ow.nb);
                wa = atomicAdd(&p.ctr->acc_used, (unsigned long long)ow.nkept);
                wfits = wb + (unsigned long long)ow.nb <= p.bean_cap && wa + (unsigned long long)ow.nkept <= p.acc_cap;
                if (!wfits) p.ctr->cap_overflow = 1;
            }
            wb = __shfl_sync(FULL, wb, 0), wa = __shfl_sync(FULL, wa, 0), wfits = __shfl_sync(FULL, wfits, 0);
            if (ow.ok && wfits) {
                if (ow.leader) p.beans[wb + ow.bean_idx] = ow.bean;
                if (ow.keeps) p.accs[wa + ow.acc_idx].ref = ow.acc_ref;
            }
            if (lane == 0) {
                cons_write_record(recw, ow);
                if (ow.ok && wfits) recw->bean_base = (uint32_t)wb, recw->acc_base = (uint32_t)wa;
            }
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) rows_sum += __shfl_xor_sync(FULL, rows_sum, d);
    if (lane == 0 && rows_sum) atomicAdd(&p.ctr->n_rows, rows_sum);
}

// ---------------------------------------------------------------------------------------------------------------
// gather: query ids + accessions -> string pool (only for results that leave the device without their text)
//   One warp per 32 records: lane = record for the lengths (a warp scan places the 32 records' strings back to back, one
//   atomic reserves the pool space), then the whole warp copies string after string, a byte per lane: reads and writes
//   of one string are one or two sectors instead of a byte-per-thread scatter.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_kernel(const __grid_constant__ PostParams p) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    if (p.ctr->cap_overflow) return;
    const unsigned long long rb = p.ctr->post_done;
    unsigned long long re = p.ctr->rec_count;
    if (re > p.rec_cap) re = p.rec_cap;
    const unsigned long long wstride = (unsigned long long)gridDim.x * (blockDim.x >> 5) * 32ull;
    for (unsigned long long base = rb + ((unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32ull; base < re; base += wstride) {
        const unsigned long long i = base + lane;
        const bool live = i < re;
        blu_record* rec = p.records + i;
        unsigned long long bytes = 0, qoff = 0, abase = 0;
        uint32_t qlen = 0, nacc = 0;
        if (live) {
            qoff = rec->query_off, qlen = rec->query_len;
            bytes = qlen;
            if (rec->status == 1) {
                abase = rec->acc_base;
                const uint32_t nbn = rec->n_beans;
                if (nbn) {
                    const blu_bean lb = p.beans[(unsigned long long)rec->bean_base + nbn - 1];
                    nacc = lb.acc_begin + lb.n_acc;  // the last bean's list ends the record's accession references
                }
                // (beans are stored in output order, their lists back to back: acc_begin is increasing)
                for (uint32_t a = 0; a < nacc; a++) bytes += (uint32_t)(p.accs[abase + a].ref & 0xFFFFull);
            }
        }
        unsigned long long inc = bytes;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long t = __shfl_up_sync(FULL, inc, d);
            if (lane >= d) inc += t;
        }
        const unsigned long long total = __shfl_sync(FULL, inc, 31);
        unsigned long long wbase = 0;
        if (lane == 31 && total) wbase = atomicAdd(&p.ctr->pool_used, total);
        wbase = __shfl_sync(FULL, wbase, 31);
        if (!p.pool) continue;  // counting pass: pool_used ends up as the size the pool needs
        if (wbase + total > p.pool_cap) {
            if (lane == 0) p.ctr->cap_overflow = 1;
            continue;
        }
        const unsigned long long mine = wbase + inc - bytes;  // where this lane's record's strings start
        // ---- copy, string by string, the whole warp on each --------------------------------------------------------------
        uint32_t namax = nacc;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const uint32_t t = __shfl_xor_sync(FULL, namax, d);
            namax = t > namax ? t : namax;
        }
        unsigned long long cur = mine;
        for (int rr = 0; rr < 32; rr++) {
            const unsigned long long so = __shfl_sync(FULL, qoff, rr), dst = __shfl_sync(FULL, cur, rr);
            const uint32_t n = __shfl_sync(FULL, qlen, rr);
            for (uint32_t k = lane; k < n; k += 32) p.pool[dst + k] = p.text[so + k];
        }
        if (live) rec->query_off = mine;
        cur += qlen;
        for (uint32_t a = 0; a < namax; a++) {
            unsigned long long ref = 0;
            if (a < nacc) ref = p.accs[abase + a].ref;
            for (int rr = 0; rr < 32; rr++) {
                const unsigned long long rf = __shfl_sync(FULL, ref, rr), dst = __shfl_sync(FULL, cur, rr);
                const uint32_t n = (uint32_t)(rf & 0xFFFFull);
                const unsigned long long so = rf >> 16;
                for (uint32_t k = lane; k < n; k += 32) p.pool[dst + k] = p.text[so + k];
            }
            if (a < nacc) {
                p.accs[abase + a].ref = (cur << 16) | (ref & 0xFFFFull);
                cur += (uint32_t)(ref & 0xFFFFull);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// duplicate query detection (reference groups by a HashMap<String,_>, mod.rs:145,192: rows of one query need
// not be contiguous).  A repeated id means the fast contiguous path is not applicable.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) dup_kernel(const __grid_constant__ DupParams p) {
    if (p.ctr->cap_overflow) return;
    const unsigned long long rb = p.ctr->post_done;
    unsigned long long n = p.ctr->rec_count;
    if (n > p.rec_cap) n = p.rec_cap;
    for (unsigned long long i = rb + (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        blu_record& r = p.records[i];
        if (r.query_off + (unsigned long long)r.query_len > p.strings_len) continue;  // (a gather pass that overflowed: the host reruns)
        if (p.table) {
            unsigned long long h = 0xcbf29ce484222325ull;
            const uint8_t* q = p.strings + r.query_off;
            for (unsigned k = 0; k < r.query_len; k++) {
                h ^= q[k];
                h *= 0x100000001b3ull;
            }
            h = mix64(h ^ r.query_len);
            if (h == 0) h = 1;
            if (p.hashes) p.hashes[i] = h;
            unsigned slot = (unsigned)h & p.mask;
            for (unsigned t = 0; t <= p.mask; t++) {
                const unsigned long long old = atomicCAS(p.table + slot, 0ull, h);
                if (old == 0ull) break;
                if (old == h) {
                    p.ctr->dup_found = 1;
                    break;
                }
                slot = (slot + 1) & p.mask;
            }
        }
        if (p.ref_delta) {
            r.query_off = (unsigned long long)((long long)r.query_off + p.ref_delta);
            if (r.status == 1 && r.n_beans) {
                const blu_bean lb = p.beans[(unsigned long long)r.bean_base + r.n_beans - 1];
                const unsigned nacc = lb.acc_begin + lb.n_acc;
                for (unsigned a = 0; a < nacc; a++) {
                    blu_acc& ac = p.accs[(unsigned long long)r.acc_base + a];
                    ac.ref = (unsigned long long)((long long)ac.ref + p.ref_delta * 65536);
                }
            }
        }
    }
}

// Cross-device duplicate check of a multi-GPU run: the id hashes of all shards, inserted into one table.
__global__ void __launch_bounds__(256) dup_merge_kernel(const unsigned long long* hashes, unsigned long long n, unsigned long long* table, uint32_t mask,
                                                        unsigned int* dup_found) {
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long h = hashes[i];
        unsigned slot = (unsigned)h & mask;
        for (unsigned t = 0; t <= mask; t++) {
            const unsigned long long old = atomicCAS(table + slot, 0ull, h);
            if (old == 0ull) break;
            if (old == h) {
                *dup_found = 1;
                break;
            }
            slot = (slot + 1) & mask;
        }
    }
}

// Tile kernel output -> the other configurations of a pass (see FanoutParams).  Threads 0..n_dst-1 of block 0 copy the
// cursors; the whole grid copies the record headers, 16 bytes per thread and step.
__global__ void __launch_bounds__(256) fanout_kernel(const __grid_constant__ FanoutParams p) {
    const Counters* s = p.src;
    const unsigned long long rb = s->post_done;
    unsigned long long re = s->rec_count;
    if (re > p.rec_cap) re = p.rec_cap;
    if (!s->cap_overflow && re > rb) {  // (after an overflow every configuration runs again: nothing to copy)
        constexpr unsigned long long kPer = sizeof(blu_record) / sizeof(uint4);
        const unsigned long long n = (re - rb) * kPer;
        const uint4* src = reinterpret_cast<const uint4*>(p.src_records + rb);
        const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
        for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n * (unsigned long long)p.n_dst; i += stride) {
            const unsigned long long d = i / n, j = i - d * n;
            reinterpret_cast<uint4*>(p.dst_records[d] + rb)[j] = src[j];
        }
    }
    if (blockIdx.x == 0 && (int)threadIdx.x < p.n_dst) {
        Counters* d = p.dst[threadIdx.x];
        // the long-run kernel adds one record per finished deferred run in every configuration: the record counts agree
        if (d->post_done != rb) report(d, DE_INTERNAL, 0);
        d->rec_count = s->rec_count;
        d->slot_count = s->slot_count;
        d->n_defer = s->n_defer;
        if (s->tail_start < d->tail_start) d->tail_start = s->tail_start;
        if (s->err_code && !d->err_code) d->err_code = s->err_code, d->err_off = s->err_off;
        if (s->cap_overflow) d->cap_overflow = 1;
    }
}

// End of a range / chunk (one thread): see AdvanceParams.
__global__ void advance_kernel(const AdvanceParams p) {
    Counters* c = p.ctr;
    unsigned long long n = c->rec_count;
    if (n > p.rec_cap) n = p.rec_cap;
    c->post_done = n;
    c->next_begin = c->tail_start != ~0ull ? c->tail_start : p.range_end;
    if (p.snapshot) {
        *p.snapshot = *c;
        __threadfence_system();
    }
    c->n_defer = 0;
    c->work_ticket = 0;
    c->tail_start = ~0ull;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------------------------
cudaError_t kernels_set_attributes() {
    cudaError_t e = cudaFuncSetAttribute(tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(StreamSmem));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(longrun_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LongSmem));
}

int tile_kernel_grid(int device) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    return kTileCtasPerSm * sms;  // one streaming CTA per resident slot
}

cudaError_t launch_tile_kernel(const RunParams& p, int grid, cudaStream_t s) {
    tile_kernel<<<grid, kTileThreads, sizeof(StreamSmem), s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_longrun_kernel(const RunParams& p, int grid, cudaStream_t s) {
    longrun_kernel<<<grid, kLongThreads, sizeof(LongSmem), s>>>(p);
    return cudaGetLastError();
}

// The post-pass kernels take their record range from the device counters (no host round trip between the tile kernel
// and them): fixed grids, grid-stride loops.
cudaError_t launch_consensus_kernel(const PostParams& p, int sms, cudaStream_t s) {
    consensus_kernel<<<sms * 16, kConsThreads, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_gather_kernel(const PostParams& p, int sms, cudaStream_t s) {
    gather_kernel<<<sms * 8, 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_dup_kernel(const DupParams& p, int sms, cudaStream_t s) {
    dup_kernel<<<sms * 8, 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_fanout_kernel(const FanoutParams& p, int sms, cudaStream_t s) {
    fanout_kernel<<<sms * 4, 256, 0, s>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_dup_merge_kernel(const unsigned long long* hashes, unsigned long long n, unsigned long long* table, uint32_t mask,
                                    unsigned int* dup_found, int sms, cudaStream_t s) {
    if (!n) return cudaSuccess;
    dup_merge_kernel<<<sms * 8, 256, 0, s>>>(hashes, n, table, mask, dup_found);
    return cudaGetLastError();
}

cudaError_t launch_advance_kernel(const AdvanceParams& p, cudaStream_t s) {
    advance_kernel<<<1, 1, 0, s>>>(p);
    return cudaGetLastError();
}

}  // namespace blu
