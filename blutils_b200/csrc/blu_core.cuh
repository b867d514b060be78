// blu_core.cuh -- per-row parsing and per-query consensus logic shared by the CUDA kernels.
//
// Everything here is `__host__ __device__` so that tests/csrc/sim_harness.cpp can compile the *same* code
// with g++ and check it against the oracle without a GPU.  The product library only ever calls these from
// device code (blu_kernels.cu); there is no CPU execution path in libblu_consensus.so.
//
// Reference semantics restated (paths relative to /root/reference):
//   row fields / truncation ......... core/src/use_cases/build_consensus_identities/mod.rs:147-209,226-244
//   top bit-score group ............. find_single_query_consensus.rs:28-64
//   single match .................... find_single_query_consensus.rs:74-150
//   multi match (sort, level walk) .. find_multi_taxa_consensus.rs:39-214
//   rank selection / filtering ...... build_blast_consensus_identity.rs:9-105, linnaean_ranks.rs:174-212
//   bean folding .................... consensus_result.rs:65-88
#pragma once
#include <string.h>
#include <stdint.h>

#include "../../include/blu_consensus.h"

#if defined(__CUDACC__)
#define BLU_HD __host__ __device__ __forceinline__
#define BLU_HD_NOINLINE __host__ __device__ __noinline__
#else
#define BLU_HD inline
#define BLU_HD_NOINLINE inline
#endif

namespace blu {

// ---- device-side error codes (first error wins; host maps them to BLU_ERR_*) ------------------------------
enum DevErr : uint32_t {
    DE_NONE = 0,
    DE_BAD_FIELD_COUNT = 1,   // row does not have 13 fields            -> DATA
    DE_BAD_NUMBER = 2,        // numeric grammar violated               -> DATA
    DE_EMPTY_STRING = 3,      // empty qseqid / saccver                 -> DATA
    DE_QUOTE_OR_CR = 4,       // '"' or '\r' byte                       -> DATA
    DE_UNMAPPED_TAXID = 5,    // top-group row whose taxid has no lineage -> DATA (fsqc.rs:59)
    DE_BAD_LINEAGE = 6,       // top-group lineage failed parse_taxonomy  -> DATA
    DE_EMPTY_ADJUSTED = 7,    // single match, no rank passes the cutoff  -> DATA (fsqc.rs:113-119)
    DE_ROOT_DISAGREE = 8,     // level 0 disagreement (index-1 underflow) -> DATA (fmtc.rs:181)
    DE_BITS_RANGE = 9,        // bit score outside i64                  -> DATA
    DE_NUM_UNSUPPORTED = 32,  // number outside the exact fast path     -> UNSUPPORTED
    DE_TOPGROUP_TOO_BIG = 33, // top group larger than the block path handles -> UNSUPPORTED
    DE_CARRY_TOO_BIG = 34,    // a single query larger than the carry buffer  -> UNSUPPORTED
    DE_INTERNAL = 64
};

// ---- lineage tables in HBM (built by blu_taxonomy.cpp) ------------------------------------------------------
struct HashSlot {
    int64_t key;
    uint32_t val;   // lineage index
    uint32_t used;  // 0 = empty
};

struct LinTables {
    const uint32_t* lin_off;     // [n_lin+1] CSR offsets into the per-position arrays
    const uint32_t* lvl_key;     // id of rank.to_string()+identifier        (fmtc.rs:153-157)
    const uint32_t* bean_key;    // id of "{rank}__{identifier}"             (consensus_result.rs:70-73)
    const uint32_t* ident_rank;  // bytewise order rank of the identifier    (bbci.rs:50-60)
    const double* cut;           // interpolated cutoff                      (linnaean_ranks.rs:220-383)
    const uint16_t* rank_cls;    // equality class of the position's LinnaeanRank
    const uint16_t* allowed_cls; // equality class of the rank get_rank_adjusted_by_identity would return here
    const uint8_t* lin_ok;       // [n_lin] 1 = lineage parsed; 0 = parse_taxonomy would fail
    const HashSlot* slots;
    uint32_t hash_mask;
    uint32_t n_lin;
};

BLU_HD uint64_t mix64(uint64_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}

// taxid -> lineage index (left join on subject_taxid == taxid, mod.rs:72-76).  0xFFFFFFFF = no match.
BLU_HD uint32_t probe_taxid(const LinTables& T, int64_t taxid) {
    uint32_t h = (uint32_t)mix64((uint64_t)taxid) & T.hash_mask;
    for (uint32_t i = 0; i <= T.hash_mask; i++) {
        HashSlot s = T.slots[h];
        if (!s.used) return 0xFFFFFFFFu;
        if (s.key == taxid) return s.val;
        h = (h + 1) & T.hash_mask;
    }
    return 0xFFFFFFFFu;
}

// ---- numbers --------------------------------------------------------------------------------------------------
// int := -?[0-9]{1,18}
BLU_HD bool parse_i64(const uint8_t* p, int len, int64_t& v) {
    int i = 0;
    bool neg = false;
    if (len > 0 && p[0] == '-') {
        neg = true;
        i = 1;
    }
    int nd = len - i;
    if (nd < 1 || nd > 18) return false;
    int64_t x = 0;
    for (; i < len; i++) {
        uint32_t d = (uint32_t)p[i] - '0';
        if (d > 9) return false;
        x = x * 10 + d;
    }
    v = neg ? -x : x;
    return true;
}

// float := -?([0-9]+(\.[0-9]*)?|\.[0-9]+)([eE][+-]?[0-9]+)?
// Returns DE_NONE, DE_BAD_NUMBER (grammar) or DE_NUM_UNSUPPORTED (valid, but not exactly computable here:
// more than 19 significant digits, mantissa >= 2^53 or |decimal exponent| > 22).
// Exact path (Clinger): m and 10^|e| are both exact doubles, so one IEEE multiply/divide is correctly rounded.
#if defined(__CUDA_ARCH__)
__device__ __constant__ double kPow10[23] = {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11,
                                             1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};
#else
static const double kPow10[23] = {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11,
                                  1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};
#endif

BLU_HD uint32_t parse_f64(const uint8_t* p, int len, double& v) {
    int i = 0;
    bool neg = false;
    if (i < len && p[i] == '-') {
        neg = true;
        i++;
    }
    uint64_t mant = 0;
    int sig = 0, nint = 0, nfrac = 0;
    bool unsupported = false;
    while (i < len) {
        uint32_t d = (uint32_t)p[i] - '0';
        if (d > 9) break;
        if (sig > 0 || d != 0) {
            if (sig < 19) mant = mant * 10 + d;
            sig++;
        }
        nint++;
        i++;
    }
    if (i < len && p[i] == '.') {
        i++;
        while (i < len) {
            uint32_t d = (uint32_t)p[i] - '0';
            if (d > 9) break;
            if (sig > 0 || d != 0) {
                if (sig < 19) mant = mant * 10 + d;
                sig++;
            }
            nfrac++;
            i++;
        }
        if (nint == 0 && nfrac == 0) return DE_BAD_NUMBER;
    } else if (nint == 0)
        return DE_BAD_NUMBER;
    int ex = 0;
    if (i < len && (p[i] == 'e' || p[i] == 'E')) {
        i++;
        bool eneg = false;
        if (i < len && (p[i] == '+' || p[i] == '-')) {
            eneg = p[i] == '-';
            i++;
        }
        int nd = 0;
        while (i < len) {
            uint32_t d = (uint32_t)p[i] - '0';
            if (d > 9) break;
            if (ex < 100000) ex = ex * 10 + (int)d;
            nd++;
            i++;
        }
        if (nd == 0) return DE_BAD_NUMBER;
        if (eneg) ex = -ex;
    }
    if (i != len) return DE_BAD_NUMBER;
    if (sig > 19) unsupported = true;
    int e10 = ex - nfrac;
    double r;
    if (mant == 0 && !unsupported) {
        r = 0.0;
    } else {
        if (unsupported || mant >= (1ULL << 53) || e10 > 22 || e10 < -22) return DE_NUM_UNSUPPORTED;
        r = (double)mant;
        if (e10 >= 0)
            r = r * kPow10[e10];
        else
            r = r / kPow10[-e10];
    }
    v = neg ? -r : r;
    return DE_NONE;
}

// Grammar-only DFA for the numeric columns nobody reads (SURVEY 8 a2: 7 of 13 columns are parsed and dropped
// by the reference, but a malformed one still aborts it).  class: 0 digit, 1 '.', 2 e/E, 3 '+', 4 '-', 5 other.
BLU_HD int num_class(uint32_t c) {
    if (c - '0' <= 9u) return 0;
    if (c == '.') return 1;
    if ((c | 0x20) == 'e') return 2;
    if (c == '+') return 3;
    if (c == '-') return 4;
    return 5;
}
// float DFA states: 0 start, 1 sign, 2 int digits*, 3 "d." *, 4 frac digits*, 5 "." (needs digit), 6 e, 7 e sign,
// 8 exp digits*, 9 error.  (* accepting)
BLU_HD int float_dfa_next(int s, int cls) {
    switch (s) {
        case 0: return cls == 0 ? 2 : cls == 4 ? 1 : cls == 1 ? 5 : 9;
        case 1: return cls == 0 ? 2 : cls == 1 ? 5 : 9;
        case 2: return cls == 0 ? 2 : cls == 1 ? 3 : cls == 2 ? 6 : 9;
        case 3: return cls == 0 ? 4 : cls == 2 ? 6 : 9;
        case 4: return cls == 0 ? 4 : cls == 2 ? 6 : 9;
        case 5: return cls == 0 ? 4 : 9;
        case 6: return cls == 0 ? 8 : (cls == 3 || cls == 4) ? 7 : 9;
        case 7: return cls == 0 ? 8 : 9;
        case 8: return cls == 0 ? 8 : 9;
        default: return 9;
    }
}
BLU_HD bool float_dfa_accept(int s) { return s == 2 || s == 3 || s == 4 || s == 8; }

BLU_HD bool check_float(const uint8_t* p, int len) {
    int s = 0;
    for (int i = 0; i < len; i++) s = float_dfa_next(s, num_class(p[i]));
    return float_dfa_accept(s);
}
BLU_HD bool check_int(const uint8_t* p, int len) {
    int i = (len > 0 && p[0] == '-') ? 1 : 0;
    int nd = len - i;
    if (nd < 1 || nd > 18) return false;
    for (; i < len; i++)
        if ((uint32_t)p[i] - '0' > 9u) return false;
    return true;
}

// ---- one row, all 13 fields ----------------------------------------------------------------------------------
struct LightRow {
    int64_t bits;     // trunc(bitscore)
    uint16_t q_len;   // length of qseqid
    uint32_t err;     // DevErr
};

// Validates the whole row (field count, grammar of the 11 numeric columns, non-empty strings, no '"'/'\r')
// and extracts what every row needs: the truncated bit score and the qseqid length.
// Columns: 0 qseqid 1 saccver 2 staxid 3 pident 4 length 5 mismatch 6 gapopen 7 qstart 8 qend 9 sstart
// 10 send 11 evalue 12 bitscore (core/src/domain/dtos/blast_builder.rs:87).
BLU_HD LightRow light_parse_row(const uint8_t* p, int len) {
    LightRow r;
    r.bits = 0;
    r.q_len = 0;
    r.err = DE_NONE;
    int f = 0, fs = 0;
    int st = 0;        // DFA state of the current float field
    bool bad = false;  // current int field has a non-digit
    uint32_t err = DE_NONE;
    int last_start = 0;
    for (int i = 0; i <= len; i++) {
        uint32_t c = i < len ? p[i] : '\t';
        if (c == '\t') {
            int flen = i - fs;
            if (f <= 1) {
                if (flen == 0 && !err) err = DE_EMPTY_STRING;
                if (f == 0) r.q_len = (uint16_t)(flen > 65535 ? 65535 : flen);
            } else if (f == 3 || f == 11 || f == 12) {
                if (!float_dfa_accept(st) && !err) err = DE_BAD_NUMBER;
                if (f == 12) last_start = fs;
            } else if (f < 13) {
                int nd = flen - ((flen > 0 && p[fs] == '-') ? 1 : 0);
                if ((bad || nd < 1 || nd > 18) && !err) err = DE_BAD_NUMBER;
            }
            f++;
            fs = i + 1;
            st = 0;
            bad = false;
            continue;
        }
        if ((c == '"' || c == '\r') && !err) err = DE_QUOTE_OR_CR;
        if (f == 3 || f == 11 || f == 12) {
            st = float_dfa_next(st, num_class(c));
        } else if (f >= 2) {
            if (c - '0' > 9u && !(c == '-' && i == fs)) bad = true;
        }
    }
    if (f != 13 && !err) err = DE_BAD_FIELD_COUNT;
    if (!err) {
        double d;
        uint32_t e = parse_f64(p + last_start, len - last_start, d);
        if (e)
            err = e;
        else if (!(d > -9223372036854775808.0 && d < 9223372036854775808.0))
            err = DE_BITS_RANGE;
        else
            r.bits = (int64_t)d;  // truncation toward zero
    }
    r.err = err;
    return r;
}

// ---- one row, through the byte-class bitmasks -----------------------------------------------------------------
// The row scan classifies every byte of the window once (tab / digit bitmasks, bit i = byte i of the window);
// a row is then validated with bit operations in a 13-iteration loop that every lane walks in lockstep (field k of
// all 32 rows at the same time), instead of a data-dependent per-byte state machine.
// `tabw` / `digw` must be readable one word past the row.
BLU_HD int blu_ctz64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __ffsll((long long)x) - 1;
#else
    return __builtin_ctzll(x);
#endif
}

// first tab at position >= cur and < e, or e
BLU_HD int next_tab(const uint64_t* tabw, int cur, int e) {
    int w = cur >> 6;
    uint64_t bits = tabw[w] >> (cur & 63);
    if (bits) {
        int p = cur + blu_ctz64(bits);
        return p < e ? p : e;
    }
    for (w++; (w << 6) < e; w++) {
        bits = tabw[w];
        if (bits) {
            int p = (w << 6) + blu_ctz64(bits);
            return p < e ? p : e;
        }
    }
    return e;
}

// bytes [a, a+len) are all ASCII digits (1 <= len <= 32)
BLU_HD bool all_digits(const uint64_t* digw, int a, int len) {
    const int sh = a & 63;
    uint64_t x = digw[a >> 6] >> sh;
    if (sh > 32) x |= digw[(a >> 6) + 1] << (64 - sh);
    const uint32_t m = len >= 32 ? 0xFFFFFFFFu : ((1u << len) - 1u);
    return ((uint32_t)x & m) == m;
}

BLU_HD LightRow parse_row_masked(const uint8_t* win, const uint64_t* tabw, const uint64_t* digw, int s, int e) {
    LightRow r;
    r.bits = 0;
    r.q_len = 0;
    uint32_t err = DE_NONE;
    int cur = s;
    for (int k = 0; k < 13; k++) {
        const int t = k < 12 ? next_tab(tabw, cur, e) : e;
        if (k < 12 && t >= e) {  // ran out of tabs
            if (!err) err = DE_BAD_FIELD_COUNT;
            break;
        }
        const int len = t - cur;
        if (k <= 1) {
            if (len == 0 && !err) err = DE_EMPTY_STRING;
            if (k == 0) r.q_len = (uint16_t)(len > 65535 ? 65535 : len);
        } else if (k == 3 || k == 11) {
            // pident / evalue: grammar only here (pident's value is parsed again for the top rows)
            if (!check_float(win + cur, len) && !err) err = DE_BAD_NUMBER;
        } else if (k == 12) {
            if (next_tab(tabw, cur, e) < e) {  // a 14th field
                if (!err) err = DE_BAD_FIELD_COUNT;
            } else {
                double d;
                uint32_t pe = parse_f64(win + cur, len, d);
                if (pe) {
                    if (!err) err = pe;
                } else if (!(d > -9223372036854775808.0 && d < 9223372036854775808.0)) {
                    if (!err) err = DE_BITS_RANGE;
                } else
                    r.bits = (int64_t)d;
            }
        } else {
            // integer column: the common case is 1..18 digits, checked on the digit mask
            const bool fast = len >= 1 && len <= 18 && all_digits(digw, cur, len);
            if (!fast && !check_int(win + cur, len) && !err) err = DE_BAD_NUMBER;
        }
        cur = t + 1;
    }
    r.err = err;
    return r;
}

// ---- fast path: the whole row in registers -----------------------------------------------------------------------
// Rows of up to 96 bytes (every BLAST row in practice) are validated from three 32-bit words of the tab mask and
// three of the digit mask, with popcount / find-first-set / count-leading-zeros instead of per-byte loops.  The fast
// path only ACCEPTS shapes it fully understands (digits-only integers, `digits[.digits]` floats without exponent in
// pident / bitscore); anything else -- including every malformed row -- returns false and is re-examined by
// parse_row_masked(), which implements the complete grammar.  So the fast path can never change a result or an
// error decision, only skip work.
BLU_HD uint32_t blu_funnel_r(uint32_t lo, uint32_t hi, uint32_t sh) {  // (hi:lo) >> sh, 0 <= sh < 32
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}
BLU_HD int blu_ffs32(uint32_t x) {  // index of the lowest set bit; x != 0
#if defined(__CUDA_ARCH__)
    return __ffs((int)x) - 1;
#else
    return __builtin_ctz(x);
#endif
}
BLU_HD int blu_clz32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __clz((int)x);
#else
    return x ? __builtin_clz(x) : 32;
#endif
}
BLU_HD int blu_popc32(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// 32 mask bits starting at (window) bit position `pos`
BLU_HD uint32_t bits_at(const uint32_t* w, int pos) { return blu_funnel_r(w[pos >> 5], w[(pos >> 5) + 1], (uint32_t)pos & 31u); }

// Non-negative float of the shapes D+[.D*][e[+-]D+] / .D+..., decided from the positions of its non-digit bytes
// (`o` = non-digit mask of the field, bit i = byte i; o != 0).  false = "not one of these shapes" (caller falls back
// to the full DFA), never a wrong accept.
BLU_HD bool float_shape_ok(const uint8_t* f, int len, uint32_t o) {
    const int k = blu_popc32(o);
    if (k > 3) return false;
    const int i1 = blu_ffs32(o);
    const uint8_t c1 = f[i1];
    if (k == 1) {
        if (c1 == '.') return len >= 2;
        return (c1 | 0x20) == 'e' && i1 >= 1 && i1 <= len - 2;
    }
    const uint32_t o2 = o & (o - 1);
    const int i2 = blu_ffs32(o2);
    const uint8_t c2 = f[i2];
    if (k == 2) {
        if (c1 == '.') return (c2 | 0x20) == 'e' && i2 >= 2 && i2 <= len - 2;
        return (c1 | 0x20) == 'e' && (c2 == '-' || c2 == '+') && i2 == i1 + 1 && i1 >= 1 && i2 <= len - 2;
    }
    const int i3 = blu_ffs32(o2 & (o2 - 1));
    const uint8_t c3 = f[i3];
    return c1 == '.' && (c2 | 0x20) == 'e' && (c3 == '-' || c3 == '+') && i3 == i2 + 1 && i2 >= 2 && i3 <= len - 2;
}

// tabw32 / digw32: the byte-class masks viewed as 32-bit words (readable 4 words past the row start).
// Returns true and fills bits / q_len when the row is valid AND of the common shape.
BLU_HD bool parse_row_fast(const uint8_t* win, const uint32_t* tabw32, const uint32_t* digw32, int s, int e, int64_t& bits, int& q_len) {
    const int len = e - s;
    if (len > 96 || len < 25) return false;
    const int wi = s >> 5;
    const uint32_t sh = (uint32_t)s & 31u;
    uint32_t t0 = blu_funnel_r(tabw32[wi], tabw32[wi + 1], sh), t1 = blu_funnel_r(tabw32[wi + 1], tabw32[wi + 2], sh),
             t2 = blu_funnel_r(tabw32[wi + 2], tabw32[wi + 3], sh);
    // clear the bits at/after the end of the row
    if (len <= 32) {
        t0 &= len == 32 ? 0xFFFFFFFFu : ((1u << len) - 1u);
        t1 = 0;
        t2 = 0;
    } else if (len <= 64) {
        t1 &= len == 64 ? 0xFFFFFFFFu : ((1u << (len - 32)) - 1u);
        t2 = 0;
    } else {
        t2 &= len == 96 ? 0xFFFFFFFFu : ((1u << (len - 64)) - 1u);
    }
    if (blu_popc32(t0) + blu_popc32(t1) + blu_popc32(t2) != 12) return false;
    // first four tabs must lie in the first 64 bytes
    int p1, p2, p3, p4;
    {
        uint32_t a = t0, b = t1;
        int base = 0;
#define BLU_POP_TAB(dst)            \
    if (!a) {                       \
        a = b, b = 0, base += 32;   \
        if (!a) return false;       \
    }                               \
    dst = base + blu_ffs32(a);      \
    a &= a - 1;
        BLU_POP_TAB(p1)
        BLU_POP_TAB(p2)
        BLU_POP_TAB(p3)
        BLU_POP_TAB(p4)
#undef BLU_POP_TAB
        if (base >= 64) return false;
    }
    // last two tabs
    int p12, p11;
    {
        uint32_t a = t2, b = t1, c = t0;
        int base = 64;
        if (!a) {
            a = b, b = c, c = 0, base = 32;
            if (!a) a = b, b = 0, base = 0;
        }
        p12 = base + 31 - blu_clz32(a);
        a &= ~(1u << (p12 - base));
        if (!a) {
            a = b, base -= 32;
            if (!a) a = c, base -= 32;  // (cannot run out: there are 12 tabs)
        }
        p11 = base + 31 - blu_clz32(a);
    }
    // field lengths (relative positions within the row)
    const int l_q = p1, l_acc = p2 - p1 - 1, l_tax = p3 - p2 - 1, l_pid = p4 - p3 - 1, l_ints = p11 - p4 - 1, l_ev = p12 - p11 - 1,
              l_bits = len - p12 - 1;
    if (l_q < 1 || l_acc < 1 || l_tax < 1 || l_tax > 18 || l_pid < 1 || l_pid > 32 || l_ints < 13 || l_ints > 30 || l_ev < 1 || l_ev > 32 ||
        l_bits < 1 || l_bits > 32)
        return false;
    // "other" = neither digit nor tab
    // taxid: digits only
    {
        const uint32_t d = bits_at(digw32, s + p2 + 1);
        const uint32_t m = (1u << l_tax) - 1u;
        if ((d & m) != m) return false;
    }
    // length .. send: seven non-empty digit-only fields separated by single tabs
    {
        const uint32_t d = bits_at(digw32, s + p4 + 1), t = bits_at(tabw32, s + p4 + 1);
        const uint32_t m = (1u << l_ints) - 1u;
        if (((d | t) & m) != m) return false;
        const uint32_t tt = t & m;
        if (blu_popc32(tt) != 6 || (tt & (tt << 1)) || (tt & 1u) || (tt >> (l_ints - 1))) return false;
    }
    // pident / evalue: digits with at most one '.', at least one digit
    {
        const uint32_t m = l_pid == 32 ? 0xFFFFFFFFu : ((1u << l_pid) - 1u);
        const uint32_t o = ~bits_at(digw32, s + p3 + 1) & m;
        if (o) {
            if (o & (o - 1)) return false;
            if (l_pid < 2 || win[s + p3 + 1 + blu_ffs32(o)] != '.') return false;
        }
    }
    {
        const uint32_t m = l_ev == 32 ? 0xFFFFFFFFu : ((1u << l_ev) - 1u);
        const uint32_t o = ~bits_at(digw32, s + p11 + 1) & m;
        if (o && !float_shape_ok(win + s + p11 + 1, l_ev, o) && !check_float(win + s + p11 + 1, l_ev)) return false;
    }
    // bit score: digits[.digits] with at most 15 digits in total -> trunc(value) is the integer part, exactly
    {
        const uint32_t m = l_bits == 32 ? 0xFFFFFFFFu : ((1u << l_bits) - 1u);
        const uint32_t o = ~bits_at(digw32, s + p12 + 1) & m;
        int n_int = l_bits;
        if (o) {
            if (o & (o - 1)) return false;
            n_int = blu_ffs32(o);
            if (l_bits < 2 || win[s + p12 + 1 + n_int] != '.') return false;
            if (l_bits - 1 > 15) return false;
        } else if (l_bits > 15)
            return false;
        const uint8_t* b = win + s + p12 + 1;
        if (n_int <= 9) {  // the usual case: 32-bit arithmetic
            uint32_t v = 0;
            for (int i = 0; i < n_int; i++) v = v * 10u + (uint32_t)(b[i] - '0');
            bits = (int64_t)v;
        } else {
            int64_t v = 0;
            for (int i = 0; i < n_int; i++) v = v * 10 + (int64_t)(b[i] - '0');
            bits = v;
        }
    }
    q_len = l_q;
    return true;
}

// ---- lean path: the numeric tail of the row in two 64-bit masks -----------------------------------------------------
// The streaming tile kernel's per-row parser.  The first two tabs (qseqid, saccver) are taken from the first 64 bytes
// of the row; the 11 numeric columns behind them ("tail", at most 64 bytes) are validated with a handful of 64-bit
// mask operations on the tab / digit masks re-aligned to the tail: tab count, no empty field, non-digit bytes only
// inside pident / evalue / bitscore and of the accepted shapes.  Like parse_row_fast() it only ACCEPTS rows it fully
// understands and returns false for everything else (the caller then runs parse_row_masked(), the complete grammar),
// so it can never change a result or an error decision.
BLU_HD int blu_popc64(uint64_t x) {
#if defined(__CUDA_ARCH__)
    return __popcll(x);
#else
    return __builtin_popcountll(x);
#endif
}
BLU_HD int blu_clz64(uint64_t x) {  // x != 0
#if defined(__CUDA_ARCH__)
    return __clzll((long long)x);
#else
    return __builtin_clzll(x);
#endif
}
// 64 mask bits starting at (window) bit position `pos` (reads words pos/32 .. pos/32+2)
BLU_HD uint64_t bits64_at(const uint32_t* w, int pos) {
    const int i = pos >> 5;
    const uint32_t sh = (uint32_t)pos & 31u;
    const uint32_t a = w[i], b = w[i + 1], c = w[i + 2];
    return (uint64_t)blu_funnel_r(a, b, sh) | ((uint64_t)blu_funnel_r(b, c, sh) << 32);
}

// n ASCII digits (0 <= n <= 8) starting at win[pos] -> value, without a per-digit loop: the eight bytes are shifted so
// that the number is right-aligned in a 64-bit little-endian word (leading bytes zero), then each half is folded with
// two multiply-adds (digit pairs, then pairs of pairs).  The caller has validated that the bytes are digits.
BLU_HD uint32_t swar4(uint32_t x) {  // bytes d0 d1 d2 d3 (d0 = lowest byte, most significant digit) -> d0 d1 d2 d3 as a number
    x &= 0x0F0F0F0Fu;
    x = x * 10u + (x >> 8);
    x &= 0x00FF00FFu;
    return (x & 0xFFFFu) * 100u + (x >> 16);
}
BLU_HD uint32_t load_u32_unaligned(const uint8_t* win, int pos);
BLU_HD uint32_t swar_digits(const uint8_t* win, int pos, int n) {
    if (n <= 0) return 0u;
    const uint64_t v = (((uint64_t)load_u32_unaligned(win, pos + 4) << 32) | (uint64_t)load_u32_unaligned(win, pos)) << (8 * (8 - n));
    return swar4((uint32_t)v) * 10000u + swar4((uint32_t)(v >> 32));
}

constexpr uint32_t kRowInfoValid = 0x80000000u;

BLU_HD bool parse_row_lean(const uint8_t* win, const uint32_t* tabw32, const uint32_t* digw32, int s, int e, int64_t& bits, int& q_len, uint32_t& info) {
    // Written without early exits: every check only clears `ok`, all indices are clamped so that every load stays inside
    // the window whatever the row looks like.  The independent parts (first two tabs, head-aligned tail words,
    // end-aligned word, the '.' bytes, the digit fold) can then overlap instead of waiting for one another's branches.
    bool ok = e >= 32;
    // ---- first two tabs (qseqid / saccver end inside the first 64 bytes) ---------------------------------------------
    int p1, p2;
    {
        const int wi = s >> 5;
        const uint32_t sh = (uint32_t)s & 31u;
        const uint32_t w0 = tabw32[wi], w1 = tabw32[wi + 1], w2 = tabw32[wi + 2];
        const uint32_t t0 = blu_funnel_r(w0, w1, sh), t1 = blu_funnel_r(w1, w2, sh);
        const uint32_t t0b = t0 & (t0 - 1u), t1b = t1 & (t1 - 1u);
        // first tab: in t0, else in t1; second: the next one after it
        const uint32_t f1 = t0 ? t0 : t1;
        const uint32_t f2 = t0 ? (t0b ? t0b : t1) : t1b;
        ok = ok && f1 != 0u && f2 != 0u;
        p1 = (t0 ? 0 : 32) + blu_ffs32(f1 | 0x80000000u);
        p2 = ((t0 && t0b) ? 0 : 32) + blu_ffs32(f2 | 0x80000000u);
    }
    const int a = s + p2 + 1;  // first byte of staxid
    const int m = e - a;       // bytes of the numeric tail
    ok = ok && p1 >= 1 && p2 - p1 >= 2 && m >= 21 && m <= 64;
    const int mc = m < 21 ? 21 : (m > 64 ? 64 : m);
    // ---- the tail through two head-aligned words (bytes a.., a+32..) and one end-aligned word (bytes e-32..e-1) ------
    const int ai = a >> 5;
    const uint32_t ash = (uint32_t)a & 31u;
    const uint32_t x0 = tabw32[ai], x1 = tabw32[ai + 1], x2 = tabw32[ai + 2];
    const uint32_t y0 = digw32[ai], y1 = digw32[ai + 1], y2 = digw32[ai + 2];
    const int eb = e >= 32 ? e - 32 : 0;
    const uint32_t te_raw = bits_at(tabw32, eb), de_raw = bits_at(digw32, eb);
    const uint32_t m0 = mc >= 32 ? 0xFFFFFFFFu : ((1u << mc) - 1u);
    const uint32_t m1 = mc >= 64 ? 0xFFFFFFFFu : (mc > 32 ? ((1u << (mc - 32)) - 1u) : 0u);
    const uint32_t ta0 = blu_funnel_r(x0, x1, ash) & m0, ta1 = blu_funnel_r(x1, x2, ash) & m1;
    const uint32_t oa0 = ~(blu_funnel_r(y0, y1, ash) | ta0) & m0, oa1 = ~(blu_funnel_r(y1, y2, ash) | ta1) & m1;  // neither digit nor tab
    ok = ok && blu_popc32(ta0) + blu_popc32(ta1) == 10;
    // no empty field: no two adjacent tabs, no tab at either end of the tail
    const uint32_t last = mc > 32 ? (ta1 >> (mc - 33)) : (ta0 >> (mc - 1));
    ok = ok && (((ta0 & (ta0 << 1)) | (ta1 & ((ta1 << 1) | (ta0 >> 31))) | (ta0 & 1u) | (last & 1u)) == 0u);
    // staxid / pident end inside the first 32 bytes of the tail
    const uint32_t ta0b = ta0 & (ta0 - 1u);
    ok = ok && ta0b != 0u;
    const int q3 = blu_ffs32(ta0 | 0x80000000u), q4 = blu_ffs32(ta0b | 0x80000000u);
    // evalue / bitscore start inside the last 32 bytes of the row
    const uint32_t me = mc >= 32 ? 0xFFFFFFFFu : (0xFFFFFFFFu << (32 - mc));  // bytes of the end-aligned word that belong to the tail
    const uint32_t te = te_raw & me;
    const uint32_t oe_all = ~(de_raw | te) & me;
    const int q12e = 31 - blu_clz32(te | 1u);
    const uint32_t te2 = te & ~(1u << q12e);
    ok = ok && te != 0u && te2 != 0u && q12e < 31;
    const int q11e = 31 - blu_clz32(te2 | 1u);
    const int q11 = mc - 32 + q11e;  // tab in front of evalue, tail coordinates
    // integer columns <= 18 digits: staxid directly, length..send (7 fields, 6 tabs) through their total span
    ok = ok && q3 <= 18 && q11 - q4 - 1 <= 30;
    // non-digit bytes may only sit in pident and in evalue / bitscore: compare the counts
    const uint32_t op = oa0 & ((1u << (q4 & 31)) - 1u) & ~((2u << (q3 & 31)) - 1u);
    const uint32_t otail = oe_all & ~((2u << (q11e & 31)) - 1u);
    ok = ok && blu_popc32(oa0) + blu_popc32(oa1) == blu_popc32(op) + blu_popc32(otail);
    // pident: digits with at most one '.', at least one digit
    {
        const uint8_t c = win[a + blu_ffs32(op | 0x80000000u)];
        ok = ok && (op == 0u || ((op & (op - 1u)) == 0u && q4 - q3 - 1 >= 2 && c == '.'));
    }
    // bit score: digits[.digits], <= 15 digits in total (trunc(value) is then exactly the integer part), <= 8 of them
    // in front of the point
    const int l_bits = 31 - q12e;
    const uint32_t ob = q12e < 31 ? (oe_all >> ((q12e + 1) & 31)) : 0u;
    const int n_int = ob ? blu_ffs32(ob) : l_bits;
    {
        const uint8_t c = win[eb + q12e + 1 + (n_int & 31)];
        ok = ok && (ob ? ((ob & (ob - 1u)) == 0u && l_bits >= 2 && l_bits <= 16 && c == '.') : l_bits <= 15) && n_int <= 8;
    }
    const uint32_t v = swar_digits(win, eb + q12e + 1, n_int > 8 ? 8 : n_int);
    // evalue: one of the common float shapes, else the DFA
    const int l_ev = q12e - q11e - 1;
    if (ok) {
        const uint32_t oe = (oe_all >> (q11e + 1)) & ((1u << l_ev) - 1u);
        if (oe && !float_shape_ok(win + eb + q11e + 1, l_ev, oe) && !check_float(win + eb + q11e + 1, l_ev)) ok = false;
    }
    bits = (int64_t)v;
    q_len = p1;
    // where fields 1..4 sit (for the consensus kernel, should this be a top row): ends of qseqid / saccver relative to the
    // row, ends of staxid / pident / length relative to the byte behind saccver's tab
    // layout: p1:6 | p2:6 | q3:5 | q4:5 | width of `length`:4 | digits in front of pident's '.' (31: no '.'):5 | valid:1
    {
        const uint32_t ta0c = ta0b & (ta0b - 1u);
        const int q5 = ta0c ? blu_ffs32(ta0c) : 32 + blu_ffs32(ta1 | 0x80000000u);
        const int ll = q5 - q4 - 1;
        const int dot = op ? blu_ffs32(op) - (q3 + 1) : 31;
        info = (ok && ll >= 1 && ll <= 15 && dot >= 0 && dot <= 31)
                   ? (kRowInfoValid | (uint32_t)p1 | ((uint32_t)p2 << 6) | ((uint32_t)q3 << 12) | ((uint32_t)q4 << 17) | ((uint32_t)ll << 22) | ((uint32_t)dot << 26))
                   : 0u;
    }
    return ok;
}

// first fields (qseqid) of the rows starting at a and b are equal
BLU_HD uint32_t load_u32_unaligned(const uint8_t* win, int pos) {
#if defined(__CUDA_ARCH__)
    const uint32_t* w = reinterpret_cast<const uint32_t*>(win + (pos & ~3));
    return __funnelshift_r(w[0], w[1], (uint32_t)(pos & 3) * 8u);
#else
    return (uint32_t)win[pos] | ((uint32_t)win[pos + 1] << 8) | ((uint32_t)win[pos + 2] << 16) | ((uint32_t)win[pos + 3] << 24);
#endif
}

BLU_HD bool same_first_field(const uint8_t* win, const uint64_t* tabw, int a, int ea, int b, int eb) {
    const uint32_t* tabw32 = reinterpret_cast<const uint32_t*>(tabw);
    // length of the first field: first tab within the first 32 bytes (the common case), else the general search
    uint32_t ta = bits_at(tabw32, a), tb = bits_at(tabw32, b);
    int la = ta ? blu_ffs32(ta) : 32, lb = tb ? blu_ffs32(tb) : 32;
    if (la >= 32 || a + la > ea) la = next_tab(tabw, a, ea) - a;
    if (lb >= 32 || b + lb > eb) lb = next_tab(tabw, b, eb) - b;
    if (la != lb) return false;
    int i = 0;
    for (; i + 4 <= la; i += 4)  // (reads stay inside the rows: i + 4 <= la)
        if (load_u32_unaligned(win, a + i) != load_u32_unaligned(win, b + i)) return false;
    for (; i < la; i++)
        if (win[a + i] != win[b + i]) return false;
    return true;
}

// Same test for the streaming kernel, which already knows the length `la` of the first field of the row at `a`: the
// la + 1 bytes "id, tab" of the two rows must be equal.  (The id at `a` holds no tab, so equal bytes put b's first tab at
// la as well; the row at `b` lies in front of `a` in the same window, so b + la stays inside it whatever b's length.)
BLU_HD bool same_qid_lean(const uint8_t* win, const uint32_t* /*tabw32*/, int a, int la, int b) {
    const int n = la + 1;
    if (n < 4) {
        for (int i = 0; i < n; i++)
            if (win[a + i] != win[b + i]) return false;
        return true;
    }
    uint32_t diff = load_u32_unaligned(win, a + n - 4) ^ load_u32_unaligned(win, b + n - 4);  // last word (may overlap the one before)
    for (int i = 0; i + 4 < n; i += 4) diff |= load_u32_unaligned(win, a + i) ^ load_u32_unaligned(win, b + i);
    return diff == 0;
}

// ---- top-group rows ---------------------------------------------------------------------------------------------
struct TopRow {
    double pident;
    int64_t alnlen;
    uint64_t acc_off;   // absolute offset of saccver in the text buffer
    uint32_t lin;       // lineage index
    uint16_t acc_len;
    uint16_t lin_len;   // number of lineage positions
};

// Fields 1..4 of an already validated row: saccver bounds, staxid -> lineage, pident, length.
BLU_HD uint32_t heavy_parse_row(const uint8_t* p, int len, uint64_t row_abs_off, const LinTables& T, TopRow& out) {
    int tabs[5];
    int nt = 0;
    for (int i = 0; i < len && nt < 5; i++)
        if (p[i] == '\t') tabs[nt++] = i;
    if (nt < 5) return DE_BAD_FIELD_COUNT;
    out.acc_off = row_abs_off + (uint64_t)tabs[0] + 1;
    int alen = tabs[1] - tabs[0] - 1;
    if (alen > 65535) return DE_NUM_UNSUPPORTED;
    out.acc_len = (uint16_t)alen;
    int64_t taxid;
    if (!parse_i64(p + tabs[1] + 1, tabs[2] - tabs[1] - 1, taxid)) return DE_BAD_NUMBER;
    uint32_t e = parse_f64(p + tabs[2] + 1, tabs[3] - tabs[2] - 1, out.pident);
    if (e) return e;
    if (!parse_i64(p + tabs[3] + 1, tabs[4] - tabs[3] - 1, out.alnlen)) return DE_BAD_NUMBER;
    uint32_t lin = probe_taxid(T, taxid);
    if (lin == 0xFFFFFFFFu) return DE_UNMAPPED_TAXID;
    if (!T.lin_ok[lin]) return DE_BAD_LINEAGE;
    out.lin = lin;
    out.lin_len = (uint16_t)(T.lin_off[lin + 1] - T.lin_off[lin]);
    return DE_NONE;
}

// A top-group row as the tile kernel emits it: numbers parsed, lineage not joined yet (the consensus kernel probes
// the taxid table, where full occupancy hides the lookup latency).
struct TopRowRaw {
    double pident;     // (or, when dec_frac != 0, its decimal form: see toprow_pident)
    int64_t alnlen;
    uint64_t acc_off;  // absolute offset of saccver in the text buffer
    int64_t taxid;
    uint32_t acc_len;
    uint32_t dec_frac;  // 0: `pident` is the value; kTopRowUnparsed: nothing is parsed, acc_off / acc_len are the ROW's offset and
                        // length (the consensus kernel runs heavy_parse_row on it); 0x80000000 | nf: the 8 bytes of `pident` hold the decimal mantissa m
                        // (low word) of a `ddd.fff` literal with nf fraction digits, value = m / 10^nf -- the tile kernel
                        // leaves that one IEEE division to the consensus kernel
};

constexpr uint32_t kTopRowUnparsed = 0x40000000u;

// value of a raw top row's pident: the exact Clinger path (mantissa < 2^53, one correctly rounded division), the same
// arithmetic parse_f64_short() performs
BLU_HD double toprow_pident(const TopRowRaw& raw) {
    if (!(raw.dec_frac & 0x80000000u)) return raw.pident;
    uint64_t bits;
    memcpy(&bits, &raw.pident, 8);
    const uint32_t m = (uint32_t)bits;
    const int nf = (int)(raw.dec_frac & 0xFFu);
    return nf > 0 ? (double)m / kPow10[nf] : (double)m;
}

// digits-only unsigned integer of at most 9 digits (the common staxid / length): 32-bit arithmetic
BLU_HD bool parse_u32_short(const uint8_t* p, int len, int64_t& v) {
    if (len < 1 || len > 9) return false;
    uint32_t x = 0;
    for (int i = 0; i < len; i++) {
        const uint32_t d = (uint32_t)p[i] - '0';
        if (d > 9u) return false;
        x = x * 10u + d;
    }
    v = (int64_t)x;
    return true;
}

// `ddd[.ddd]` with at most 9 digits in total: exact Clinger path (mantissa < 2^53, one IEEE divide) without the
// generic parser's 64-bit bookkeeping.  false = some other shape (caller uses parse_f64).
BLU_HD bool parse_f64_short(const uint8_t* p, int len, double& v) {
    if (len < 1 || len > 10) return false;
    uint32_t m = 0;
    int nd = 0, frac = -1;
    for (int i = 0; i < len; i++) {
        const uint32_t c = p[i];
        const uint32_t d = c - '0';
        if (d <= 9u) {
            m = m * 10u + d;
            nd++;
            if (frac >= 0) frac++;
        } else if (c == '.' && frac < 0)
            frac = 0;
        else
            return false;
    }
    if (nd == 0 || nd > 9) return false;
    v = frac > 0 ? (double)m / kPow10[frac] : (double)m;
    return true;
}

BLU_HD uint32_t split_top_row(const uint8_t* win, const uint64_t* tabw, int s, int e, uint64_t lo, TopRowRaw& out) {
    const int t0 = next_tab(tabw, s, e);
    const int t1 = t0 < e ? next_tab(tabw, t0 + 1, e) : e;
    const int t2 = t1 < e ? next_tab(tabw, t1 + 1, e) : e;
    const int t3 = t2 < e ? next_tab(tabw, t2 + 1, e) : e;
    const int t4 = t3 < e ? next_tab(tabw, t3 + 1, e) : e;
    if (t4 >= e) return DE_BAD_FIELD_COUNT;
    out.acc_off = lo + (uint64_t)t0 + 1;
    const int alen = t1 - t0 - 1;
    if (alen > 65535) return DE_NUM_UNSUPPORTED;
    out.acc_len = (uint32_t)alen;
    out.dec_frac = 0;
    if (!parse_u32_short(win + t1 + 1, t2 - t1 - 1, out.taxid) && !parse_i64(win + t1 + 1, t2 - t1 - 1, out.taxid)) return DE_BAD_NUMBER;
    if (!parse_f64_short(win + t2 + 1, t3 - t2 - 1, out.pident)) {
        uint32_t er = parse_f64(win + t2 + 1, t3 - t2 - 1, out.pident);
        if (er) return er;
    }
    if (!parse_u32_short(win + t3 + 1, t4 - t3 - 1, out.alnlen) && !parse_i64(win + t3 + 1, t4 - t3 - 1, out.alnlen)) return DE_BAD_NUMBER;
    return DE_NONE;
}

// Fields 1..4 of a validated row whose field positions are known (packed by parse_row_lean) -- the tile kernel's top-row
// splitter: no tab search, no mask access, SWAR digit folds for staxid (<= 16 digits), length (<= 8) and pident's decimal mantissa
// (`ddd[.ddd]`, <= 9 digits; the division is left to toprow_pident() in the consensus kernel).  Returns false for any
// other shape (the caller then emits the row unparsed).  Same values as split_top_row() (checked row by row in
// tests/csrc/sim_harness.cpp).
BLU_HD bool top_row_from_info(const uint8_t* win, int s, uint32_t info, uint64_t lo, TopRowRaw& out) {
    const int p1 = (int)(info & 63u), p2 = (int)((info >> 6) & 63u), q3 = (int)((info >> 12) & 31u), q4 = (int)((info >> 17) & 31u),
              ll = (int)((info >> 22) & 15u), dot = (int)((info >> 26) & 31u);
    const int a = s + p2 + 1;
    const int lp = q4 - q3 - 1;
    // pident: `dot` digits, then (unless dot == 31: digits only) a '.', then the rest -- parse_row_lean checked the shape
    const int ni = dot == 31 ? lp : dot;
    const int nf = dot == 31 ? 0 : lp - dot - 1;
    if (!(info & kRowInfoValid) || q3 > 16 || ll > 8 || ni > 8 || nf > 8 || ni + nf < 1 || ni + nf > 9) return false;
    out.acc_off = lo + (uint64_t)(s + p1 + 1);
    out.acc_len = (uint32_t)(p2 - p1 - 1);
    out.taxid = q3 <= 8 ? (int64_t)swar_digits(win, a, q3)
                        : (int64_t)((uint64_t)swar_digits(win, a, q3 - 8) * 100000000ull + (uint64_t)swar_digits(win, a + q3 - 8, 8));
    out.alnlen = (int64_t)swar_digits(win, a + q4 + 1, ll);
    uint32_t p10 = 1u;
    for (int i = 0; i < nf; i++) p10 *= 10u;
    const uint64_t dec = (uint64_t)(swar_digits(win, a + q3 + 1, ni) * p10 + swar_digits(win, a + q3 + 2 + ni, nf));
    memcpy(&out.pident, &dec, 8);
    out.dec_frac = 0x80000000u | (uint32_t)nf;
    return true;
}

// the join: taxid -> lineage (mod.rs:72-76); a miss / unparsable lineage in a top group is what makes the reference panic
BLU_HD uint32_t join_top_row(const TopRowRaw& raw, const LinTables& T, TopRow& out) {
    out.pident = toprow_pident(raw);
    out.alnlen = raw.alnlen;
    out.acc_off = raw.acc_off;
    out.acc_len = (uint16_t)raw.acc_len;
    const uint32_t lin = probe_taxid(T, raw.taxid);
    if (lin == 0xFFFFFFFFu) return DE_UNMAPPED_TAXID;
    if (!T.lin_ok[lin]) return DE_BAD_LINEAGE;
    out.lin = lin;
    out.lin_len = (uint16_t)(T.lin_off[lin + 1] - T.lin_off[lin]);
    return DE_NONE;
}

// Same as heavy_parse_row, with the field boundaries taken from the tab mask.  `lo` = absolute offset of win[0].
BLU_HD uint32_t heavy_parse_row_masked(const uint8_t* win, const uint64_t* tabw, int s, int e, uint64_t lo, const LinTables& T, TopRow& out) {
    const int t0 = next_tab(tabw, s, e);
    const int t1 = t0 < e ? next_tab(tabw, t0 + 1, e) : e;
    const int t2 = t1 < e ? next_tab(tabw, t1 + 1, e) : e;
    const int t3 = t2 < e ? next_tab(tabw, t2 + 1, e) : e;
    const int t4 = t3 < e ? next_tab(tabw, t3 + 1, e) : e;
    if (t4 >= e) return DE_BAD_FIELD_COUNT;
    out.acc_off = lo + (uint64_t)t0 + 1;
    const int alen = t1 - t0 - 1;
    if (alen > 65535) return DE_NUM_UNSUPPORTED;
    out.acc_len = (uint16_t)alen;
    int64_t taxid;
    if (!parse_i64(win + t1 + 1, t2 - t1 - 1, taxid)) return DE_BAD_NUMBER;
    uint32_t er = parse_f64(win + t2 + 1, t3 - t2 - 1, out.pident);
    if (er) return er;
    if (!parse_i64(win + t3 + 1, t4 - t3 - 1, out.alnlen)) return DE_BAD_NUMBER;
    uint32_t lin = probe_taxid(T, taxid);
    if (lin == 0xFFFFFFFFu) return DE_UNMAPPED_TAXID;
    if (!T.lin_ok[lin]) return DE_BAD_LINEAGE;
    out.lin = lin;
    out.lin_len = (uint16_t)(T.lin_off[lin + 1] - T.lin_off[lin]);
    return DE_NONE;
}

// ---- record stages ----------------------------------------------------------------------------------------------
// A record starts as record_header() (no consensus, no beans).  The tile kernel turns it into a pending record for the
// consensus kernel; write_outcome() then sets what the consensus decided.  The host only ever sees status 0 and 1.
constexpr uint8_t kStatusNoConsensus = 0;  // NoConsensusFound: a hit-less header, or a query whose consensus failed
constexpr uint8_t kStatusFound = 1;        // ConsensusFound
constexpr uint8_t kStatusPending = 2;      // waiting for the consensus kernel (device only)

BLU_HD blu_record record_header(uint64_t query_off, uint32_t query_len, uint32_t n_rows, int64_t bit_score) {
    blu_record r;
    r.query_off = query_off;
    r.query_len = query_len;
    r.n_rows = n_rows;
    r.keep_mask = 0;
    r.perc_identity = 0.0;
    r.bit_score = bit_score;
    r.ref_lineage = 0;
    r.bean_base = 0;
    r.n_beans = 0;
    r.acc_base = 0;
    r.status = kStatusNoConsensus;
    r.single_match = 0;
    r.mutated = 0;
    r.reached_pos = 0;
    r.allowed_pos = -1;
    r.bean_level = 0;
    r.pad[0] = r.pad[1] = 0;
    return r;
}

// Until the consensus kernel has run, a pending record's bean_base / n_beans hold the query's first top-row slot and the
// size of its top group: only these three functions know that.
BLU_HD blu_record pending_record(blu_record r, uint32_t slot, uint32_t n_top) {
    r.status = kStatusPending;
    r.bean_base = slot;
    r.n_beans = n_top;
    return r;
}
BLU_HD uint32_t pending_slot(const blu_record& r) { return r.bean_base; }
BLU_HD uint32_t pending_rows(const blu_record& r) { return r.n_beans; }

// What the consensus decides for a query: every record field but the header and where its beans / accession references
// went.  Outcome{} is a failure (ok = false).
struct Outcome {
    uint64_t keep_mask;   // the cutoff part (cutoff_outcome / apply_cutoffs) ...
    int reached_pos, allowed_pos;
    bool mutated;
    double perc_identity;  // ... and what the top group decided
    uint32_t ref_lineage, n_beans;
    int bean_level;
    bool single_match, ok;
};

// The cutoff part (build_blast_consensus_identity.rs:22-37,66-95): `keep` = the reference-lineage positions that go into the
// output taxonomy, `allowed` = maxAllowedRank's position or -1, `idx` = the bean's position, the reached one when nothing is
// kept (adjusted_taxonomy.last().unwrap_or(_bean)).
BLU_HD Outcome cutoff_outcome(uint64_t keep, int allowed, int idx, bool mutated) {
    Outcome o = {};
    o.keep_mask = keep;
    o.reached_pos = keep ? 63 - blu_clz64(keep) : idx;
    o.allowed_pos = allowed;
    o.mutated = mutated;
    return o;
}

// A consensus found: the cutoff part `o` plus the reference row's identity and lineage, the beans and their level.
BLU_HD Outcome found_outcome(Outcome o, double perc_identity, uint32_t ref_lineage, uint32_t n_beans, int bean_level, bool single_match) {
    o.perc_identity = perc_identity;
    o.ref_lineage = ref_lineage;
    o.n_beans = n_beans;
    o.bean_level = bean_level;
    o.single_match = single_match;
    o.ok = true;
    return o;
}

// A single match (find_single_query_consensus.rs:74-150): `keep` = every position whose cutoff the row passes (not empty);
// one bean at the last of them, no maxAllowedRank.
BLU_HD Outcome single_outcome(uint64_t keep, double perc_identity, uint32_t ref_lineage) {
    const Outcome cut = cutoff_outcome(keep, -1, 0, false);
    return found_outcome(cut, perc_identity, ref_lineage, 1, cut.reached_pos, true);
}

// The record fields an outcome decides.  A failed query keeps its id (the duplicate-id check must see it) and owns no beans
// or accession references.
BLU_HD void write_outcome(blu_record* rec, const Outcome& o) {
    if (o.ok) {
        rec->keep_mask = o.keep_mask;
        rec->perc_identity = o.perc_identity;
        rec->ref_lineage = o.ref_lineage;
        rec->n_beans = o.n_beans;
        rec->single_match = o.single_match ? 1 : 0;
        rec->mutated = o.mutated ? 1 : 0;
        rec->reached_pos = (int8_t)o.reached_pos;
        rec->allowed_pos = (int8_t)o.allowed_pos;
        rec->bean_level = (int8_t)o.bean_level;
        rec->status = kStatusFound;
    } else {
        rec->bean_base = 0, rec->n_beans = 0, rec->acc_base = 0;
        rec->status = kStatusNoConsensus;
    }
}

// ---- consensus --------------------------------------------------------------------------------------------------
// Where the per-query output goes: the record (its header written, bean_base / acc_base set), and its reserved beans /
// accession references (g of each).  The consensus writes the record through write_outcome().
struct QueryOut {
    blu_record* rec;
    blu_bean* beans;
    blu_acc* accs;
};

BLU_HD int bytes_cmp(const uint8_t* a, int la, const uint8_t* b, int lb) {
    int n = la < lb ? la : lb;
    for (int i = 0; i < n; i++) {
        int d = (int)a[i] - (int)b[i];
        if (d) return d;
    }
    return la - lb;
}

// the cutoff part of an outcome, by rank selection on a reference lineage (build_blast_consensus_identity.rs:22-37,66-95)
BLU_HD Outcome apply_cutoffs(const LinTables& T, uint32_t ref_lin, double identity, bool whole_filter, int idx) {
    const uint32_t o = T.lin_off[ref_lin];
    const int k = (int)(T.lin_off[ref_lin + 1] - o);
    int allowed = -1;
    for (int j = 0; j < k; j++)
        if (!(identity > T.cut[o + j])) {  // skip_while(identity > cut) linnaean_ranks.rs:182-189
            allowed = j;
            break;
        }
    uint64_t mask = 0;
    int kept = 0;
    for (int j = 0; j < k; j++)
        if (identity >= T.cut[o + j]) {  // linnaean_ranks.rs:208
            if (whole_filter || kept <= idx) mask |= 1ULL << j;  // enumerate AFTER the filter, take_while(index <= bean_index)
            kept++;
        }
    return cutoff_outcome(mask, allowed, idx, allowed >= 0 && T.rank_cls[o + idx] != T.allowed_cls[o + allowed]);
}

// |G| == 1 (find_single_query_consensus.rs:74-150)
BLU_HD uint32_t consensus_single(const TopRow& r, const LinTables& T, QueryOut out) {
    const uint32_t o = T.lin_off[r.lin];
    const int k = r.lin_len;
    uint64_t mask = 0;
    int last = -1;
    for (int j = 0; j < k; j++)
        if (r.pident >= T.cut[o + j]) {
            mask |= 1ULL << j;
            last = j;
        }
    if (last < 0) {
        write_outcome(out.rec, Outcome{});
        return DE_EMPTY_ADJUSTED;
    }
    out.beans[0].first_lineage = r.lin;
    out.beans[0].occurrences = 1;
    out.beans[0].acc_begin = 0;
    out.beans[0].n_acc = 1;
    out.accs[0].ref = (r.acc_off << 16) | (uint64_t)r.acc_len;
    write_outcome(out.rec, single_outcome(mask, r.pident, r.lin));
    return DE_NONE;
}

// sort comparator of find_multi_taxa_consensus.rs:41-54, made total by the file order (stable sort)
BLU_HD bool row_less(const TopRow* rows, const uint8_t* text, int a, int b) {
    const TopRow& x = rows[a];
    const TopRow& y = rows[b];
    if (x.lin_len != y.lin_len) return x.lin_len < y.lin_len;
    if (x.pident < y.pident) return true;
    if (x.pident > y.pident) return false;
    if (x.alnlen != y.alnlen) return x.alnlen < y.alnlen;
    int c = bytes_cmp(text + x.acc_off, x.acc_len, text + y.acc_off, y.acc_len);
    if (c) return c < 0;
    return a < b;
}

// |G| > 1 (find_multi_taxa_consensus.rs:22-217 + build_blast_consensus_identity.rs).
// rows[0..g) in file order; `text` is the base the acc_off offsets are relative to (generic pointer).
// scratch: order[g], bean_of[g], bean_first[g], bean_cnt[g], bean_ord[g]  (uint16_t each, caller-provided).
BLU_HD_NOINLINE uint32_t consensus_multi(const TopRow* rows, int g, const uint8_t* text, const LinTables& T, int strategy,
                                         uint16_t* scratch, QueryOut out) {
    uint16_t* order = scratch;
    uint16_t* bean_of = scratch + g;
    uint16_t* bean_first = scratch + 2 * g;
    uint16_t* bean_cnt = scratch + 3 * g;
    uint16_t* bean_ord = scratch + 4 * g;
    // S = stable sort (insertion sort for small g, heap-free shell otherwise: comparator is total)
    for (int i = 0; i < g; i++) order[i] = (uint16_t)i;
    if (g <= 64) {
        for (int i = 1; i < g; i++) {
            uint16_t v = order[i];
            int j = i - 1;
            while (j >= 0 && row_less(rows, text, v, order[j])) {
                order[j + 1] = order[j];
                j--;
            }
            order[j + 1] = v;
        }
    } else {
        // heap sort (total order => stability is irrelevant)
        auto sift = [&](int start, int end) {
            int root = start;
            while (2 * root + 1 <= end) {
                int child = 2 * root + 1, sw = root;
                if (row_less(rows, text, order[sw], order[child])) sw = child;
                if (child + 1 <= end && row_less(rows, text, order[sw], order[child + 1])) sw = child + 1;
                if (sw == root) return;
                uint16_t t = order[root];
                order[root] = order[sw];
                order[sw] = t;
                root = sw;
            }
        };
        for (int s = (g - 2) / 2; s >= 0; s--) sift(s, g - 1);
        for (int e = g - 1; e > 0; e--) {
            uint16_t t = order[e];
            order[e] = order[0];
            order[0] = t;
            sift(0, e - 1);
        }
    }
    const TopRow& ref = rows[strategy == BLU_STRATEGY_CAUTIOUS ? order[0] : order[g - 1]];  // fmtc.rs:60-63
    const int m = rows[order[0]].lin_len;  // shortest lineage; levels >= m are skipped (take_while + continue)
    // level walk (fmtc.rs:137-214): first level where the level keys disagree
    int diverge = -1;
    double max_pident = 0.0;
    for (int i = 0; i < m; i++) {
        uint32_t k0 = T.lvl_key[T.lin_off[rows[0].lin] + i];
        bool same = true;
        for (int r = 1; r < g; r++)
            if (T.lvl_key[T.lin_off[rows[r].lin] + i] != k0) {
                same = false;
                break;
            }
        if (!same) {
            diverge = i;
            break;
        }
    }
    int idx, level;
    bool single;
    double identity;
    if (diverge == 0) {
        write_outcome(out.rec, Outcome{});
        return DE_ROOT_DISAGREE;
    }
    if (diverge > 0) {
        for (int r = 0; r < g; r++)
            if (rows[r].pident > max_pident) max_pident = rows[r].pident;  // fold from 0.0 (fmtc.rs:182-185)
        idx = diverge - 1;
        level = diverge;
        single = false;
        identity = max_pident;
    } else {
        idx = m - 1;
        level = m - 1;
        single = true;
        identity = ref.pident;
    }
    // fold beans at `level` in S order (consensus_result.rs:65-88)
    int nb = 0;
    for (int s = 0; s < g; s++) {
        const TopRow& r = rows[order[s]];
        uint32_t key = T.bean_key[T.lin_off[r.lin] + level];
        int b = -1;
        for (int j = 0; j < nb; j++)
            if (T.bean_key[T.lin_off[rows[bean_first[j]].lin] + level] == key) {
                b = j;
                break;
            }
        if (b < 0) {
            b = nb++;
            bean_first[b] = order[s];
            bean_cnt[b] = 0;
        }
        bean_cnt[b]++;
        bean_of[s] = (uint16_t)b;
    }
    // sort beans: occurrences desc, identifier asc (bbci.rs:50-60); deterministic tie-break on the key id
    for (int j = 0; j < nb; j++) bean_ord[j] = (uint16_t)j;
    for (int i = 1; i < nb; i++) {
        uint16_t v = bean_ord[i];
        int j = i - 1;
        while (j >= 0) {
            uint16_t w = bean_ord[j];
            bool less;
            if (bean_cnt[v] != bean_cnt[w])
                less = bean_cnt[v] > bean_cnt[w];
            else {
                uint32_t pv = T.lin_off[rows[bean_first[v]].lin] + level, pw = T.lin_off[rows[bean_first[w]].lin] + level;
                if (T.ident_rank[pv] != T.ident_rank[pw])
                    less = T.ident_rank[pv] < T.ident_rank[pw];
                else
                    less = T.bean_key[pv] < T.bean_key[pw];
            }
            if (!less) break;
            bean_ord[j + 1] = w;
            j--;
        }
        bean_ord[j + 1] = v;
    }
    // emit beans + accession lists (S order, consecutive duplicates removed: Vec::dedup)
    uint32_t na = 0;
    for (int bi = 0; bi < nb; bi++) {
        int b = bean_ord[bi];
        uint32_t begin = na;
        int prev = -1;
        for (int s = 0; s < g; s++) {
            if (bean_of[s] != b) continue;
            const TopRow& r = rows[order[s]];
            if (prev >= 0) {
                const TopRow& q = rows[prev];
                if (q.acc_len == r.acc_len && bytes_cmp(text + q.acc_off, q.acc_len, text + r.acc_off, r.acc_len) == 0) continue;
            }
            out.accs[na].ref = (r.acc_off << 16) | (uint64_t)r.acc_len;
            na++;
            prev = order[s];
        }
        out.beans[bi].first_lineage = rows[bean_first[b]].lin;
        out.beans[bi].occurrences = bean_cnt[b];
        out.beans[bi].acc_begin = begin;
        out.beans[bi].n_acc = na - begin;
    }
    write_outcome(out.rec, found_outcome(apply_cutoffs(T, ref.lin, identity, single && nb == 1, idx), ref.pident, ref.lin, (uint32_t)nb, level, false));
    return DE_NONE;
}

}  // namespace blu
