// Stage 1 (K1): eventalign TSV tokeniser + line filter.  One WARP per 3840-byte text chunk, no block barriers,
// text staged by TMA bulk copies (cp.async.bulk + mbarrier) one chunk ahead of the parse; chunks that provably hold
// nothing of interest are passed over after a look at the first two columns of their lines.
//
// Replaces the reader / tokeniser / per-line filters of the reference's extract_features
// (extract_contexts.py:140-176): readlines + line.split()[:12], the '<12 fields' drop (:149-152),
// the contig lookup (:154-160), the NNNNNN drop (:167) and the "does this k-mer touch an 'M'"
// test that gates everything after (:176, :242, :269).
//
// Persistent warps take RUNS of consecutive chunks (dynamic claim, one atomic per run) and carry "was the last kept line
// a candidate" from chunk to chunk.  Per chunk:
//   0. lane 0 has already asked the TMA engine for the 4096 staged bytes of this chunk (32 B look-behind, the
//      3840-byte chunk, 224 B look-ahead) while the previous chunk was being parsed; it now issues the copy of the
//      warp's next chunk into the other buffer and the warp waits on this buffer's mbarrier;
//   1. each lane builds the newline bit map of 4 x 32 B in registers (SWAR compare, 3 instructions per word, + IDP.4A bit
//      packing) and derives the line starts inside its own 128 bytes;
//   2a. quiet test (only when the last kept line was not a candidate): every lane looks at the line(s) starting in its
//      128 bytes -- 8-byte register compare with the warp's contig hint, position decoded from one 8-byte register load,
//      one bit test in the per-position candidate bitmap (L1/L2 resident).  If every line is "hint contig, plain position,
//      not a candidate" the chunk is done: none of its lines can get a record or change the carried state, whatever the
//      rest of the line holds.  (~91 % of the chunks for GATC.)
//   3. otherwise the full parse: non-whitespace map -> field starts = nonws & ~(nonws << 1); per-lane line counts
//      prefix-summed with two ballots into a 32-entry line list; one lane per line: rank/select on the field-start bits
//      finds columns 1, 2, 10 and 12 without touching the bytes in between (the ~58 B read name is never walked); 12-column
//      check, contig lookup, NNNNNN test, position, candidate bit;
//   4. warp ballots decide which lines matter (candidate, successor of a candidate, first kept line of the run, or
//      every kept line in dense mode); those get a 32-byte raw record {line offset, position, contig, flags, the first 128
//      field-start bits of the line}.  Their values (event index, currents, k-mer equality, read-name span, the k-mer's
//      target bits) are filled in by stage 2 at full lane occupancy, which finds the columns from the field-start bits
//      instead of walking the line again.  Finishing the records here -- from the staged bytes, or in L2-hot batches of 32 --
//      was measured at +3 ms and +10 ms on this kernel: long dependent chains in a warp that has one chunk of prefetch
//      in flight starve the memory pipeline.
//      Record slots are reserved per warp in blocks of 256, so the global allocation counter sees ~1 atomic per 300 chunks.
// Lines whose first 12 columns do not fit the look-ahead are classified byte-wise straight from global memory.
// Algorithmic HBM traffic: the text itself (once) + 32 B per record (~1 B per line in sparse mode).
#include "parse.cuh"

namespace {

constexpr int CHUNK = MC_TILE_BYTES;          // 3840 = 30 * 128: ~30 lines of ~128 B, one per lane
constexpr int LOOKB = 32;
constexpr int LOOKA = 224;
constexpr int WB = LOOKB + CHUNK + LOOKA;     // 4096 bytes staged per chunk
constexpr int NW = WB / 32;                   // 128 mask words = 4 per lane
#ifndef MC_SCAN_WARPS
#define MC_SCAN_WARPS 24
#endif
#ifndef MC_SCAN_MIN_CTAS
#define MC_SCAN_MIN_CTAS 1
#endif
#ifndef MC_SCAN_RUN
#define MC_SCAN_RUN 128
#endif

constexpr int WARPS = MC_SCAN_WARPS;
constexpr int THREADS = WARPS * 32;
constexpr int LCAP = 32;                      // lines per pass (one per lane)
constexpr int RESERVE = 256;                  // record slots reserved per global atomic
static_assert(WB == 4096 && NW == 128, "chunk geometry");
static_assert(CHUNK % 16 == 0, "chunks must keep 16-byte alignment");
static_assert(MC_TEXT_PAD >= LOOKA + 64, "text padding must cover the look-ahead");

struct WarpSmem {
    alignas(16) uint8_t text[2][WB];     // double-buffered staged bytes (TMA destination, 16-byte aligned)
    alignas(16) uint32_t fs[NW + 8];     // field-start bits (zero padded)
    alignas(16) uint32_t nl[NW + 4];     // newline bits
    uint16_t lstart[LCAP + 4];
    uint32_t cnt[8];                     // per-warp event counters (flushed once at the end)
    unsigned long long key[4];           // the hint contig's name in 8-byte pieces (quiet test; names of up to 31 bytes)
    alignas(8) unsigned long long bar[2];
    unsigned long long rname[8];         // read-first mode: the read name of the last line seen, zero padded (names of up to 64 bytes)
};

// ---- TMA / mbarrier wrappers ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// bounded wait: returns false if the phase never completes (reported through the overflow counter instead of hanging)
__device__ __forceinline__ bool mbar_wait(unsigned long long *bar, uint32_t parity) {
    const uint32_t a = smem_u32(bar);
    for (uint32_t spin = 0; spin < (1u << 26); ++spin) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
        if (done) return true;
    }
    return false;
}

// ---- byte classification ---------------------------------------------------------------------------------------------
// 8 msb-form words (0x80 per flagged byte) -> 32 flag bits in byte order, as pack16 does for 4
// (not two pack16 calls: their OR form costs k_scan about 40 more instructions than this sum)
__device__ __forceinline__ uint32_t pack32(uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3, uint32_t m4, uint32_t m5,
                                           uint32_t m6, uint32_t m7) {
    const uint32_t lo = 0x08040201u, hi = 0x80402010u;
    const uint32_t a = __dp4a(m1, hi, __dp4a(m0, lo, 0u));
    const uint32_t b = __dp4a(m3, hi, __dp4a(m2, lo, 0u));
    const uint32_t c = __dp4a(m5, hi, __dp4a(m4, lo, 0u));
    const uint32_t d = __dp4a(m7, hi, __dp4a(m6, lo, 0u));
    return (a >> 7) + b * 2u + c * 512u + d * 131072u;
}

// ---- generic field walk (rare: lines whose first 12 columns do not fit the 160-bit window) ------------------------------
// position of the n-th (0-based) field start at or after smem offset s; NW*32 when it lies beyond the staged bytes
__device__ __noinline__ int select_fs_walk(const uint32_t *fs, int s, int n) {
    int w = s >> 5;
    uint32_t m = fs[w] & (0xFFFFFFFFu << (s & 31));
    int c = __popc(m);
    while (c <= n) {
        n -= c;
        if (++w >= NW) return NW * 32;
        m = fs[w];
        c = __popc(m);
    }
    for (; n > 0; --n) m &= m - 1u;
    return (w << 5) + __ffs(m) - 1;
}
__device__ __forceinline__ int next_bit(const uint32_t *m, int q) {
    int w = q >> 5;
    uint32_t v = m[w] & (0xFFFFFFFFu << (q & 31));
    while (v == 0u) {
        if (++w >= NW) return NW * 32;
        v = m[w];
    }
    return (w << 5) + __ffs(v) - 1;
}

// ---- field location: 160-bit window of field-start bits aligned at the line start, branch-free rank/select -------------
template <bool WANT3>
__device__ __forceinline__ void line_fields(const WarpSmem &S, int s, int &f0, int &f1, int &f9, int &f11, int &f3) {
    const int w0 = s >> 5, sh = s & 31;
    const uint32_t a0 = S.fs[w0], a1 = S.fs[w0 + 1], a2 = S.fs[w0 + 2], a3 = S.fs[w0 + 3], a4 = S.fs[w0 + 4], a5 = S.fs[w0 + 5];
    const uint32_t W0 = __funnelshift_r(a0, a1, sh), W1 = __funnelshift_r(a1, a2, sh), W2 = __funnelshift_r(a2, a3, sh),
                   W3 = __funnelshift_r(a3, a4, sh), W4 = __funnelshift_r(a4, a5, sh);
    const int c0 = __popc(W0), c1 = c0 + __popc(W1), c2 = c1 + __popc(W2), c3 = c2 + __popc(W3), c4 = c3 + __popc(W4);
    if (c4 >= 12) {
        auto sel = [&](int k) {
            const int wi = (k >= c0) + (k >= c1) + (k >= c2) + (k >= c3);
            const uint32_t m = wi == 0 ? W0 : wi == 1 ? W1 : wi == 2 ? W2 : wi == 3 ? W3 : W4;
            const int base = wi == 0 ? 0 : wi == 1 ? c0 : wi == 2 ? c1 : wi == 3 ? c2 : c3;
            return s + 32 * wi + nth_bit(m, k - base);
        };
        if ((W0 & 1u) && c0 >= 2) {          // the line starts with its first column and the second starts within 32 bytes
            f0 = s;
            f1 = s + __ffs(W0 & (W0 - 1u)) - 1;
        } else {
            f0 = sel(0);
            f1 = sel(1);
        }
        if (WANT3) f3 = c0 >= 4 ? s + nth_bit(W0, 3) : sel(3);      // column 4 (read name): inside the first 32 bytes as a rule
        if (c2 <= 9 && c3 > 11) {
            // usual layout (a ~128-byte line): columns 10 and 12 both start inside the fourth window word
            uint32_t m = W3;
            const int j = 9 - c2;
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (j > t) m &= m - 1u;
            for (int t = 4; t < j; ++t) m &= m - 1u;
            f9 = s + 96 + __ffs(m) - 1;
            m &= m - 1u;
            m &= m - 1u;
            f11 = s + 96 + __ffs(m) - 1;
        } else {
            f9 = sel(9);
            f11 = sel(11);
        }
    } else {
        // fewer than 12 field starts within 160 bytes: short line or unusually wide columns -> generic walk
        f0 = select_fs_walk(S.fs, s, 0);
        f1 = select_fs_walk(S.fs, s, 1);
        f9 = select_fs_walk(S.fs, s, 9);
        f11 = select_fs_walk(S.fs, s, 11);
        if (WANT3) f3 = select_fs_walk(S.fs, s, 3);
    }
}

// first 8 bytes at smem offset q (any alignment) as a little-endian u64
__device__ __forceinline__ unsigned long long load8(const uint8_t *text, int q) {
    const uint32_t *wp = reinterpret_cast<const uint32_t *>(text + (q & ~3));
    const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2];
    const int sh = 8 * (q & 3);
    const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
    return ((unsigned long long)hi << 32) | lo;
}

// position column decoded from its first 8 bytes in registers: up to 7 digits and the byte that ends them.
// Returns 1 (pos set), 0 (not a number / not followed by whitespace) or -1 (8 or more digits: take the byte loop).
__device__ __forceinline__ int parse_pos8(unsigned long long k8, int &pos) {
    const uint32_t lo = (uint32_t)k8, hi = (uint32_t)(k8 >> 32);
    const uint32_t xl = lo ^ 0x30303030u, xh = hi ^ 0x30303030u;
    const uint32_t ndl = (((xl & 0x7f7f7f7fu) + 0x76767676u) | lo) & 0x80808080u;      // 0x80 where the byte is not a digit
    const uint32_t ndh = (((xh & 0x7f7f7f7fu) + 0x76767676u) | hi) & 0x80808080u;
    if ((ndl | ndh) == 0u) return -1;
    const int n = ndl ? ((__ffs(ndl) - 1) >> 3) : 4 + ((__ffs(ndh) - 1) >> 3);          // leading digits: 0..7
    const uint32_t term = (n < 4 ? (lo >> (8 * n)) : (hi >> (8 * n - 32))) & 0xFFu;
    if (n == 0 || term > 0x20u) return 0;
    // right-align the digits in the 8 bytes (leading zero digits below them), then two 4-digit conversions
    const int sh = 64 - 8 * n;                                                           // 8..56
    const uint32_t H = sh < 32 ? __funnelshift_l(xl, xh, sh) : (xl << (sh - 32));
    const uint32_t L = sh < 32 ? (xl << sh) : 0u;
    pos = (int)(conv4(L) * 10000u + conv4(H));
    return 1;
}

// ---- read-first mode (sparse scan with -q): read names of neighbouring lines ------------------------------------------
// length of the token at smem offset q (bytes > 0x20), -1 when it is longer than 64 bytes
__device__ __forceinline__ int token_len64(const uint8_t *text, int q) {
    for (int j = 0; j < 9; ++j) {
        const unsigned long long v = load8(text, q + 8 * j);
        const uint32_t lo = gt20_msb((uint32_t)v) ^ 0x80808080u, hi = gt20_msb((uint32_t)(v >> 32)) ^ 0x80808080u;   // 0x80 = whitespace
        if (lo) return 8 * j + ((__ffs(lo) - 1) >> 3);
        if (hi) return 8 * j + 4 + ((__ffs(hi) - 1) >> 3);
    }
    return -1;
}
__device__ __forceinline__ unsigned long long low_bytes(unsigned long long v, int n) {          // first n (0..8) bytes of v
    return n >= 8 ? v : (v & ((1ull << (8 * n)) - 1ull));
}
// token of `len` bytes at q equal to the zero-padded pieces key[]
__device__ __forceinline__ bool token_is(const uint8_t *text, int q, int len, const unsigned long long *key) {
    bool eq = true;
    for (int j = 0; 8 * j < len; ++j) eq = eq && low_bytes(load8(text, q + 8 * j), len - 8 * j) == key[j];
    return eq;
}
// the `len` bytes at qa equal the `len` bytes at qb
__device__ __forceinline__ bool spans_equal(const uint8_t *text, int qa, int qb, int len) {
    bool eq = true;
    for (int j = 0; 8 * j < len; ++j) eq = eq && low_bytes(load8(text, qa + 8 * j) ^ load8(text, qb + 8 * j), len - 8 * j) == 0ull;
    return eq;
}
// digits of a position column decoded by parse_pos8 (1..7)
__device__ __forceinline__ int pos_digits8(unsigned long long k8) {
    const uint32_t lo = (uint32_t)k8, hi = (uint32_t)(k8 >> 32);
    const uint32_t xl = lo ^ 0x30303030u, xh = hi ^ 0x30303030u;
    const uint32_t ndl = (((xl & 0x7f7f7f7fu) + 0x76767676u) | lo) & 0x80808080u;
    const uint32_t ndh = (((xh & 0x7f7f7f7fu) + 0x76767676u) | hi) & 0x80808080u;
    return ndl ? ((__ffs(ndl) - 1) >> 3) : 4 + ((__ffs(ndh) - 1) >> 3);
}

enum { ST_KEPT = 1u, ST_CAND = 2u, ST_SHORT = 4u, ST_UNKNOWN = 8u, ST_NNN = 16u, ST_BADPOS = 32u };

// contig / NNNNNN / position / candidate test of one line whose columns 1, 2, 10 start at f0, f1, f9
template <class B>
__device__ __forceinline__ uint32_t classify_line(const B &t, int f0, int f1, int f9, const mc_refindex &R, int hint, int64_t hint_base,
                                                  int hint_len, int known_cid, int nnn_state /* 1 yes, 0 no, -1 unknown */,
                                                  int pos_state /* 1 pos set, 0 bad, -1 unknown */, int &cid, int &pos) {
    cid = known_cid >= 0 ? known_cid : contig_lookup(t, f0, R, hint);
    if (cid < 0) return ST_UNKNOWN;
    if (nnn_state > 0 || (nnn_state < 0 && is_nnnnnn(t, f9))) return ST_NNN;
    if (pos_state == 0 || (pos_state < 0 && !parse_uint(t, f1, pos))) return ST_BADPOS;
    uint32_t st = ST_KEPT;
    const int len = (cid == hint) ? hint_len : __ldg(R.d_len + cid);
    if (pos < len) {
        const int64_t g = ((cid == hint) ? hint_base : __ldg(R.d_base + cid)) + pos;
        if ((__ldg(R.d_cand + (g >> 5)) >> (g & 31)) & 1u) st |= ST_CAND;
    }
    return st;
}

// a line whose first 12 columns outran the staged look-ahead: byte-wise from global memory
__device__ __noinline__ uint32_t classify_from_global(const uint8_t *d_text, int64_t limit, int64_t goff, const mc_refindex &R, int hint,
                                                      int64_t hint_base, int hint_len, int &cid, int &pos) {
    const GlobalBytes t{d_text + goff, limit - goff};
    int nf = 0, f0 = 0, f1 = 0, f9 = 0;
    bool in_tok = false;
    for (int i = 0; i < (1 << 20); ++i) {
        const int c = t[i];
        if (c == 0x0a) break;
        const bool ws = c <= 0x20;
        if (!ws && !in_tok) {
            if (nf == 0) f0 = i; else if (nf == 1) f1 = i; else if (nf == 9) f9 = i;
            ++nf;
            in_tok = true;
            if (nf >= 12) break;
        } else if (ws) in_tok = false;
    }
    if (nf < 12) return ST_SHORT;
    return classify_line(t, f0, f1, f9, R, hint, hint_base, hint_len, -1, -1, -1, cid, pos);
}

// RF ("read-first" mode, the sparse scan under -q): the first kept line of every READ gets a record too, so that stage 4 can
// filter whole reads by quality and still find the line that closes a window left open at the end of a read -- the first
// kept line of the next read that passes (extract_contexts.py:167 runs before :179).  The warp carries the read name of
// the last line it saw and "this read already has a kept line"; a chunk is quiet only if all its lines carry that name.
template <bool RF>
__global__ void __launch_bounds__(THREADS, MC_SCAN_MIN_CTAS)
k_scan(const uint8_t *__restrict__ d_text, int64_t nbytes, int64_t text_limit16, int64_t n_chunks64, int run_len, mc_refindex R,
       int dense, mc_record *__restrict__ d_rec, unsigned long long rec_cap, uint32_t *__restrict__ d_tile_tab,
       uint32_t *__restrict__ d_run_tab, unsigned long long *__restrict__ d_counters) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    WarpSmem &S = reinterpret_cast<WarpSmem *>(smem_raw)[wib];
    const int warp_global = (int)blockIdx.x * WARPS + wib;      // chunk indices fit 32 bits (mc_scan checks)
    const int n_warps = (int)gridDim.x * WARPS;
    const int n_chunks = (int)n_chunks64;
    const int n_runs = (n_chunks + run_len - 1) / run_len;       // a run = run_len consecutive chunks parsed by one warp
    const uint32_t lt_mask = (1u << lane) - 1u;

    // byte == 0x0a in three instructions per word: a LOP3 folds only one immediate, so the 0x7f mask is made a run-time
    // value (nbytes is never negative, which the compiler cannot know) and lives in a register: (w ^ imm) & reg is one LOP3
    const uint32_t K7F = 0x7f7f7f7fu | ((uint32_t)((unsigned long long)nbytes >> 63) << 7);
    auto eq0a_r = [&](uint32_t w) -> uint32_t {
        const uint32_t t = ((w ^ 0x0a0a0a0au) & K7F) + K7F;       // bit 7 set iff the low 7 bits differ from 0x0a
        return ~(t | w) & 0x80808080u;
    };

    // warp-uniform state
    int hint = -1;
    int64_t hint_base = 0;
    int hint_len = 0, hint_nlen = 0;
    unsigned long long hint_key = 0ull;                           // first bytes of the hint contig's name (fast compare)
    auto set_hint = [&](int c) {
        hint = c;
        hint_base = __ldg(R.d_base + c);
        hint_len = __ldg(R.d_len + c);
        const int o0 = __ldg(R.d_name_off + c);
        hint_nlen = __ldg(R.d_name_off + c + 1) - o0;
        hint_key = 0ull;
        for (int j = 0; j < hint_nlen && j < 7; ++j) hint_key |= (unsigned long long)__ldg(R.d_names + o0 + j) << (8 * j);
        __syncwarp();
        if (lane < 4) {
            unsigned long long kk = 0ull;
            for (int j = 8 * lane; j < hint_nlen && j < 8 * lane + 8; ++j) kk |= (unsigned long long)__ldg(R.d_names + o0 + j) << (8 * (j & 7));
            S.key[lane] = kk;
        }
        __syncwarp();
    };
    set_hint(0);
    unsigned long long slot_cur = 0ull;                           // next free reserved record slot
    unsigned slot_left = 0u;                                      // slots left in the warp's reserved block
    unsigned c_lines = 0, c_kept = 0;                             // c_lines per lane, c_kept warp-uniform; rarer events in S.cnt
    if (lane < 8) S.cnt[lane] = 0u;

    if (lane == 0) {
        mbar_init(&S.bar[0], 1);
        mbar_init(&S.bar[1], 1);
        fence_barrier_init();
    }
    __syncwarp();
    uint32_t phase0 = 0u, phase1 = 0u;

    // stage a chunk: interior chunks by one TMA bulk copy (asynchronous), edge chunks by guarded loads (synchronous)
    // chunks 1 .. c_bulk_hi have all 4096 staged bytes inside the (padded) text; chunks >= c_tail_lo touch its end
    const int64_t q_hi = text_limit16 - WB + LOOKB, q_tail = nbytes - WB + LOOKB;
    const int c_bulk_hi = q_hi < 0 ? -1 : (int)min(q_hi / CHUNK, (int64_t)0x7fffffff);
    const int c_tail_lo = q_tail < 0 ? 0 : (int)min(q_tail / CHUNK + 1, (int64_t)0x7fffffff);
    auto stage = [&](int c, int b) -> bool {
        const int64_t g0 = (int64_t)c * CHUNK - LOOKB;
        if (c >= 1 && c <= c_bulk_hi) {
            if (lane == 0) {
                fence_proxy_async();                               // earlier generic reads of this buffer are done (__syncwarp)
                tma_load_1d(S.text[b], d_text + g0, WB, &S.bar[b]);
            }
            return true;
        }
        for (int i = lane; i < WB / 16; i += 32) {
            const int64_t g = g0 + 16 * i;
            uint4 v = make_uint4(0x0a0a0a0au, 0x0a0a0a0au, 0x0a0a0a0au, 0x0a0a0a0au);
            if (g >= 0 && g < text_limit16) v = __ldg(reinterpret_cast<const uint4 *>(d_text + g));
            *reinterpret_cast<uint4 *>(S.text[b] + 16 * i) = v;
        }
        return false;
    };

    // RF: does every lane's line carry the read name S.rname?  nm = where the lane's name starts in the staged bytes (-1: no
    // line).  16 lanes x 4 bytes cover a name (<= 63 bytes) and the byte that must end it; two lines per step, one per half
    // warp, so the shared-memory reads are free of bank conflicts.  Warp-uniform result.
    int rname_len = -1;            // length of the read name in S.rname (-1: unknown / too long)
    auto rf_all_match = [&](const uint8_t *text, int nm) -> bool {
        const int j = lane & 15;
        const uint32_t kw = reinterpret_cast<const uint32_t *>(S.rname)[j];
        const int nb = rname_len - 4 * j;                                  // name bytes from this lane's word on
        const uint32_t kmask = nb >= 4 ? 0xFFFFFFFFu : nb <= 0 ? 0u : ((1u << (8 * nb)) - 1u);
        const bool term_lane = j == (rname_len >> 2);
        const int term_sh = 8 * (rname_len & 3);
        const uint32_t *tw32 = reinterpret_cast<const uint32_t *>(text);
        uint32_t have = __ballot_sync(0xffffffffu, nm >= 0);
        while (have) {
            const int oa = __ffs(have) - 1;
            have &= have - 1u;
            const int ob = have ? __ffs(have) - 1 : -1;
            have &= have - 1u;                                             // (0 & anything stays 0)
            const int o = lane < 16 ? oa : ob;
            const int a = __shfl_sync(0xffffffffu, nm, o < 0 ? 0 : o) + 4 * j;
            const uint32_t v = __funnelshift_r(tw32[a >> 2], tw32[(a >> 2) + 1], 8 * (a & 3));
            bool bad = ((v ^ kw) & kmask) != 0u;
            if (term_lane && ((v >> term_sh) & 0xFFu) > 0x20u) bad = true;
            if (o < 0) bad = false;
            if (__any_sync(0xffffffffu, bad)) return false;
        }
        return true;
    };

    // Runs are claimed dynamically: run `warp_global` first, then one atomic per run on the run cursor.  Inside a run the
    // state of the last kept line (prev_state) carries from chunk to chunk, so only the first kept line of a RUN is a
    // "filler" record that stage 2 may have to drop.
    int buf = 0;
    bool cur_async = false;
    int chunk = warp_global < n_runs ? warp_global * run_len : n_chunks;
    int run_end = min(chunk + run_len, n_chunks);
    if (chunk < n_chunks) cur_async = stage(chunk, 0);
    int prev_state = -1;           // -1: no kept line yet in this run, 0: last kept line not a candidate, 1: candidate
    bool read_has_kept = false;    // RF: the read S.rname names already has a kept line in this run
    unsigned run_total = 0u, run_filler = 0u;                     // records / filler flag of the run so far

    while (chunk < n_chunks) {
        const int64_t G0 = (int64_t)chunk * CHUNK - LOOKB;        // global offset of staged byte 0
        const bool tail = chunk >= c_tail_lo;                     // chunk touches the end of the text (G0 + WB > nbytes)
        __syncwarp();
        // ---- 0. prefetch the next chunk (claiming the next run at the end of this one), wait for this chunk ------------------
        int next = chunk + 1, next_end = run_end;
        const bool last_of_run = next >= run_end;
        if (last_of_run) {
            unsigned long long got = 0ull;
            if (lane == 0) got = atomicAdd(&d_counters[MC_C_RUN_CURSOR], 1ull);
            got = __shfl_sync(0xffffffffu, got, 0) + (unsigned long long)n_warps;
            next = got < (unsigned long long)n_runs ? (int)got * run_len : n_chunks;
            next_end = min(next + run_len, n_chunks);
        }
        bool next_async = false;
        if (next < n_chunks) next_async = stage(next, buf ^ 1);
        if (cur_async) {
            const uint32_t ph = buf ? phase1 : phase0;
            if (!mbar_wait(&S.bar[buf], ph) && lane == 0) atomicAdd(&S.cnt[5], 1u);
            if (buf) phase1 ^= 1u; else phase0 ^= 1u;
        }
        __syncwarp();
        const uint8_t *text = S.text[buf];
        const SmemBytes T{text};

        // ---- 1. newline map: lane owns words lane, lane+32, lane+64, lane+96 -------------------------------------------------
        // byte == 0x0a in three instructions per word (LOP3, IADD, LOP3) with the three masks held in registers
        // (the non-whitespace / field-start map is built only when a pass of this chunk needs the full parse, see 3b)
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int w = 32 * r + lane;
            const uint4 va = *reinterpret_cast<const uint4 *>(text + 32 * w);
            const uint4 vb = *reinterpret_cast<const uint4 *>(text + 32 * w + 16);
            S.nl[w] = pack32(eq0a_r(va.x), eq0a_r(va.y), eq0a_r(va.z), eq0a_r(va.w), eq0a_r(vb.x), eq0a_r(vb.y), eq0a_r(vb.z),
                             eq0a_r(vb.w));
        }
        if (lane == 0) S.nl[NW] = 0xFFFFFFFFu;
        __syncwarp();
        bool full_ready = false;   // field-start map and e_last built for this chunk

        // ---- 2. line list: lane owns words 4*lane .. 4*lane+3 ------------------------------------------------------------------
        // line starts: byte p starts a line iff byte p-1 is '\n'; owned words are LOOKB/32 .. (LOOKB+CHUNK)/32 - 1, global p < nbytes
        uint4 lsv;
        {
            const uint4 nlv = *reinterpret_cast<const uint4 *>(&S.nl[4 * lane]);
            const uint32_t nprev = lane ? S.nl[4 * lane - 1] : 0u;
            lsv.x = (nlv.x << 1) | (nprev >> 31);
            lsv.y = (nlv.y << 1) | (nlv.x >> 31);
            lsv.z = (nlv.z << 1) | (nlv.y >> 31);
            lsv.w = (nlv.w << 1) | (nlv.z >> 31);
            constexpr int W_LO = LOOKB / 32, W_HI = (LOOKB + CHUNK) / 32;      // owned words [W_LO, W_HI)
            static_assert(W_LO == 1 && W_HI == 121, "the lane tests below assume words 1..120 are owned");
            const int w0 = 4 * lane;
            if (lane == 0) lsv.x = 0u;                                          // word 0 is look-behind
            if (lane >= 30) {                                                   // words 121..127 are look-ahead
                if (lane == 31) lsv.x = 0u;
                lsv.y = 0u; lsv.z = 0u; lsv.w = 0u;
            }
            if (tail) {
                auto clip = [&](uint32_t v, int w) {
                    const int64_t room = nbytes - (G0 + 32 * w);
                    return room <= 0 ? 0u : (room < 32 ? (v & ((1u << room) - 1u)) : v);
                };
                lsv.x = clip(lsv.x, w0);
                lsv.y = clip(lsv.y, w0 + 1);
                lsv.z = clip(lsv.z, w0 + 2);
                lsv.w = clip(lsv.w, w0 + 3);
            }
        }
        const int my_cnt = __popc(lsv.x) + __popc(lsv.y) + __popc(lsv.z) + __popc(lsv.w);
        c_lines += (unsigned)my_cnt;                               // per lane; summed over the warp at the end

        // ---- 2a. quick look at every line of the chunk: "<hint contig><ws><digits><ws>" -> position -> candidate bit ----------
        // A chunk in which every line passes this test on a non-candidate position, entered with the last kept line not a
        // candidate, emits nothing and leaves that state as it is whatever else its lines hold (kept or not, a line on a
        // non-candidate position neither gets a record nor changes "last kept line is not a candidate"): it is done here,
        // without the field-start map, the line list or the per-line parse.  Lanes test the lines that start inside their
        // own 128 bytes (usually one, so one round).
        bool quiet_chunk = false;
        if (!dense && prev_state == 0 && hint_nlen >= 1 && hint_nlen <= 31 && (!RF || (read_has_kept && rname_len >= 1))) {
            uint32_t w0 = lsv.x, w1 = lsv.y, w2 = lsv.z, w3 = lsv.w;
            bool ok = true;
            int rf_round = 0, rf_nm1 = -1;                         // RF: where the read name of this lane's second line starts
            for (;; ++rf_round) {
                if (!__any_sync(0xffffffffu, (w0 | w1 | w2 | w3) != 0u)) break;
                if ((w0 | w1 | w2 | w3) != 0u) {
                    const int jw = w0 ? 0 : w1 ? 1 : w2 ? 2 : 3;
                    const uint32_t m = w0 ? w0 : w1 ? w1 : w2 ? w2 : w3;
                    const int s0 = 32 * (4 * lane + jw) + __ffs(m) - 1;
                    const uint32_t cl = m & (m - 1u);
                    if (jw == 0) w0 = cl; else if (jw == 1) w1 = cl; else if (jw == 2) w2 = cl; else w3 = cl;
                    // the name in 8-byte pieces, then the whitespace byte that must follow it
                    bool name_ok = true;
                    for (int j = 0; 8 * j <= hint_nlen; ++j) {
                        const unsigned long long v = load8(text, s0 + 8 * j), kk = S.key[j];
                        const int rem = hint_nlen - 8 * j;             // name bytes from this piece on
                        if (rem >= 8) name_ok = name_ok && v == kk;
                        else name_ok = name_ok && (v & ((1ull << (8 * rem)) - 1ull)) == kk && ((v >> (8 * rem)) & 0xFFull) <= 0x20ull;
                    }
                    ok = false;
                    if (name_ok) {
                        int p0 = 0;
                        const unsigned long long p8 = load8(text, s0 + hint_nlen + 1);
                        if (parse_pos8(p8, p0) == 1) {
                            ok = true;
                            if (p0 < hint_len) {
                                const int64_t g = hint_base + p0;
                                ok = ((__ldg(R.d_cand + (g >> 5)) >> (g & 31)) & 1u) == 0u;
                            }
                            if (RF && ok) {
                                // "<ws><k-mer of up to 7 bytes><ws><the carried read name><ws>" right after the position
                                const int km = s0 + hint_nlen + 1 + pos_digits8(p8) + 1;
                                const unsigned long long k8 = load8(text, km);
                                const uint32_t wl = gt20_msb((uint32_t)k8) ^ 0x80808080u, wh = gt20_msb((uint32_t)(k8 >> 32)) ^ 0x80808080u;
                                const int klen = wl ? ((__ffs(wl) - 1) >> 3) : wh ? 4 + ((__ffs(wh) - 1) >> 3) : 8;
                                ok = klen >= 1 && klen <= 7 && rf_round < 2;
                                const int nm = km + klen + 1;
                                if (rf_round == 0) {
                                    // first line of this lane (nearly every lane has one): the name against the carried one,
                                    // 4 bytes at a time, then the byte that must end it; uniform trip count
                                    const uint32_t *tw32 = reinterpret_cast<const uint32_t *>(text) + (nm >> 2);
                                    const uint32_t *kw32 = reinterpret_cast<const uint32_t *>(S.rname);
                                    const int sh = 8 * (nm & 3), nfull = rname_len >> 2;
                                    uint32_t prev = tw32[0], acc = 0u;
                                    for (int j = 0; j < nfull; ++j) {
                                        const uint32_t nxt = tw32[j + 1];
                                        acc |= __funnelshift_r(prev, nxt, sh) ^ kw32[j];
                                        prev = nxt;
                                    }
                                    const uint32_t v = __funnelshift_r(prev, tw32[nfull + 1], sh);
                                    const int nb = 8 * (rname_len & 3);
                                    acc |= (v ^ kw32[nfull]) & ((1u << nb) - 1u);
                                    ok = ok && acc == 0u && ((v >> nb) & 0xFFu) <= 0x20u;
                                } else {
                                    rf_nm1 = nm;       // second lines are few: compared below, a line per half warp
                                }
                            }
                        }
                    }
                }
                if (!__all_sync(0xffffffffu, ok)) { ok = false; break; }
            }
            if (RF && ok) ok = rf_all_match(text, rf_nm1);         // ... and the carried read name
            quiet_chunk = ok;                                      // warp-uniform
            if (ok && lane == 0) S.cnt[6] += 1u;
        }

        // ---- 2b. line list of a chunk that needs the full parse ---------------------------------------------------------------
        // exclusive prefix of the per-lane counts: two ballots when every lane holds at most 3 line starts (always, for
        // ~128-byte lines), a shuffle scan otherwise
        int my_first = 0, total_lines = 0;
        if (!quiet_chunk) {
            if (__ballot_sync(0xffffffffu, my_cnt > 3) == 0u) {
                const uint32_t b0 = __ballot_sync(0xffffffffu, my_cnt & 1), b1 = __ballot_sync(0xffffffffu, my_cnt & 2);
                my_first = __popc(b0 & lt_mask) + 2 * __popc(b1 & lt_mask);
                total_lines = __popc(b0) + 2 * __popc(b1);
            } else {
                int incl = my_cnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int tt = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += tt;
                }
                total_lines = __shfl_sync(0xffffffffu, incl, 31);
                my_first = incl - my_cnt;
            }
            // record slots for this chunk are taken from the warp's reserved block; make sure it can hold every line
            if (slot_left < (unsigned)total_lines) {
                unsigned long long got = 0ull;
                const unsigned want = total_lines > RESERVE ? (unsigned)total_lines : (unsigned)RESERVE;
                if (lane == 0) got = atomicAdd(&d_counters[MC_C_RECORDS], (unsigned long long)want);
                slot_cur = __shfl_sync(0xffffffffu, got, 0);
                slot_left = want;
            }
        }
        unsigned n_emitted = 0u;

        int e_last = -1;           // end of the chunk's last line (built with the field-start map)
        uint32_t filler = 0u;      // the chunk's first record exists only because its predecessor line is in another chunk
        for (int pass0 = 0; pass0 < total_lines; pass0 += 32) {
            // list entries [pass0, pass0+33) (one extra so every lane knows where its line ends)
            {
                int idx = my_first - pass0;
                uint32_t w0 = lsv.x, w1 = lsv.y, w2 = lsv.z, w3 = lsv.w;
                if (my_cnt <= 2) {
                    // usual case, no loops: at most two line starts inside this lane's 128 bytes
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        if (t < my_cnt) {
                            const int jw = w0 ? 0 : w1 ? 1 : w2 ? 2 : 3;
                            const uint32_t m = w0 ? w0 : w1 ? w1 : w2 ? w2 : w3;
                            if (idx >= 0 && idx <= 32) S.lstart[idx] = (uint16_t)(32 * (4 * lane + jw) + __ffs(m) - 1);
                            ++idx;
                            const uint32_t cl = m & (m - 1u);
                            if (jw == 0) w0 = cl; else if (jw == 1) w1 = cl; else if (jw == 2) w2 = cl; else w3 = cl;
                        }
                    }
                } else {
                    const uint32_t wv[4] = {w0, w1, w2, w3};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint32_t m = wv[j];
                        while (m) {
                            const int b = __ffs(m) - 1;
                            m &= m - 1u;
                            if (idx >= 0 && idx <= 32) S.lstart[idx] = (uint16_t)(32 * (4 * lane + j) + b);
                            ++idx;
                        }
                    }
                }
            }
            __syncwarp();
            const int n_pass = min(32, total_lines - pass0);
            // ---- 3. full parse: field-start map of the chunk (once), then one lane per line -------------------------------
            if (!full_ready) {
                full_ready = true;
                uint32_t prev_top = 0u;                               // was the last byte of word 32r-1 non-whitespace
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int w = 32 * r + lane;
                    const uint4 va = *reinterpret_cast<const uint4 *>(text + 32 * w);
                    const uint4 vb = *reinterpret_cast<const uint4 *>(text + 32 * w + 16);
                    const uint32_t nonws = pack32(gt20_msb(va.x), gt20_msb(va.y), gt20_msb(va.z), gt20_msb(va.w), gt20_msb(vb.x),
                                                  gt20_msb(vb.y), gt20_msb(vb.z), gt20_msb(vb.w));
                    // top bit of the previous word: lane-1 of this round, or lane 31 of the previous round for lane 0
                    const uint32_t top = nonws >> 31;
                    uint32_t pt = __shfl_up_sync(0xffffffffu, top, 1);
                    if (lane == 0) pt = prev_top;
                    prev_top = __shfl_sync(0xffffffffu, top, 31);
                    S.fs[w] = nonws & ~((nonws << 1) | pt);
                }
                if (lane < 8) S.fs[NW + lane] = 0u;
                // end of the chunk's last line = first newline at or after the last owned byte; found by the lanes that hold
                // the look-ahead words instead of a single lane walking the bit map
                if (!tail) {
                    constexpr int WLAST = (LOOKB + CHUNK - 1) >> 5, BLAST = (LOOKB + CHUNK - 1) & 31;
                    static_assert(NW - WLAST <= 32, "look-ahead words must fit one per lane");
                    int cand_e = NW * 32;
                    if (WLAST + lane < NW) {
                        uint32_t m = S.nl[WLAST + lane];
                        if (lane == 0) m &= 0xFFFFFFFFu << BLAST;
                        if (m) cand_e = 32 * (WLAST + lane) + __ffs(m) - 1;
                    }
                    e_last = __reduce_min_sync(0xffffffffu, cand_e);
                }                  // else the text ends inside this chunk: e_last stays -1, the bit-map walk finds the end
                __syncwarp();
            }
            uint32_t status = 0u;
            int cid = -1, pos = 0, s = 0;
            bool staged = false;       // first 12 columns inside the staged bytes (else: classified from global memory)
            int f3 = 0;                // RF: where column 4 (the read name) starts
            if (lane < n_pass) {
                s = S.lstart[lane];
                const int e = (pass0 + lane + 1 < total_lines) ? (int)S.lstart[lane + 1] - 1 : (e_last >= 0 ? e_last : next_bit(S.nl, s));
                // columns 1, 2, 10, 12 from a 160-bit window of the field-start bits aligned at the line start
                int f0, f1, f9, f11;
                line_fields<RF>(S, s, f0, f1, f9, f11, f3);
                if (f11 < e) {
                    staged = true;
                    // contig: compare the first bytes with the warp's hint in registers, full lookup on a miss
                    const unsigned long long k8 = load8(text, f0);
                    // names of up to 7 bytes compare in registers: the name bytes and the whitespace right after them
                    const bool hit = hint_nlen <= 7 && (k8 & ((1ull << (8 * hint_nlen)) - 1ull)) == hint_key &&
                                     ((k8 >> (8 * hint_nlen)) & 0xFFull) <= 0x20ull;
                    // model_kmer == 'NNNNNN' (:167): first byte in the common case, one 8-byte register compare otherwise
                    int nnn = 0;
                    if (text[f9] == 'N') {
                        const unsigned long long m8 = load8(text, f9);
                        nnn = ((m8 & 0xFFFFFFFFFFFFull) == 0x4E4E4E4E4E4Eull && ((m8 >> 48) & 0xFFull) <= 0x20ull) ? 1 : 0;
                    }
                    const int pst = parse_pos8(load8(text, f1), pos);
                    status = classify_line(T, f0, f1, f9, R, hint, hint_base, hint_len, hit ? hint : -1, nnn, pst, cid, pos);
                } else if (e >= NW * 32 || f11 >= NW * 32) {
                    status = classify_from_global(d_text, nbytes + MC_TEXT_PAD - 64, G0 + s, R, hint, hint_base, hint_len, cid, pos);
                    atomicAdd(&S.cnt[4], 1u);
                } else {
                    status = ST_SHORT;
                }
            }
            if (status & (ST_SHORT | ST_UNKNOWN | ST_NNN | ST_BADPOS))
                atomicAdd(&S.cnt[(status & ST_SHORT) ? 0 : (status & ST_UNKNOWN) ? 1 : (status & ST_NNN) ? 2 : 3], 1u);

            // ---- 4. which lines matter: ballots over the 32 lines of this pass -----------------------------------------
            const uint32_t kept_m = __ballot_sync(0xffffffffu, (status & ST_KEPT) != 0u);
            c_kept += (unsigned)__popc(kept_m);
            const uint32_t cand_m = __ballot_sync(0xffffffffu, (status & ST_CAND) != 0u);
            bool emit = false, filler_lane = false;
            if (RF) {
                // read name of every line of the pass against the line before it (bytes of column 4; anything unusual -- a
                // line parsed from global memory, fewer than 4 columns, a name of more than 64 bytes -- counts as a change)
                // usual case: every line of the pass carries the name the warp already holds (one cooperative compare)
                const bool valid = lane < n_pass;
                const uint32_t unusual = __ballot_sync(0xffffffffu, valid && !staged);
                uint32_t new_m = 0u;
                if (unusual != 0u || rname_len < 1 || !rf_all_match(text, valid ? f3 : -1)) {
                int nq = 0, nlen = -1;
                if (valid && staged) {
                    nq = f3;
                    nlen = token_len64(text, nq);
                    if (nlen == 0) nlen = -1;
                }
                const int pq = __shfl_up_sync(0xffffffffu, nq, 1), plen = __shfl_up_sync(0xffffffffu, nlen, 1);
                bool same = false;
                if (valid && nlen > 0) {
                    if (lane == 0) same = nlen == rname_len && token_is(text, nq, nlen, S.rname);
                    else same = nlen == plen && spans_equal(text, nq, pq, nlen);
                }
                const uint32_t pass_m = n_pass >= 32 ? 0xFFFFFFFFu : ((1u << n_pass) - 1u);
                new_m = __ballot_sync(0xffffffffu, !same) & pass_m;
                // the name of the pass's last line is what the next line is compared with
                const int lq = __shfl_sync(0xffffffffu, nq, n_pass - 1), llen = __shfl_sync(0xffffffffu, nlen, n_pass - 1);
                __syncwarp();
                if (llen > 0 && lane < 8) S.rname[lane] = 8 * lane < llen ? low_bytes(load8(text, lq + 8 * lane), llen - 8 * lane) : 0ull;
                rname_len = (llen > 0 && llen <= 63) ? llen : -1;          // (the cooperative compare covers 63 bytes + the byte that ends the name)
                __syncwarp();
                }
                if (status & ST_KEPT) {
                    const uint32_t nle = new_m & ((2u << lane) - 1u);           // read changes at or before this line
                    bool had;
                    if (nle == 0u) had = read_has_kept || (kept_m & lt_mask) != 0u;
                    else had = (kept_m & lt_mask & ~((1u << (31 - __clz(nle))) - 1u)) != 0u;
                    if (!had) emit = true;                                      // first kept line of its read
                }
                if (new_m == 0u) read_has_kept = read_has_kept || kept_m != 0u;
                else read_has_kept = (kept_m >> (31 - __clz(new_m))) != 0u;
            }
            if (status & ST_KEPT) {
                if (dense || (status & ST_CAND)) emit = true;
                else {
                    const uint32_t below = kept_m & lt_mask;
                    const int st = below ? (int)((cand_m >> (31 - __clz(below))) & 1u) : prev_state;
                    if (st != 0) emit = true;    // predecessor is a candidate, or this is the first kept line of the run
                    if (st < 0 && !RF) filler_lane = true;       // (RF: stage 2 keeps it, it may be the first kept line of its read)
                }
            }
            const uint32_t emit_m = __ballot_sync(0xffffffffu, emit);
            if (__ballot_sync(0xffffffffu, filler_lane)) filler = 1u;
            if (kept_m) {
                const int top = 31 - __clz(kept_m);
                prev_state = (int)((cand_m >> top) & 1u);
                const int new_hint = __shfl_sync(0xffffffffu, cid, top);       // contig hint follows the last kept line
                if (new_hint != hint) set_hint(new_hint);
            }
            // ---- 5. raw records ------------------------------------------------------------------------------------------
            if (emit) {
                const unsigned long long slot = slot_cur + __popc(emit_m & lt_mask);
                if (slot < rec_cap) {
                    // raw record: line offset, position, contig, candidate flag and -- so that stage 2 need not walk the line
                    // again -- the first 128 field-start bits of the line (where its columns begin), parked in the fields
                    // stage 2 fills in: event_idx, diff, name_off, name_len.  pad bit 1: no window (line classified from
                    // global memory).
                    uint32_t fl = MC_RF_RAW | ((status & ST_CAND) ? MC_RF_CAND : 0u);
                    uint32_t W0 = 0u, W1 = 0u, W2 = 0u, W3 = 0u;
                    if (staged) {
                        const int w0 = s >> 5, sh = s & 31;
                        const uint32_t a0 = S.fs[w0], a1 = S.fs[w0 + 1], a2 = S.fs[w0 + 2], a3 = S.fs[w0 + 3], a4 = S.fs[w0 + 4];
                        W0 = __funnelshift_r(a0, a1, sh);
                        W1 = __funnelshift_r(a1, a2, sh);
                        W2 = __funnelshift_r(a2, a3, sh);
                        W3 = __funnelshift_r(a3, a4, sh);
                    } else {
                        fl |= 2u << 24;
                    }
                    const int64_t goff = G0 + s;
                    uint4 a, b;
                    a.x = (uint32_t)(goff & 0xFFFFFFFFll);                              // line_lo
                    a.y = ((uint32_t)(goff >> 32) & 0xFFFFu) | (W3 << 16);              // line_hi | window bits 96..111
                    a.z = (uint32_t)pos;                                                // pos
                    a.w = W0;                                                           // window bits 0..31
                    b.x = W1; b.y = W2;                                                 // window bits 32..95
                    b.z = (W3 >> 16) | ((uint32_t)cid << 16);                           // window bits 112..127 | contig
                    b.w = fl;                                                           // flags | kbits (stage 2) | pad
                    uint4 *dst = reinterpret_cast<uint4 *>(d_rec + slot);
                    dst[0] = a;
                    dst[1] = b;
                } else {
                    atomicAdd(&S.cnt[5], 1u);
                }
            }
            {
                const unsigned ne = (unsigned)__popc(emit_m);
                slot_cur += ne;
                slot_left -= ne;
                n_emitted += ne;
            }
            __syncwarp();
        }
        if (lane == 0) {
            // {first slot, count | filler flag | state of the last kept line so far in the run (0 none, 1 not a candidate,
            // 2 candidate)} as one 8-byte store
            reinterpret_cast<uint2 *>(d_tile_tab)[chunk] =
                make_uint2((uint32_t)(slot_cur - n_emitted), n_emitted | (filler << 16) | ((uint32_t)(prev_state + 1) << 17));
        }
        run_total += n_emitted;
        run_filler |= filler;
        if (last_of_run) {
            // per-run entry for stage 2 (which orders the records run by run): {records of the run, first record is a filler |
            // state of the run's last kept line (0 none, 1 not a candidate, 2 candidate) << 1}
            if (lane == 0) reinterpret_cast<uint2 *>(d_run_tab)[chunk / run_len] = make_uint2(run_total, run_filler | ((uint32_t)(prev_state + 1) << 1));
            run_total = 0u;
            run_filler = 0u;
            prev_state = -1;
            rname_len = -1;
            read_has_kept = false;
        }
        chunk = next;
        run_end = next_end;
        buf ^= 1;
        cur_async = next_async;
    }

    // ---- counters: one global atomic per warp and counter ------------------------------------------------------------------
    __syncwarp();
    c_lines = __reduce_add_sync(0xffffffffu, c_lines);
    if (lane == 0) {
        if (c_lines) atomicAdd(&d_counters[MC_C_LINES], (unsigned long long)c_lines);
        if (c_kept) atomicAdd(&d_counters[MC_C_KEPT], (unsigned long long)c_kept);
        if (S.cnt[6]) atomicAdd(&d_counters[MC_C_QUIET], (unsigned long long)S.cnt[6]);
    }
    if (lane < 6) {
        const int which = lane == 0 ? MC_C_SHORT : lane == 1 ? MC_C_UNKNOWN_CONTIG : lane == 2 ? MC_C_NNN : lane == 3 ? MC_C_BADPOS
                        : lane == 4 ? MC_C_LONGLINE : MC_C_OVERFLOW;
        const unsigned v = S.cnt[lane];
        if (v) atomicAdd(&d_counters[which], (unsigned long long)v);
    }
}

}  // namespace

static int g_run_len_override = 0;
extern "C" int mc_scan_set_run_len(int run_len) {
    const int before = g_run_len_override;
    g_run_len_override = run_len < 0 ? 0 : (run_len > 4096 ? 4096 : run_len);
    return before;
}

extern "C" int64_t mc_num_tiles(int64_t nbytes) { return nbytes <= 0 ? 0 : (nbytes + CHUNK - 1) / CHUNK; }

// persistent grid of mc_scan and the run length it uses for nbytes of text (stage 2 walks the same runs)
static int scan_geometry(int64_t n_chunks, int64_t *blocks_out, int *run_len_out) {
    int dev = 0, sms = 0;
    MC_CUDA_CHECK(cudaGetDevice(&dev));
    MC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    int64_t blocks = (n_chunks + WARPS - 1) / WARPS;
    const int64_t resident = (int64_t)sms * MC_SCAN_MIN_CTAS;     // persistent: MC_SCAN_MIN_CTAS CTAs per SM
    if (blocks > resident) blocks = resident;
    // run length: as long as possible (fewer run-first "filler" passes) while every warp still gets >= 8 runs to balance on
    int run_len = MC_SCAN_RUN;
    while (run_len > 1 && n_chunks < blocks * WARPS * 8 * (int64_t)run_len) run_len >>= 1;
    if (g_run_len_override > 0) run_len = g_run_len_override;
    *blocks_out = blocks;
    *run_len_out = run_len;
    return MC_OK;
}
extern "C" int mc_scan_run_len(int64_t nbytes) {
    const int64_t n_chunks = mc_num_tiles(nbytes);
    if (n_chunks == 0) return 1;
    int64_t blocks = 0;
    int run_len = 1;
    if (scan_geometry(n_chunks, &blocks, &run_len)) return -1;
    return run_len;
}

extern "C" int mc_scan(const uint8_t *d_text, int64_t nbytes, const mc_refindex *ref, int dense, mc_record *d_rec,
                       int64_t rec_cap, uint32_t *d_tile_tab, uint32_t *d_run_tab, uint64_t *d_counters, void *stream) {
    MC_REQUIRE(d_text && ref && d_rec && d_tile_tab && d_run_tab && d_counters, "null pointer");
    MC_REQUIRE(nbytes >= 0 && rec_cap >= 0, "negative size");
    MC_REQUIRE((reinterpret_cast<uintptr_t>(d_text) & 15) == 0, "d_text must be 16-byte aligned");
    MC_REQUIRE((reinterpret_cast<uintptr_t>(d_tile_tab) & 7) == 0, "d_tile_tab must be 8-byte aligned");
    MC_REQUIRE(ref->k >= 1 && ref->k <= MC_MAXK, "k out of range");
    MC_REQUIRE(ref->n_contigs >= 1 && ref->n_contigs < 65535, "contig count out of range");
    MC_REQUIRE(nbytes < (1ll << 47), "chunk too large");
    MC_REQUIRE(rec_cap < (1ll << 32), "record capacity must fit 32 bits");
    const int64_t n_chunks = mc_num_tiles(nbytes);
    if (n_chunks == 0) return MC_OK;
    MC_REQUIRE(n_chunks < (1ll << 30), "too many chunks (chunk of text larger than 4 TB)");
    const size_t smem = sizeof(WarpSmem) * WARPS;
    const bool read_first = dense == 2;                           // sparse + the first kept line of every read (-q)
    MC_CUDA_CHECK(cudaFuncSetAttribute(read_first ? k_scan<true> : k_scan<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t blocks = 0;
    int run_len = 1;
    {
        const int rc = scan_geometry(n_chunks, &blocks, &run_len);
        if (rc) return rc;
    }
    // 16-byte loads / bulk copies are allowed up to the end of the caller's '\n' padding
    const int64_t text_limit16 = ((nbytes + MC_TEXT_PAD) / 16) * 16;
    // the run cursor must start at zero whatever the caller did with the counter block
    MC_CUDA_CHECK(cudaMemsetAsync(d_counters + MC_C_RUN_CURSOR, 0, sizeof(uint64_t), (cudaStream_t)stream));
    if (read_first)
        k_scan<true><<<(unsigned)blocks, THREADS, smem, (cudaStream_t)stream>>>(d_text, nbytes, text_limit16, n_chunks, run_len, *ref, 0, d_rec,
                                                                               (unsigned long long)rec_cap, d_tile_tab, d_run_tab,
                                                                               reinterpret_cast<unsigned long long *>(d_counters));
    else
        k_scan<false><<<(unsigned)blocks, THREADS, smem, (cudaStream_t)stream>>>(d_text, nbytes, text_limit16, n_chunks, run_len, *ref, dense ? 1 : 0,
                                                                                d_rec, (unsigned long long)rec_cap, d_tile_tab, d_run_tab,
                                                                                reinterpret_cast<unsigned long long *>(d_counters));
    MC_LAUNCH_CHECK();
    return MC_OK;
}
