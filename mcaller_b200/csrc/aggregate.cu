// make_bed drop-in: per-position aggregation straight from a `.diffs.<k>` text file (make_bed.py:67-164).
// Rows are tab-split exactly like the reference (8 fields, or 7 for the old format); the locus key is
// (chrom, pos, context, strand); depth / methylated counts are integer atomics in an open-addressing table and the
// first-seen order of make_bed.py:134 is recovered from the smallest line offset per key.
//
// Variants that need per-read lists (SURVEY.md section 8f rank 3):
//   -p positions  (make_bed.py:73-74, :84, :115-127): rows are filtered through a hash set of (chrom, pos, strand) and the
//                 k current deviations of every surviving row feed one-sample t-tests per locus and column.  The device
//                 produces, per locus and column, numpy's pairwise mean and the pairwise sum of squared deviations
//                 (scipy.stats.ttest_1samp: mean, _moment(a, 2), both np.add.reduce); the host turns them into t and p.
//   --vo          (:96-97, :147-151, :158-159): a row index (locus slot, line offset, probability span) lets the host join
//                 the probability strings of each locus in file order.
// Decimal text -> float64 is exact (correctly rounded) for <= 19 significant digits and decimal exponents in [-27, 0]:
// m * 10^-p = (m / 5^p) * 2^-p with one 128-by-64-bit division rounded to nearest even.
#include "common.cuh"

namespace {

struct DiffsRow {
    int64_t end;                 // position of the terminating '\n' (or nbytes)
    int nf;                      // tab-separated fields
    int64_t f[9];                // field starts
};

// split on '\t' up to the newline (the newline stays outside the last field)
__device__ __forceinline__ void split_row(const uint8_t *__restrict__ text, int64_t nbytes, int64_t p, DiffsRow &r) {
    int nf = 0;
    r.f[0] = p;
    int64_t q = p;
    for (; q < nbytes; ++q) {
        const uint8_t c = __ldg(text + q);
        if (c == '\n') break;
        if (c == '\t') { ++nf; if (nf < 9) r.f[nf] = q + 1; }
    }
    r.nf = nf + 1;
    r.end = q;
}

__device__ __forceinline__ unsigned long long fnv_span(const uint8_t *__restrict__ text, int64_t a, int64_t b, unsigned long long h) {
    for (int64_t i = a; i < b; ++i) h = (h ^ __ldg(text + i)) * 1099511628211ull;
    return h;
}
__device__ __forceinline__ unsigned long long fnv_sep(unsigned long long h) { return (h ^ 9ull) * 1099511628211ull; }
// second, independent hash of the same bytes (other basis, other multiplier, extra shift-xor): stored next to the slot's key so
// that two different loci with the same 64-bit key are noticed instead of merged
__device__ __forceinline__ unsigned long long chk_span(const uint8_t *__restrict__ text, int64_t a, int64_t b, unsigned long long g) {
    for (int64_t i = a; i < b; ++i) {
        g = (g ^ __ldg(text + i)) * 0x9E3779B97F4A7C15ull;
        g ^= g >> 29;
    }
    return g;
}
__device__ __forceinline__ unsigned long long chk_sep(unsigned long long g) { return ((g ^ 9ull) * 0x9E3779B97F4A7C15ull) ^ (g >> 31); }

// 0 = use the row, 1 = malformed, 2 = centre of the context is not 'M' (:84), 3 = not in the positions set (:84)
__device__ __forceinline__ int classify_row(const uint8_t *__restrict__ text, int64_t nbytes, int64_t p, const unsigned long long *posset,
                                            unsigned long long posmask, DiffsRow &r, unsigned long long &h, unsigned long long *check = nullptr) {
    split_row(text, nbytes, p, r);
    if (r.nf != 8 && r.nf != 7) return 1;                        // reference: unpack error
    const int64_t c0 = r.f[0], c0e = r.f[1] - 1, p0 = r.f[2], p0e = r.f[3] - 1, x0 = r.f[3], x0e = r.f[4] - 1, s0 = r.f[5], s0e = r.f[6] - 1;
    if (posset) {
        // (csome, pos, str(int(pos)+1), strand) in pos_set: the host keeps only entries whose end column is start + 1
        unsigned long long k = fnv_span(text, c0, c0e, 14695981039346656037ull);
        k = fnv_span(text, p0, p0e, fnv_sep(k));
        k = fnv_span(text, s0, s0e, fnv_sep(k));
        if (k == 0ull) k = 1ull;
        bool found = false;
        unsigned long long slot = k & posmask;
        for (unsigned long long probe = 0; probe <= posmask; ++probe) {
            const unsigned long long cur = posset[slot];
            if (cur == k) { found = true; break; }
            if (cur == 0ull) break;
            slot = (slot + 1) & posmask;
        }
        if (!found) return 3;
    }
    const int64_t xl = x0e - x0;
    if (xl <= 0 || __ldg(text + x0 + xl / 2) != 'M') return 2;
    h = fnv_span(text, c0, c0e, 14695981039346656037ull);
    h = fnv_span(text, p0, p0e, fnv_sep(h));
    h = fnv_span(text, x0, x0e, fnv_sep(h));
    h = fnv_span(text, s0, s0e, fnv_sep(h));
    if (h == 0ull) h = 1ull;
    if (check) {
        unsigned long long g = chk_span(text, c0, c0e, 0x243F6A8885A308D3ull);
        g = chk_span(text, p0, p0e, chk_sep(g));
        g = chk_span(text, x0, x0e, chk_sep(g));
        g = chk_span(text, s0, s0e, chk_sep(g));
        *check = g ? g : 1ull;
    }
    return 0;
}

__global__ void __launch_bounds__(256)
k_diffs_aggregate(const uint8_t *__restrict__ text, int64_t nbytes, unsigned long long base_off, const unsigned long long *__restrict__ posset,
                  unsigned long long posmask, mc_locus_entry *__restrict__ table, unsigned long long mask,
                  unsigned long long *__restrict__ counters) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nbytes) return;
    if (p > 0 && __ldg(text + p - 1) != '\n') return;          // not a line start
    DiffsRow r;
    unsigned long long h = 0ull, chk = 0ull;
    const int st = classify_row(text, nbytes, p, posset, posmask, r, h, &chk);
    atomicAdd(&counters[0], 1ull);                               // lines
    if (st == 1) { atomicAdd(&counters[1], 1ull); return; }
    if (st == 2) { atomicAdd(&counters[2], 1ull); return; }
    if (st == 3) { atomicAdd(&counters[4], 1ull); return; }
    if (r.nf == 7) atomicAdd(&counters[5], 1ull);                // old-format rows (no probability column)
    const int64_t l0 = r.f[6];
    const bool is_m = (l0 < r.end || r.nf == 8) && __ldg(text + l0) == 'm';      // label[0] == 'm' (:93)
    unsigned long long slot = h & mask;
    for (unsigned long long probe = 0; probe <= mask; ++probe) {
        unsigned long long cur = table[slot].hash;
        if (cur == 0ull) {
            cur = atomicCAS(&table[slot].hash, 0ull, h);
            if (cur == 0ull) cur = h;
        }
        if (cur == h) {
            atomicAdd(&table[slot].depth, 1u);
            if (is_m) atomicAdd(&table[slot].meth, 1u);
            atomicMin(&table[slot].first_off, base_off + (unsigned long long)p);
            // the first row of a locus leaves its check hash; a later row with the same key but other bytes is a collision
            const unsigned long long seen = atomicCAS(&table[slot].check, 0ull, chk);
            if (seen != 0ull && seen != chk) atomicAdd(&counters[7], 1ull);
            return;
        }
        slot = (slot + 1) & mask;
    }
    atomicAdd(&counters[3], 1ull);                               // table full
}

// move every used entry of a table into a larger one (the file is streamed in pieces and the table grows with the loci seen)
__global__ void __launch_bounds__(256)
k_diffs_rehash(const mc_locus_entry *__restrict__ old_table, unsigned long long old_size, mc_locus_entry *__restrict__ table,
               unsigned long long mask, unsigned long long *__restrict__ counters) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= old_size) return;
    const mc_locus_entry e = old_table[i];
    if (e.hash == 0ull) return;
    unsigned long long slot = e.hash & mask;
    for (unsigned long long probe = 0; probe <= mask; ++probe) {
        const unsigned long long cur = atomicCAS(&table[slot].hash, 0ull, e.hash);
        if (cur == 0ull) {                                       // keys are distinct in the old table: the slot is ours
            table[slot].first_off = e.first_off;
            table[slot].check = e.check;
            table[slot].depth = e.depth;
            table[slot].meth = e.meth;
            return;
        }
        slot = (slot + 1) & mask;
    }
    atomicAdd(&counters[3], 1ull);
}

// second pass: one index entry per used row (any order; the host sorts by line offset)
__global__ void __launch_bounds__(256)
k_diffs_rows(const uint8_t *__restrict__ text, int64_t nbytes, const unsigned long long *__restrict__ posset, unsigned long long posmask,
             const mc_locus_entry *__restrict__ table, unsigned long long mask, mc_diffs_row *__restrict__ rows,
             unsigned long long row_cap, unsigned long long *__restrict__ d_nrows) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nbytes) return;
    if (p > 0 && __ldg(text + p - 1) != '\n') return;
    DiffsRow r;
    unsigned long long h = 0ull;
    if (classify_row(text, nbytes, p, posset, posmask, r, h) != 0) return;
    unsigned long long slot = h & mask;
    bool found = false;
    for (unsigned long long probe = 0; probe <= mask; ++probe) {
        const unsigned long long cur = table[slot].hash;
        if (cur == h) { found = true; break; }
        if (cur == 0ull) break;
        slot = (slot + 1) & mask;
    }
    if (!found) return;                                          // dropped by a full table in pass 1
    const unsigned long long idx = atomicAdd(d_nrows, 1ull);
    if (idx >= row_cap) return;
    mc_diffs_row o;
    o.line_off = (uint64_t)p;
    o.slot = (uint32_t)slot;
    o.values_off = (uint32_t)(r.f[4] - p);
    o.values_len = (uint32_t)(r.f[5] - 1 - r.f[4]);
    // prob.strip() (:97): the 8th field without surrounding whitespace; old-format rows have none
    int64_t a = r.nf == 8 ? r.f[7] : r.end, b = r.end;
    while (a < b && __ldg(text + a) <= 0x20) ++a;
    while (b > a && __ldg(text + b - 1) <= 0x20) --b;
    o.prob_off = (uint32_t)(a - p);
    o.prob_len = (uint32_t)(b - a);
    o.pad = 0u;
    rows[idx] = o;
}

// ---- exact decimal -> double ------------------------------------------------------------------------------------------
__constant__ unsigned long long c_pow5[28] = {1ull, 5ull, 25ull, 125ull, 625ull, 3125ull, 15625ull, 78125ull, 390625ull, 1953125ull,
    9765625ull, 48828125ull, 244140625ull, 1220703125ull, 6103515625ull, 30517578125ull, 152587890625ull, 762939453125ull,
    3814697265625ull, 19073486328125ull, 95367431640625ull, 476837158203125ull, 2384185791015625ull, 11920928955078125ull,
    59604644775390625ull, 298023223876953125ull, 1490116119384765625ull, 7450580596923828125ull};
__constant__ double c_p10[23] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17,
                                 1e18, 1e19, 1e20, 1e21, 1e22};

// m / 5^p * 2^-p, correctly rounded (m != 0, 0 <= p <= 27)
__device__ double div_pow5_exact(unsigned long long m, int p) {
    const unsigned long long d = c_pow5[p];
    const int lm = __clzll((long long)m), ld = __clzll((long long)d);
    const unsigned long long a = m << lm, b = d << ld;           // top bits set: a / b in (1/2, 2)
    unsigned long long hi, lo;
    int e2;                                                      // value = Q * 2^e2 with Q the 64-bit quotient below
    if (a >= b) { hi = a >> 1; lo = a << 63; e2 = -63; } else { hi = a; lo = 0ull; e2 = -64; }
    for (int i = 0; i < 64; ++i) {                               // restoring division of hi:lo by b (hi < b)
        const unsigned long long carry = hi >> 63;
        hi = (hi << 1) | (lo >> 63);
        lo <<= 1;
        if (carry || hi >= b) { hi -= b; lo |= 1ull; }
    }
    const unsigned long long Q = lo;                             // bit 63 set
    const bool sticky = hi != 0ull;
    unsigned long long mant = Q >> 11;
    const unsigned long long rb = Q & 0x7FFull;
    if (rb > 0x400ull || (rb == 0x400ull && (sticky || (mant & 1ull)))) ++mant;
    // m / d = (a / b) * 2^(ld - lm);  a / b = Q * 2^e2;  mant = Q / 2^11
    return ldexp((double)mant, e2 + 11 + ld - lm - p);           // (double)mant is exact (<= 2^53)
}

// Python float() of a feature token written by the .diffs writer: [+-] digits [. digits] [e[+-]digits] | nan | inf.
// Returns false when the token is something else (the reference's float() may still accept it; counted as unparsed).
__device__ bool parse_float_token(const uint8_t *__restrict__ text, int64_t a, int64_t b, double &out, bool &inexact) {
    inexact = false;
    while (a < b && __ldg(text + a) <= 0x20) ++a;
    while (b > a && __ldg(text + b - 1) <= 0x20) --b;
    if (a >= b) return false;
    bool neg = false;
    int c = __ldg(text + a);
    if (c == '-' || c == '+') { neg = c == '-'; ++a; if (a >= b) return false; }
    const int64_t n = b - a;
    auto lower = [&](int64_t i) { const int ch = __ldg(text + i); return (ch >= 'A' && ch <= 'Z') ? ch + 32 : ch; };
    if (n == 3 && lower(a) == 'n' && lower(a + 1) == 'a' && lower(a + 2) == 'n') { out = __longlong_as_double(0x7ff8000000000000ll); return true; }
    if ((n == 3 && lower(a) == 'i' && lower(a + 1) == 'n' && lower(a + 2) == 'f') ||
        (n == 8 && lower(a) == 'i' && lower(a + 1) == 'n' && lower(a + 2) == 'f' && lower(a + 3) == 'i' && lower(a + 4) == 'n' &&
         lower(a + 5) == 'i' && lower(a + 6) == 't' && lower(a + 7) == 'y')) {
        out = neg ? -__longlong_as_double(0x7ff0000000000000ll) : __longlong_as_double(0x7ff0000000000000ll);
        return true;
    }
    unsigned long long m = 0ull;
    int nd = 0, sig = 0, e10 = 0;
    bool lost = false;
    auto digit = [&](int d, bool frac) {
        ++nd;
        if (sig < 19) { m = m * 10ull + (unsigned)d; if (m) ++sig; if (frac) --e10; }
        else { if (d) lost = true; if (!frac) ++e10; }            // beyond 19 significant digits: truncated
    };
    int64_t q = a;
    while (q < b && (c = __ldg(text + q)) >= '0' && c <= '9') { digit(c - '0', false); ++q; }
    if (q < b && __ldg(text + q) == '.') {
        ++q;
        while (q < b && (c = __ldg(text + q)) >= '0' && c <= '9') { digit(c - '0', true); ++q; }
    }
    if (nd == 0) return false;
    if (q < b && ((c = __ldg(text + q)) == 'e' || c == 'E')) {
        ++q;
        bool eneg = false;
        if (q < b && ((c = __ldg(text + q)) == '-' || c == '+')) { eneg = c == '-'; ++q; }
        int ev = 0, ned = 0;
        while (q < b && (c = __ldg(text + q)) >= '0' && c <= '9') { if (ev < 100000) ev = ev * 10 + (c - '0'); ++ned; ++q; }
        if (ned == 0) return false;
        e10 += eneg ? -ev : ev;
    }
    if (q != b) return false;
    double v;
    if (m == 0ull) v = 0.0;
    else if (lost) { inexact = true; v = e10 < 0 ? ((double)m / (e10 >= -22 ? c_p10[-e10] : pow(10.0, (double)-e10))) : (double)m * pow(10.0, (double)e10); }
    else if (e10 == 0) v = __ull2double_rn(m);
    else if (e10 < 0 && e10 >= -27) v = div_pow5_exact(m, -e10);
    else if (e10 > 0 && e10 <= 19 && m <= 0xFFFFFFFFFFFFFFFFull / (unsigned long long)c_p10[e10]) v = __ull2double_rn(m * (unsigned long long)c_p10[e10]);
    else { inexact = true; v = e10 < 0 ? (double)m / pow(10.0, (double)-e10) : (double)m * pow(10.0, (double)e10); }
    out = neg ? -v : v;
    return true;
}

// [float(v) for v in values.split(',')][:-1] of one row (make_bed.py:91): thread per (sorted) row
__global__ void __launch_bounds__(256)
k_diffs_values(const uint8_t *__restrict__ text, const mc_diffs_row *__restrict__ rows, const uint32_t *__restrict__ order, int64_t n_rows,
               double *__restrict__ vals, uint32_t *__restrict__ ncol, unsigned long long *__restrict__ counters) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const mc_diffs_row r = rows[order[i]];
    const int64_t a = (int64_t)r.line_off + r.values_off, b = a + r.values_len;
    int nc = 0;
    int64_t t0 = a;
    double prev = 0.0;
    bool have_prev = false;
    for (int64_t q = a; q <= b; ++q) {
        if (q == b || __ldg(text + q) == ',') {
            double v = 0.0;
            bool inexact = false;
            if (!parse_float_token(text, t0, q, v, inexact)) { atomicAdd(&counters[6], 1ull); v = __longlong_as_double(0x7ff8000000000000ll); }
            if (inexact) atomicAdd(&counters[7], 1ull);
            if (have_prev) {                                     // the previous token was not the last one: keep it
                if (nc < MC_MAXK + 1) vals[i * (MC_MAXK + 1) + nc] = prev;
                ++nc;
            }
            prev = v;
            have_prev = true;
            t0 = q + 1;
        }
    }
    ncol[i] = (uint32_t)nc;
}

// per locus (CSR over the sorted rows) and column: n, np.mean(x), np.add.reduce((x - mean)**2)
__global__ void __launch_bounds__(128)
k_diffs_colstats(const double *__restrict__ vals, const uint32_t *__restrict__ ncol, const uint32_t *__restrict__ locus_off, int64_t n_loci,
                 int ncols, double *__restrict__ stats) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_loci * ncols) return;
    const int64_t l = t / ncols;
    const int c = (int)(t % ncols);
    const int64_t r0 = locus_off[l], n = (int64_t)locus_off[l + 1] - r0;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    auto x = [&](int64_t i) { return c < (int)ncol[i] ? vals[i * (MC_MAXK + 1) + c] : nan; };   // ragged rows: pandas fills NaN
    const double mean = __ddiv_rn(mc_pairwise_sum(x, r0, n), (double)n);
    auto sq = [&](int64_t i) { const double d = __dsub_rn(x(i), mean); return __dmul_rn(d, d); };
    const double ss = mc_pairwise_sum(sq, r0, n);
    stats[2 * t] = mean;
    stats[2 * t + 1] = ss;
}

}  // namespace

static int check_sets(const void *d_posset, int64_t posset_size, int64_t table_size) {
    MC_REQUIRE(table_size > 0 && (table_size & (table_size - 1)) == 0, "table size must be a power of two");
    MC_REQUIRE(!d_posset || (posset_size > 0 && (posset_size & (posset_size - 1)) == 0), "positions set size must be a power of two");
    return MC_OK;
}

extern "C" int mc_diffs_aggregate_ex(const uint8_t *d_text, int64_t nbytes, int64_t base_off, const uint64_t *d_posset,
                                     int64_t posset_size, mc_locus_entry *d_table, int64_t table_size, uint64_t *d_counters,
                                     void *stream) {
    MC_REQUIRE(d_text && d_table && d_counters, "null pointer");
    MC_REQUIRE(base_off >= 0, "negative base offset");
    int rc = check_sets(d_posset, posset_size, table_size);
    if (rc) return rc;
    if (nbytes <= 0) return MC_OK;
    k_diffs_aggregate<<<(unsigned)((nbytes + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_text, nbytes, (unsigned long long)base_off, reinterpret_cast<const unsigned long long *>(d_posset),
        (unsigned long long)(d_posset ? posset_size - 1 : 0), d_table, (unsigned long long)(table_size - 1),
        reinterpret_cast<unsigned long long *>(d_counters));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_diffs_rehash(const mc_locus_entry *d_old, int64_t old_size, mc_locus_entry *d_table, int64_t table_size,
                               uint64_t *d_counters, void *stream) {
    MC_REQUIRE(d_old && d_table && d_counters, "null pointer");
    MC_REQUIRE(table_size > 0 && (table_size & (table_size - 1)) == 0, "table size must be a power of two");
    if (old_size <= 0) return MC_OK;
    k_diffs_rehash<<<(unsigned)((old_size + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_old, (unsigned long long)old_size, d_table, (unsigned long long)(table_size - 1), reinterpret_cast<unsigned long long *>(d_counters));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_diffs_rows(const uint8_t *d_text, int64_t nbytes, const uint64_t *d_posset, int64_t posset_size,
                             const mc_locus_entry *d_table, int64_t table_size, mc_diffs_row *d_rows, int64_t row_cap, uint64_t *d_nrows,
                             void *stream) {
    MC_REQUIRE(d_text && d_table && d_rows && d_nrows, "null pointer");
    MC_REQUIRE(row_cap >= 0, "negative capacity");
    int rc = check_sets(d_posset, posset_size, table_size);
    if (rc) return rc;
    MC_REQUIRE(nbytes < (1ll << 32) * 64, "file too large");
    if (nbytes <= 0) return MC_OK;
    k_diffs_rows<<<(unsigned)((nbytes + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_text, nbytes, reinterpret_cast<const unsigned long long *>(d_posset), (unsigned long long)(d_posset ? posset_size - 1 : 0), d_table,
        (unsigned long long)(table_size - 1), d_rows, (unsigned long long)row_cap, reinterpret_cast<unsigned long long *>(d_nrows));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_diffs_colstats(const uint8_t *d_text, const mc_diffs_row *d_rows, const uint32_t *d_order, int64_t n_rows,
                                 const uint32_t *d_locus_off, int64_t n_loci, int ncols, double *d_vals, uint32_t *d_ncol,
                                 double *d_stats, uint64_t *d_counters, void *stream) {
    MC_REQUIRE(d_text && d_rows && d_order && d_locus_off && d_vals && d_ncol && d_stats && d_counters, "null pointer");
    MC_REQUIRE(ncols >= 1 && ncols <= MC_MAXK + 1, "column count out of range");
    if (n_rows <= 0 || n_loci <= 0) return MC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    k_diffs_values<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(d_text, d_rows, d_order, n_rows, d_vals, d_ncol,
                                                                     reinterpret_cast<unsigned long long *>(d_counters));
    MC_LAUNCH_CHECK();
    const int64_t nt = n_loci * ncols;
    k_diffs_colstats<<<(unsigned)((nt + 127) / 128), 128, 0, st>>>(d_vals, d_ncol, d_locus_off, n_loci, ncols, d_stats);
    MC_LAUNCH_CHECK();
    return MC_OK;
}
