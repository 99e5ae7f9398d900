// Byte-level parsing helpers shared by the scan kernel (shared-memory bytes) and the record finishing kernel
// (global-memory bytes): contig-name compare, integer / exact-decimal parsing, NNNNNN test.
#pragma once
#include "common.cuh"

__constant__ double c_pow10[23] = {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11,
                                   1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};

// ---- byte sources: warp-private shared memory (fast path) or global memory (slow path) ---------------------------------
struct SmemBytes {
    const uint8_t *p;
    __device__ __forceinline__ int operator[](int i) const { return p[i]; }
};
struct GlobalBytes {
    const uint8_t *p;
    int64_t limit;     // bytes readable from p
    __device__ __forceinline__ int operator[](int64_t i) const { return i < limit ? __ldg(p + i) : 0x0a; }
};

template <class B>
__device__ __forceinline__ bool contig_match(const B &t, int q, const mc_refindex &R, int cid) {
    const int o0 = __ldg(R.d_name_off + cid), L = __ldg(R.d_name_off + cid + 1) - o0;
    for (int j = 0; j < L; ++j)
        if (t[q + j] != __ldg(R.d_names + o0 + j)) return false;
    return t[q + L] <= 0x20;
}
template <class B>
__device__ __forceinline__ int contig_cmp(const B &t, int q, const mc_refindex &R, int cid) {
    const int o0 = __ldg(R.d_name_off + cid), L = __ldg(R.d_name_off + cid + 1) - o0;
    for (int j = 0; j < L; ++j) {
        const int a = t[q + j], b = __ldg(R.d_names + o0 + j);
        if (a <= 0x20) return -1;
        if (a != b) return a - b;
    }
    return t[q + L] <= 0x20 ? 0 : 1;
}
// contigs are sorted by name on the host: hint first, then binary search
template <class B>
__device__ __forceinline__ int contig_lookup(const B &t, int q, const mc_refindex &R, int hint) {
    if (contig_match(t, q, R, hint)) return hint;
    int lo = 0, hi = R.n_contigs - 1;
    while (lo <= hi) {
        const int mid = (lo + hi) >> 1;
        const int c = contig_cmp(t, q, R, mid);
        if (c == 0) return mid;
        if (c < 0) hi = mid - 1; else lo = mid + 1;
    }
    return -1;
}
template <class B>
__device__ __forceinline__ bool parse_uint(const B &t, int q, int &out) {
    int v = 0, nd = 0, c;
    while ((c = t[q]) >= '0' && c <= '9') { v = v * 10 + (c - '0'); ++nd; ++q; if (nd > 9) return false; }
    if (nd == 0 || c > 0x20) return false;
    out = v;
    return true;
}
template <class B>
__device__ __forceinline__ bool parse_int(const B &t, int q, int &out) {
    bool neg = false;
    if (t[q] == '-') { neg = true; ++q; } else if (t[q] == '+') ++q;
    int v;
    if (!parse_uint(t, q, v)) return false;
    out = neg ? -v : v;
    return true;
}
// plain decimal -> correctly rounded double (mantissa <= 2^53, <= 18 digits: one exact division)
template <class B>
__device__ __forceinline__ bool parse_decimal(const B &t, int q, double &out) {
    bool neg = false;
    int c = t[q];
    if (c == '-') { neg = true; ++q; } else if (c == '+') ++q;
    unsigned long long m = 0;
    int nd = 0, nfrac = 0;
    while ((c = t[q]) >= '0' && c <= '9') { m = m * 10ull + (unsigned)(c - '0'); ++nd; ++q; if (nd > 18) return false; }
    if (c == '.') {
        ++q;
        while ((c = t[q]) >= '0' && c <= '9') { m = m * 10ull + (unsigned)(c - '0'); ++nd; ++nfrac; ++q; if (nd > 18) return false; }
    }
    if (nd == 0 || c > 0x20 || m > (1ull << 53)) return false;
    const double v = __ddiv_rn((double)m, c_pow10[nfrac]);
    out = neg ? -v : v;
    return true;
}
template <class B>
__device__ __forceinline__ bool is_nnnnnn(const B &t, int q) {
    if (t[q] != 'N') return false;
    return t[q + 1] == 'N' && t[q + 2] == 'N' && t[q + 3] == 'N' && t[q + 4] == 'N' && t[q + 5] == 'N' && t[q + 6] <= 0x20;
}


// reference_kmer (col 3) == model_kmer (col 10): token compare up to the first whitespace on either side
template <class B>
__device__ __forceinline__ bool tokens_equal(const B &t, int64_t a, int64_t b) {
    for (;;) {
        const int ca = t[a++], cb = t[b++];
        const bool ea = ca <= 0x20, eb = cb <= 0x20;
        if (ea || eb) return ea && eb;
        if (ca != cb) return false;
    }
}

// event index, np.round(event_mean - model_mean, 4) and the k-mer equality flag of one line (extract_contexts.py:150,
// :169, :286); f5/f6/f2/f9/f10 are byte offsets of the columns from the start of `t`
template <class B>
__device__ __forceinline__ void parse_values(const B &t, int f2, int f5, int f6, int f9, int f10, int &event_idx, double &diff,
                                             uint32_t &flags) {
    event_idx = 0;
    if (!parse_int(t, f5, event_idx)) flags |= MC_RF_BADIDX;
    double ev = 0.0, md = 0.0;
    if (!parse_decimal(t, f6, ev) || !parse_decimal(t, f10, md)) { flags |= MC_RF_BADNUM; diff = 0.0; }
    else diff = __ddiv_rn(rint(__dmul_rn(__dsub_rn(ev, md), 1e4)), 1e4);
    if (tokens_equal(t, f2, f9)) flags |= MC_RF_EQ;
}

// ---- byte and bit helpers in registers -------------------------------------------------------------------------------------
// 0x80 per byte of w that is > 0x20 (not whitespace)
__device__ __forceinline__ uint32_t gt20_msb(uint32_t w) { return (((w & 0x7f7f7f7fu) + 0x5f5f5f5fu) | w) & 0x80808080u; }
// 4 msb-form words (0x80 per flagged byte) -> 16 flag bits in byte order.  IDP.4A sums 0x80 * weight per byte: two words
// fill bits 7..14 of one accumulator.
__device__ __forceinline__ uint32_t pack16(uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
    const uint32_t lo = 0x08040201u, hi = 0x80402010u;
    const uint32_t a = __dp4a(m1, hi, __dp4a(m0, lo, 0u)), b = __dp4a(m3, hi, __dp4a(m2, lo, 0u));
    return (a >> 7) | (b << 1);
}
// position of the j-th (0-based) set bit of m, j < popc(m)
__device__ __forceinline__ int nth_bit(uint32_t m, int j) {
#pragma unroll
    for (int t = 0; t < 6; ++t)
        if (j > t) m &= m - 1u;
    for (int t = 6; t < j; ++t) m &= m - 1u;                     // words with more than 7 set bits: rare
    return __ffs(m) - 1;
}
// 4 digit values, most significant in byte 0 -> 0..9999
__device__ __forceinline__ uint32_t conv4(uint32_t h) {
    const uint32_t t = ((h * 2561u) >> 8) & 0x00ff00ffu;
    return (t * 6553601u) >> 16;
}

// ---- 8-byte register fast paths for the values of a record (any other shape falls back to the byte loops of parse.cuh) ----
// 0x80 per byte of v that is not an ASCII digit
__device__ __forceinline__ unsigned long long nondigit8(unsigned long long v) {
    const unsigned long long x = v ^ 0x3030303030303030ull;
    return (((x & 0x7f7f7f7f7f7f7f7full) + 0x7676767676767676ull) | v) & 0x8080808080808080ull;
}
// n (1..7) digit bytes at the low end of v -> value
__device__ __forceinline__ uint32_t digits_value(unsigned long long v, int n) {
    const unsigned long long x = (v ^ 0x3030303030303030ull) << (64 - 8 * n);      // right-aligned digit values, zeros below
    return conv4((uint32_t)x) * 10000u + conv4((uint32_t)(x >> 32));
}
// "<1..7 digits><ws>" -> value; false for any other shape
__device__ __forceinline__ bool fast_uint8(unsigned long long v, int &out) {
    const unsigned long long nd = nondigit8(v);
    if (nd == 0ull) return false;
    const int n = (__ffsll((long long)nd) - 1) >> 3;
    if (n == 0 || ((v >> (8 * n)) & 0xFFull) > 0x20ull) return false;
    out = (int)digits_value(v, n);
    return true;
}
// "<digits>.<digits><ws>" with at most 7 bytes before the whitespace -> mantissa and number of fraction digits
__device__ __forceinline__ bool fast_decimal8(unsigned long long v, uint32_t &mant, int &nfrac) {
    const unsigned long long nd = nondigit8(v);
    if (nd == 0ull) return false;
    const int p1 = (__ffsll((long long)nd) - 1) >> 3;             // first non-digit: must be the point
    if (p1 == 0 || p1 > 6 || ((v >> (8 * p1)) & 0xFFull) != 0x2eull) return false;
    const unsigned long long low = (1ull << (8 * p1)) - 1ull;
    const unsigned long long w = (v & low) | ((v >> 8) & ~low);    // the point removed: 7 bytes
    const unsigned long long nd2 = ((nd & low) | ((nd >> 8) & ~low)) & 0x0080808080808080ull;
    if (nd2 == 0ull) return false;
    const int p2 = (__ffsll((long long)nd2) - 1) >> 3;            // first non-digit after it: must be whitespace
    if (((w >> (8 * p2)) & 0xFFull) > 0x20ull) return false;
    mant = digits_value(w, p2);
    nfrac = p2 - p1;
    return true;
}
// token at pa == token at pb for tokens of up to 7 bytes: 1 / 0, or -1 when one of them is longer (byte loop decides)
__device__ __forceinline__ int fast_tokens_equal8(unsigned long long a, unsigned long long b) {
    auto ws8 = [](unsigned long long v) {                          // 0x80 per byte <= 0x20
        return ~((((v & 0x7f7f7f7f7f7f7f7full) + 0x5f5f5f5f5f5f5f5full) | v)) & 0x8080808080808080ull;
    };
    const unsigned long long wa = ws8(a), wb = ws8(b);
    if (wa == 0ull || wb == 0ull) return -1;
    const int la = (__ffsll((long long)wa) - 1) >> 3, lb = (__ffsll((long long)wb) - 1) >> 3;
    if (la != lb) return 0;
    return (((a ^ b) & ((1ull << (8 * la)) - 1ull)) == 0ull) ? 1 : 0;
}

// ---- finishing a raw record of stage 1 from the text in global memory (stage 2) ----------------------------------------------
// 8 bytes at any alignment from two aligned 8-byte loads
__device__ __forceinline__ unsigned long long load8_unaligned(const uint8_t *p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const unsigned long long *q = reinterpret_cast<const unsigned long long *>(a & ~(uintptr_t)7);
    const int sh = 8 * (int)(a & 7);
    const unsigned long long lo = __ldg(q);
    if (sh == 0) return lo;
    const unsigned long long hi = __ldg(q + 1);
    return (lo >> sh) | (hi << (64 - sh));
}
// do the L bytes at pa and pb differ (the '\n' padding after the text keeps the 8-byte loads legal).  Both sides are
// streamed as aligned 8-byte words and realigned in registers: 1 + ceil(L / 8) loads per side, all independent.
__device__ __forceinline__ bool bytes_differ(const uint8_t *pa, const uint8_t *pb, int L) {
    const uintptr_t ua = reinterpret_cast<uintptr_t>(pa), ub = reinterpret_cast<uintptr_t>(pb);
    const unsigned long long *qa = reinterpret_cast<const unsigned long long *>(ua & ~(uintptr_t)7);
    const unsigned long long *qb = reinterpret_cast<const unsigned long long *>(ub & ~(uintptr_t)7);
    const int sa = 8 * (int)(ua & 7), sb = 8 * (int)(ub & 7);
    unsigned long long a_lo = __ldg(qa), b_lo = __ldg(qb), diff = 0ull;
#pragma unroll 5
    for (int j = 0; j < L; j += 8) {
        const unsigned long long a_hi = __ldg(++qa), b_hi = __ldg(++qb);
        const unsigned long long va = sa ? ((a_lo >> sa) | (a_hi << (64 - sa))) : a_lo;
        const unsigned long long vb = sb ? ((b_lo >> sb) | (b_hi << (64 - sb))) : b_lo;
        unsigned long long d = va ^ vb;
        if (L - j < 8) d &= (1ull << (8 * (L - j))) - 1ull;               // 1..7 tail bytes
        diff |= d;
        a_lo = a_hi;
        b_lo = b_hi;
    }
    return diff != 0ull;
}

// Event index (column 6), np.round(event_mean - model_mean, 4) (7, 11) and the k-mer equality flag (3 vs 10) of the line
// at lp, of which `room` bytes are readable; f2..f10 are the line offsets of those columns.  The usual shapes ("1234",
// "87.41", 6-mers) are decoded from 8-byte register loads, anything else by the byte loops of parse_values -- both give
// the same float64.
__device__ __forceinline__ void mc_finish_values(const uint8_t *lp, int64_t room, int f2, int f5, int f6, int f9, int f10, int &ev_idx,
                                                 double &diff, uint32_t &fl) {
    uint32_t m_ev = 0u, m_md = 0u;
    int n_ev = 0, n_md = 0;
    const int teq = fast_tokens_equal8(load8_unaligned(lp + f2), load8_unaligned(lp + f9));
    if (f10 + 16 < room && teq >= 0 && fast_uint8(load8_unaligned(lp + f5), ev_idx) &&
        fast_decimal8(load8_unaligned(lp + f6), m_ev, n_ev) && fast_decimal8(load8_unaligned(lp + f10), m_md, n_md)) {
        const double ev = __ddiv_rn((double)m_ev, c_pow10[n_ev]), md = __ddiv_rn((double)m_md, c_pow10[n_md]);
        diff = __ddiv_rn(rint(__dmul_rn(__dsub_rn(ev, md), 1e4)), 1e4);
        if (teq) fl |= MC_RF_EQ;
    } else {
        parse_values(GlobalBytes{lp, room}, f2, f5, f6, f9, f10, ev_idx, diff, fl);
    }
}

// Walks the columns of the record's line in the text (16-byte SWAR steps over the non-whitespace map; columns split on
// runs of bytes <= 0x20 like str.split(), extract_contexts.py:150) and parses what the window builder needs: read-name span
// (column 4) and the values of mc_finish_values.  Clears MC_RF_RAW.
__device__ __forceinline__ void mc_finish_record(const uint8_t *__restrict__ text, int64_t limit, mc_record &r) {
    const int64_t line = mc_rec_line(r);
    // 16-byte steps from the aligned address at or below the line start; the '\n' padding after the text makes every
    // line end inside readable memory
    const int64_t a0 = line & ~15ll;
    const int skip = (int)(line - a0);
    int nf = 0, f2 = 0, f3 = 0, name_end = -1, f5 = 0, f6 = 0, f9 = 0, f10 = 0;
    uint32_t prev_nonws = 0u;          // was the byte before this step non-whitespace (the byte before the line is '\n')
    bool done = false;
    constexpr int MAX_STEPS = 256;     // 4 KB: twice the documented limit for the first 12 columns of a line
    for (int step = 0; step < MAX_STEPS && !done; ++step) {
        const int64_t g = a0 + 16ll * step;
        if (g >= limit) break;
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(text + g));
        uint32_t nonws = pack16(gt20_msb(v.x), gt20_msb(v.y), gt20_msb(v.z), gt20_msb(v.w));
        if (step == 0) nonws &= 0xFFFFu << skip;                 // ignore the bytes before the line start
        // no newline test: a recorded line is a kept line, its first 12 columns start before its end (stage 1 checked), so
        // the walk stops at the 11th column; MAX_STEPS bounds it for records that did not come from stage 1
        const int base = 16 * step - skip;                       // line-relative offset of byte 0 of this step
        uint32_t fs = nonws & ~((nonws << 1) | prev_nonws);
        if (name_end < 0 && nf >= 4) {                           // first whitespace (or the newline) after the read name
            const uint32_t z = ~nonws & 0xFFFFu & ((step == 0) ? (0xFFFFu << skip) : 0xFFFFu);
            const uint32_t zz = z & ~((1u << max(f3 - base, 0)) - 1u);
            if (zz) name_end = base + __ffs(zz) - 1;
        }
        while (fs) {
            const int b = __ffs(fs) - 1;
            fs &= fs - 1u;
            const int pos = base + b;
            switch (nf) {
                case 2: f2 = pos; break;
                case 3: f3 = pos; break;
                case 5: f5 = pos; break;
                case 6: f6 = pos; break;
                case 9: f9 = pos; break;
                case 10: f10 = pos; break;
                default: break;
            }
            ++nf;
            if (nf == 4 && name_end < 0) {                       // the name may end inside this same step
                const uint32_t z = ~nonws & 0xFFFFu & ~((1u << b) - 1u);
                if (z) name_end = base + __ffs(z) - 1;
            }
            if (nf == 11) { done = true; break; }
        }
        prev_nonws = (nonws >> 15) & 1u;
    }
    uint32_t fl = r.flags & ~MC_RF_RAW;
    int ev_idx = 0;
    double diff = 0.0;
    if (nf < 11 || name_end < 0 || f3 > 65535 || name_end - f3 > 65535) fl |= MC_RF_BADNUM | MC_RF_BADIDX;   // cannot happen for a kept line
    else mc_finish_values(text + line, limit - line, f2, f5, f6, f9, f10, ev_idx, diff, fl);
    r.name_off = (uint16_t)f3;
    r.name_len = (uint16_t)(name_end < 0 ? 0 : name_end - f3);
    r.event_idx = ev_idx;
    r.diff = diff;
    r.flags = (uint8_t)fl;
}

// Stage 1 parks the first 128 field-start bits of the recorded line (bit b: a column starts at line offset b) in the
// raw record's event_idx / diff / name_off / name_len fields (pad bit 1: none).  With them the columns are located by
// rank/select and only the bytes of the needed tokens are read: columns 3, 6, 7, 10, 11 and the end of the read name.
// Falls back to the walk above when a needed column starts beyond the window.
__device__ __forceinline__ void mc_finish_record_win(const uint8_t *__restrict__ text, int64_t limit, mc_record &r) {
    const uint32_t *rw = reinterpret_cast<const uint32_t *>(&r);
    const uint32_t W0 = rw[3], W1 = rw[4], W2 = rw[5], W3 = (rw[1] >> 16) | (rw[6] << 16);
    const int c0 = __popc(W0), c1 = c0 + __popc(W1), c2 = c1 + __popc(W2), c3 = c2 + __popc(W3);
    const int64_t line = mc_rec_line(r);
    if ((r.pad & 2u) || c3 < 11 || line + 160 >= limit) {            // no window / column 11 beyond it: walk the line
        r.pad = 0;
        mc_finish_record(text, limit, r);
        return;
    }
    // columns start where the window has a set bit; they are needed in order, so walk the bits once: lowest set bit, clear
    // it, move to the next word when the current one is used up
    uint32_t m = W0;
    int wi = 0;
    auto next = [&]() {
        while (m == 0u && wi < 3) {
            ++wi;
            m = wi == 1 ? W1 : wi == 2 ? W2 : W3;
        }
        const int q = 32 * wi + __ffs(m) - 1;
        m &= m - 1u;
        return q;
    };
    next();                                                          // column 1 (contig)
    next();                                                          // column 2 (position)
    const int f2 = next(), f3 = next(), f4 = next(), f5 = next(), f6 = next();
    next();                                                          // column 8 (event_stdv)
    next();                                                          // column 9 (event_length)
    const int f9 = next(), f10 = next();
    const uint8_t *lp = text + line;
    // end of the read name: the bytes before column 5 are whitespace; step back over them (one tab in nanopolish output)
    // (the 8 bytes before column 5 in one load that does not depend on the others; a byte loop for anything unusual)
    int name_end;
    {
        const unsigned long long t8 = f4 >= 8 ? load8_unaligned(lp + f4 - 8) : 0ull;
        const uint32_t nh = gt20_msb((uint32_t)(t8 >> 32)), nlw = gt20_msb((uint32_t)t8);     // 0x80 per non-whitespace byte
        const int tw = nh ? (__clz(nh) >> 3) : nlw ? 4 + (__clz(nlw) >> 3) : 8;               // whitespace bytes right before column 5
        name_end = f4 - tw;
        if (tw == 8 || name_end <= f3) {
            name_end = f4 - 1;
            while (name_end > f3 && __ldg(lp + name_end - 1) <= 0x20) --name_end;
        }
    }
    uint32_t fl = r.flags & ~MC_RF_RAW;
    int ev_idx = 0;
    double diff = 0.0;
    mc_finish_values(lp, limit - line, f2, f5, f6, f9, f10, ev_idx, diff, fl);
    r.name_off = (uint16_t)f3;
    r.name_len = (uint16_t)(name_end - f3);
    r.event_idx = ev_idx;
    r.diff = diff;
    r.flags = (uint8_t)fl;
    r.pad = 0;
}
