// Shared helpers for libmcaller_b200 (sm_100a).  Device code only sees plain structs of device pointers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/mcaller_b200.h"

void mc_set_error(const char *fmt, ...);

#define MC_CUDA_CHECK(expr)                                                                  \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            mc_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return MC_ECUDA;                                                                 \
        }                                                                                    \
    } while (0)

#define MC_LAUNCH_CHECK() MC_CUDA_CHECK(cudaGetLastError())

#define MC_REQUIRE(cond, msg)                       \
    do {                                            \
        if (!(cond)) {                              \
            mc_set_error("%s: %s", __func__, msg);  \
            return MC_EINVAL;                       \
        }                                           \
    } while (0)

// ---- k-mer bit window over a site bitmap: bits [g, g+k) of the bitmap, LSB = position g ---------------
__device__ __forceinline__ uint32_t mc_kmer_bits(const uint32_t *__restrict__ bm, int64_t g, int k) {
    int64_t w = g >> 5;
    int b = (int)(g & 31);
    uint32_t lo = __ldg(bm + w), hi = __ldg(bm + w + 1);
    uint32_t v = __funnelshift_r(lo, hi, b);
    return v & ((1u << k) - 1u);
}

// ---- block-wide exclusive scan of one int per thread (blockDim.x <= 1024, multiple of 32) -------------
template <int THREADS>
__device__ __forceinline__ int mc_block_exscan(int v, int *s_warp /* [THREADS/32 + 1] */, int &total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int x = (lane < THREADS / 32) ? s_warp[lane] : 0;
        int xi = x;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, xi, d);
            if (lane >= d) xi += t;
        }
        if (lane < THREADS / 32) s_warp[lane] = xi - x;
        if (lane == 31) s_warp[THREADS / 32] = xi;
    }
    __syncthreads();
    total = s_warp[THREADS / 32];
    int res = s_warp[wid] + inc - v;
    __syncthreads();
    return res;
}

// device exclusive scan (uint32 in -> uint32 out, records.cu) of n_cap items, or of the first *d_n of them when the count
// lives on the device (items beyond it count as zero); d_total (may be null) receives the sum
int mc_exscan_u32(const uint32_t *d_in, uint32_t *d_out, int64_t n_cap, const uint64_t *d_n /* may be null */,
                  uint64_t *d_total /* may be null */, void *d_ws, cudaStream_t st);
int64_t mc_exscan_ws_bytes(int64_t n);

// item count kept on the device (stage outputs), clamped to the capacity the launch was sized for
__device__ __forceinline__ int64_t mc_dev_count(const unsigned long long *d_n, int64_t cap) {
    const unsigned long long v = *d_n;
    return v < (unsigned long long)cap ? (int64_t)v : cap;
}

// byte offset of a record's line in the text
__device__ __forceinline__ int64_t mc_rec_line(const mc_record &r) { return ((int64_t)r.line_hi << 32) | (int64_t)r.line_lo; }

// Read-quality key of a read name: name.split(':')[0].split('_')[0] (read_qual.py:11-12 / extract_contexts.py:166), the
// bytes at p up to whitespace, ':' or '_' (at most max_len of them), hashed by FNV-1a with two bases.  The fastq ingest
// (k_fq_insert) builds its table and stage 4 (k_seg_quality) probes it with this one function; the host twin is
// read_qual.fnv_pair.
struct mc_read_key {
    unsigned long long hash;   // never 0 (0 marks an empty table slot)
    uint32_t check;            // high word of the second hash
    uint32_t len;
};
__device__ __forceinline__ mc_read_key mc_read_key_of(const uint8_t *p, int64_t max_len) {
    unsigned long long h = 14695981039346656037ull, h2 = 0x84222325cbf29ce4ull;
    int64_t len = 0;
    for (; len < max_len; ++len) {
        const unsigned c = __ldg(p + len);
        if (c <= 0x20u || c == ':' || c == '_') break;
        h = (h ^ c) * 1099511628211ull;
        h2 = (h2 ^ c) * 1099511628211ull;
    }
    return {h == 0ull ? 1ull : h, (uint32_t)(h2 >> 32), (uint32_t)len};
}

// numpy's pairwise summation (np.add.reduce over a contiguous float64 vector) of f(x_i), i in [i0, i0 + n):
// sequential below 8 values, 8 running lanes + sequential tail up to 128, and above that numpy splits at n/2 rounded down
// to a multiple of 8 and adds the two halves.  The halving is walked with an explicit stack (depth <= log2(n / 64)) instead
// of device-side recursion, whose frames would need more than the default 1 KB of stack for a few thousand values.
template <class F>
__device__ __forceinline__ double mc_pairwise_block(F f, int64_t i0, int64_t n) {
    if (n < 8) {
        double res = 0.0;
        for (int64_t i = 0; i < n; ++i) res = __dadd_rn(res, f(i0 + i));
        return res;
    }
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = f(i0 + j);
    int64_t i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], f(i0 + i + j));
    }
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, f(i0 + i));
    return res;
}
template <class F>
__device__ double mc_pairwise_sum(F f, int64_t i0, int64_t n) {
    if (n <= 128) return mc_pairwise_block(f, i0, n);
    constexpr int DEPTH = 40;
    int64_t st_i0[DEPTH], st_n[DEPTH];
    double st_left[DEPTH];
    int st_phase[DEPTH];                      // 0: nothing done, 1: left half running, 2: right half running
    int sp = 0;
    st_i0[0] = i0; st_n[0] = n; st_phase[0] = 0; st_left[0] = 0.0;
    double ret = 0.0;
    for (;;) {
        if (st_phase[sp] == 0) {
            if (st_n[sp] <= 128 || sp + 1 >= DEPTH) {          // leaf (the depth bound cannot bind for n < 2^40)
                ret = mc_pairwise_block(f, st_i0[sp], st_n[sp]);
            } else {
                int64_t n2 = st_n[sp] / 2;
                n2 -= n2 % 8;
                st_phase[sp] = 1;
                st_i0[sp + 1] = st_i0[sp]; st_n[sp + 1] = n2; st_phase[sp + 1] = 0;
                ++sp;
                continue;
            }
        }
        // `ret` holds the sum of the frame at sp: hand it to the parent
        for (;;) {
            if (sp == 0) return ret;
            --sp;
            if (st_phase[sp] == 1) {                             // left half done: run the right half
                int64_t n2 = st_n[sp] / 2;
                n2 -= n2 % 8;
                st_left[sp] = ret;
                st_phase[sp] = 2;
                st_i0[sp + 1] = st_i0[sp] + n2; st_n[sp + 1] = st_n[sp] - n2; st_phase[sp + 1] = 0;
                ++sp;
                break;
            }
            ret = __dadd_rn(st_left[sp], ret);                   // both halves done
        }
    }
}

// ---- float64 activations of scikit-learn's MLPClassifier (classify.cu inference, train.cu fitting) ----------------
// scipy.special.expit, the logistic output
__device__ __forceinline__ double mc_expit(double x) { return x < 0.0 ? exp(x) / (1.0 + exp(x)) : 1.0 / (1.0 + exp(-x)); }

// tanh(x) = sign(x) (1 - t) / (1 + t), t = exp(-2|x|), without branches: n = rint(y log2 e), r = y - n ln 2 (two-step), exp(r) by
// its degree-13 Taylor polynomial on |r| <= ln2 / 2 (remainder < 5e-18), 2^n through the exponent field.  Absolute error
// ~2e-16 -- the hidden activations feed a dot product whose result only has to match scikit-learn's float64 to 1e-12 --
// at a third of the instructions of the library routine and with every lane on the same path (the float64 tanh was 55 % of
// k_mlp_1hidden's instructions at 14 of 32 lanes active).
__device__ __forceinline__ double mc_tanh(double x) {
    double y = -2.0 * fabs(x);
    y = fmax(y, -80.0);                                        // t < 2e-35: the quotient is 1 to the last bit
    const double n = rint(y * 1.4426950408889634074);
    double r = fma(n, -6.93147180369123816490e-01, y);
    r = fma(n, -1.90821492927058770002e-10, r);
    double p = 1.6059043836821613e-10;                         // 1/13!
    p = fma(p, r, 2.0876756987868100e-09);                     // 1/12!
    p = fma(p, r, 2.5052108385441720e-08);                     // 1/11!
    p = fma(p, r, 2.7557319223985890e-07);                     // 1/10!
    p = fma(p, r, 2.7557319223985893e-06);                     // 1/9!
    p = fma(p, r, 2.4801587301587302e-05);                     // 1/8!
    p = fma(p, r, 1.9841269841269841e-04);                     // 1/7!
    p = fma(p, r, 1.3888888888888889e-03);                     // 1/6!
    p = fma(p, r, 8.3333333333333332e-03);                     // 1/5!
    p = fma(p, r, 4.1666666666666664e-02);                     // 1/4!
    p = fma(p, r, 1.6666666666666666e-01);                     // 1/3!
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    const double t = p * __longlong_as_double((long long)(1023 + (int)n) << 52);
    // (1 - t) / (1 + t) without the division routine: 1 + t lies in [1, 2], a single-precision reciprocal is refined by two
    // Newton steps (24 -> 48 -> 96 bits) and the quotient gets one residual correction (<= 1 ulp)
    const double d = 1.0 + t, u = 1.0 - t;
    double rc = (double)__frcp_rn((float)d);
    double e = fma(-d, rc, 1.0);
    rc = fma(rc, e, rc);
    e = fma(-d, rc, 1.0);
    rc = fma(rc, e, rc);
    double q = u * rc;
    q = fma(fma(-d, q, u), rc, q);
    return copysign(q, x);
}
