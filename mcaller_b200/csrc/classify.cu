// Stage 6 (K3): per-observation classifier -- model[key].predict_proba([x])[0][1] and the 0.5 label threshold of
// the reference (extract_contexts.py:195-207) for the estimator types mCaller can be run with (-c NN/RF/LR/NBC;
// the estimator type is whatever the pickle holds, mCaller.py:137, SURVEY.md section 5).
//
// Arithmetic is float64 like scikit-learn's.  The work per call is ~1.6 kFLOP (MLP 7-100-1) and there is one call
// per ~85 KB of TSV, so this stage is <1 % of the step; the layer widths (K=7, N=100) would leave a tcgen05 tile
// >90 % padding and bf16/tf32 operands cannot meet the 1e-5 probability tolerance, so the MLP runs on the FP64
// FMA pipe: one warp per call, lanes over hidden units, weights served from L1/L2 (7 KB per model).
#include "common.cuh"

namespace {

constexpr int MAX_WIDTH = 512;     // widest MLP layer supported
constexpr int WARPS = 8;

__device__ __forceinline__ double activate(double v, int act) {
    switch (act) {
        case MC_ACT_TANH: return mc_tanh(v);
        case MC_ACT_LOGISTIC: return mc_expit(v);
        case MC_ACT_RELU: return v > 0.0 ? v : 0.0;
        default: return v;
    }
}

// sklearn MLPClassifier._forward_pass_fast (neural_network/_multilayer_perceptron.py) for a binary classifier:
// hidden activations, logistic output, P(class 1) = mc_expit(z).
// Persistent warps: a block stages the weights and intercepts of both models in shared memory once (7-100-1: 7.2 KB per
// model) and its warps then stride over the calls, so the inner loops read nothing but shared memory; the features of a
// warp's next call are fetched while the current one is evaluated.  STAGED = false (models too wide for shared memory)
// reads the weights through the read-only cache instead.
template <bool STAGED>
__global__ void __launch_bounds__(WARPS * 32)
k_mlp(mc_call *__restrict__ calls, int64_t n_cap, const unsigned long long *__restrict__ d_n, mc_model m0, mc_model m1, int width, int nw0,
      int nb0, int nw1, int nb1, int alias) {
    extern __shared__ __align__(16) double s_mlp[];          // [weights 0][biases 0][weights 1][biases 1][WARPS][2][width]
    const int64_t n = mc_dev_count(d_n, n_cap);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *s_act = s_mlp;
    if (STAGED) {
        for (int j = threadIdx.x; j < nw0; j += WARPS * 32) s_mlp[j] = __ldg(m0.d_weights + j);
        for (int j = threadIdx.x; j < nb0; j += WARPS * 32) s_mlp[nw0 + j] = __ldg(m0.d_biases + j);
        for (int j = threadIdx.x; j < nw1; j += WARPS * 32) s_mlp[nw0 + nb0 + j] = __ldg(m1.d_weights + j);
        for (int j = threadIdx.x; j < nb1; j += WARPS * 32) s_mlp[nw0 + nb0 + nw1 + j] = __ldg(m1.d_biases + j);
        s_act = s_mlp + nw0 + nb0 + nw1 + nb1;
        __syncthreads();
    }
    double *a = s_act + (size_t)warp * 2 * width, *b = a + width;
    const int64_t stride = (int64_t)gridDim.x * WARPS;
    int64_t i = (int64_t)blockIdx.x * WARPS + warp;
    // features (and row kind / model selector) of the call the warp handles next
    auto fetch = [&](int64_t idx, double &f, int &kind_sel) {
        f = 0.0;
        kind_sel = -1;
        if (idx < n) {
            const mc_call &c = calls[idx];
            kind_sel = c.kind == MC_CALL ? (int)c.model_sel : -1;
            if (lane <= MC_MAXK) f = c.feat[lane];
        }
    };
    double f_cur;
    int ks_cur;
    fetch(i, f_cur, ks_cur);
    for (; i < n; i += stride) {
        double f_next;
        int ks_next;
        fetch(i + stride, f_next, ks_next);
        if (ks_cur >= 0) {
            const mc_model &m = ks_cur ? m1 : m0;
            // model 1 follows model 0 in shared memory unless both selectors name the same model (alias)
            const double *w = STAGED ? ((ks_cur && !alias) ? s_mlp + nw0 + nb0 : s_mlp) : m.d_weights;
            const double *bi = STAGED ? ((ks_cur && !alias) ? s_mlp + nw0 + nb0 + nw1 : s_mlp + nw0) : m.d_biases;
            auto ld = [&](const double *p) { return STAGED ? *p : __ldg(p); };
            double *x = a, *y = b;
            if (lane < m.sizes[0]) x[lane] = f_cur;
            __syncwarp();
            for (int l = 0; l < m.n_layers; ++l) {
                const int ni = m.sizes[l], no = m.sizes[l + 1];
                const bool last = (l + 1 == m.n_layers);
                if (no >= 8) {
                    // four outputs per lane at a time: independent FMA / activation chains interleave and hide each other's latency
                    for (int o0 = 0; o0 < no; o0 += 128) {
                        double acc[4];
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc[j] = 0.0;
                        for (int k = 0; k < ni; ++k) {
                            const double ak = x[k];
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const int o = o0 + lane + 32 * j;
                                if (o < no) acc[j] = fma(ak, ld(w + (size_t)k * no + o), acc[j]);
                            }
                        }
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int o = o0 + lane + 32 * j;
                            if (o < no) {
                                const double z = acc[j] + ld(bi + o);          // dot product first, then the intercept (as sklearn)
                                y[o] = last ? z : activate(z, m.hidden_act);
                            }
                        }
                    }
                } else {
                    for (int o = 0; o < no; ++o) {
                        double acc = 0.0;
                        for (int k = lane; k < ni; k += 32) acc = fma(x[k], ld(w + (size_t)k * no + o), acc);
                        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
                        acc += ld(bi + o);
                        if (lane == 0) y[o] = last ? acc : activate(acc, m.hidden_act);
                    }
                }
                __syncwarp();
                double *t = x; x = y; y = t;
                w += (size_t)ni * no;
                bi += no;
            }
            const double out = mc_expit(x[0]);
            __syncwarp();
            if (lane == 0) {
                mc_call &c = calls[i];
                c.prob = out;
                c.label = (uint8_t)(out >= 0.5);
            }
        }
        f_cur = f_next;
        ks_cur = ks_next;
    }
}

// The shape every shipped pickle has -- one hidden layer, at most 9 inputs (k + 1 <= 9), one logistic output -- four lanes
// per call (eight calls per warp): a lane keeps its call's features in registers and owns every fourth hidden unit, so the
// activation (float64 tanh: ~80 % of the instructions) is evaluated 25 times per lane for 8 calls instead of 4 times for
// one, nothing passes through shared memory but the staged weights, and the output dot product is finished with two
// shuffles.  Same arithmetic as k_mlp: dot product in input order, then the intercept, activation, logistic output.
constexpr int MLP_MAX_IN = MC_MAXK + 1;

// rows that need a probability (kind MC_CALL) -> dense index list, so the classifier kernels run with every lane busy
// (rows of other kinds -- too-many-skips and multi-M events, empty slots -- are ~30 % of the rows for GATC)
__global__ void __launch_bounds__(256) k_call_index(const mc_call *__restrict__ calls, int64_t n_cap, const unsigned long long *__restrict__ d_n,
                                                   uint32_t *__restrict__ idx, unsigned long long *__restrict__ d_nidx) {
    __shared__ unsigned int s_warp[8];
    __shared__ unsigned long long s_base;
    const int64_t n = mc_dev_count(d_n, n_cap);
    if ((int64_t)blockIdx.x * blockDim.x >= n) return;       // block-uniform
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool is_call = i < n && calls[i].kind == MC_CALL;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t m = __ballot_sync(0xffffffffu, is_call);
    if (lane == 0) s_warp[wid] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int tot = 0u;
        for (int w = 0; w < 8; ++w) { const unsigned int c = s_warp[w]; s_warp[w] = tot; tot += c; }
        s_base = tot ? atomicAdd(d_nidx, (unsigned long long)tot) : 0ull;
    }
    __syncthreads();
    if (is_call) idx[s_base + s_warp[wid] + __popc(m & ((1u << lane) - 1u))] = (uint32_t)i;
}
__global__ void __launch_bounds__(WARPS * 32)
k_mlp_1hidden(mc_call *__restrict__ calls, const uint32_t *__restrict__ idx, const unsigned long long *__restrict__ d_nidx, mc_model m0,
              mc_model m1, int nw0, int nb0, int nw1, int nb1, int alias) {
    extern __shared__ __align__(16) double s_mlp[];          // [weights 0][biases 0][weights 1][biases 1]
    const int64_t n = (int64_t)*d_nidx;                      // call rows in the index list
    if ((int64_t)blockIdx.x * WARPS * 8 >= n) return;        // nothing for this block: skip staging the weights
    for (int j = threadIdx.x; j < nw0; j += WARPS * 32) s_mlp[j] = __ldg(m0.d_weights + j);
    for (int j = threadIdx.x; j < nb0; j += WARPS * 32) s_mlp[nw0 + j] = __ldg(m0.d_biases + j);
    for (int j = threadIdx.x; j < nw1; j += WARPS * 32) s_mlp[nw0 + nb0 + j] = __ldg(m1.d_weights + j);
    for (int j = threadIdx.x; j < nb1; j += WARPS * 32) s_mlp[nw0 + nb0 + nw1 + j] = __ldg(m1.d_biases + j);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane & 3, grp = lane >> 2;
    const int64_t stride = (int64_t)gridDim.x * WARPS * 8;
    for (int64_t base = ((int64_t)blockIdx.x * WARPS + warp) * 8; base < n; base += stride) {      // warp-uniform
        int64_t i = base + grp;
        int ks = -1;
        double x[MLP_MAX_IN];
#pragma unroll
        for (int k = 0; k < MLP_MAX_IN; ++k) x[k] = 0.0;
        if (i < n) {
            i = (int64_t)__ldg(idx + i);
            const mc_call &c = calls[i];
            ks = (int)c.model_sel;
#pragma unroll
            for (int k = 0; k < MLP_MAX_IN; ++k) x[k] = c.feat[k];
        }
        const bool second = ks > 0;
        const mc_model &m = second ? m1 : m0;
        const int ni = m.sizes[0], H = m.sizes[1], act = m.hidden_act;
        const double *w0 = (second && !alias) ? s_mlp + nw0 + nb0 : s_mlp;
        const double *b0 = (second && !alias) ? s_mlp + nw0 + nb0 + nw1 : s_mlp + nw0;
        const double *w1 = w0 + (size_t)ni * H, *b1 = b0 + H;
        double out = 0.0;
        if (ks >= 0) {
            for (int o0 = g; o0 < H; o0 += 16) {              // four hidden units per lane at a time: independent chains
                double z[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) z[j] = 0.0;
#pragma unroll
                for (int k = 0; k < MLP_MAX_IN; ++k) {
                    if (k < ni) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const int o = o0 + 4 * j;
                            if (o < H) z[j] = fma(x[k], w0[(size_t)k * H + o], z[j]);
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int o = o0 + 4 * j;
                    if (o < H) out = fma(act == MC_ACT_TANH ? mc_tanh(z[j] + b0[o]) : activate(z[j] + b0[o], act), w1[o], out);   // dot product first, then the intercept
                }
            }
        }
        out += __shfl_xor_sync(0xffffffffu, out, 1);
        out += __shfl_xor_sync(0xffffffffu, out, 2);
        if (ks >= 0 && g == 0) {
            const double p = mc_expit(out + b1[0]);
            mc_call &c = calls[i];
            c.prob = p;
            c.label = (uint8_t)(p >= 0.5);
        }
    }
}

// LogisticRegression.predict_proba (binary): mc_expit(x.w + b); GaussianNB.predict_proba: exp(jll_1 - logsumexp(jll))
__global__ void __launch_bounds__(256) k_linear(mc_call *__restrict__ calls, int64_t n_cap, const unsigned long long *__restrict__ d_n,
                                               mc_model m0, mc_model m1) {
    const int64_t n = mc_dev_count(d_n, n_cap);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    mc_call &c = calls[i];
    if (c.kind != MC_CALL) return;
    const mc_model &m = c.model_sel ? m1 : m0;
    double p;
    if (m.kind == MC_LR) {
        double z = __ldg(m.d_biases);
        for (int k = 0; k < m.n_in; ++k) z += c.feat[k] * __ldg(m.d_weights + k);
        p = mc_expit(z);
    } else {
        const double *theta = m.d_weights, *var = m.d_weights + 2 * m.n_in;
        double jll[2];
        for (int cl = 0; cl < 2; ++cl) {
            double nij = 0.0, s = 0.0;
            for (int k = 0; k < m.n_in; ++k) nij += log(2.0 * 3.14159265358979323846 * __ldg(var + cl * m.n_in + k));
            nij *= -0.5;
            for (int k = 0; k < m.n_in; ++k) {
                const double d = c.feat[k] - __ldg(theta + cl * m.n_in + k);
                s += d * d / __ldg(var + cl * m.n_in + k);
            }
            jll[cl] = __ldg(m.d_biases + cl) + nij - 0.5 * s;
        }
        const double mx = jll[0] > jll[1] ? jll[0] : jll[1];
        const double lse = mx + log(exp(jll[0] - mx) + exp(jll[1] - mx));
        p = exp(jll[1] - lse);
    }
    c.prob = p;
    c.label = (uint8_t)(p >= 0.5);
}

// RandomForestClassifier.predict_proba: mean over trees of the leaf class-1 fraction; the walk compares float32(x)
// with the float64 threshold (sklearn tree/_tree.pyx).  A block owns 256 calls and streams the trees through shared
// memory (node table of one tree at a time), so every node read in the walk is an smem read.
__global__ void __launch_bounds__(256)
k_rf(mc_call *__restrict__ calls, int64_t n_cap, const unsigned long long *__restrict__ d_n, mc_model m0, mc_model m1, int max_nodes) {
    extern __shared__ __align__(16) uint8_t rf_smem[];
    const int64_t n = mc_dev_count(d_n, n_cap);
    if ((int64_t)blockIdx.x * blockDim.x >= n) return;       // block-uniform
    double *s_thr = reinterpret_cast<double *>(rf_smem);
    double *s_p1 = s_thr + max_nodes;
    int32_t *s_left = reinterpret_cast<int32_t *>(s_p1 + max_nodes);
    int32_t *s_right = s_left + max_nodes;
    int32_t *s_feat = s_right + max_nodes;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n && calls[i].kind == MC_CALL;
    float x[MC_MAXK + 1];
    int sel = 0;
    if (active) {
        sel = calls[i].model_sel;
        for (int k = 0; k <= MC_MAXK; ++k) x[k] = (float)calls[i].feat[k];
    }
    double acc = 0.0;
    for (int pass = 0; pass < 2; ++pass) {
        const mc_model &m = pass ? m1 : m0;
        // skip a model nobody in the block uses
        const int any = __syncthreads_or(active && sel == pass);
        if (!any || m.n_trees == 0) continue;
        for (int t = 0; t < m.n_trees; ++t) {
            const int o0 = __ldg(m.d_tree_off + t), nn = __ldg(m.d_tree_off + t + 1) - o0;
            __syncthreads();
            for (int j = threadIdx.x; j < nn; j += blockDim.x) {
                s_thr[j] = __ldg(m.d_threshold + o0 + j);
                s_p1[j] = __ldg(m.d_leaf_p1 + o0 + j);
                s_left[j] = __ldg(m.d_left + o0 + j);
                s_right[j] = __ldg(m.d_right + o0 + j);
                s_feat[j] = __ldg(m.d_feature + o0 + j);
            }
            __syncthreads();
            if (active && sel == pass) {
                int node = 0;
                while (s_left[node] >= 0) node = ((double)x[s_feat[node]] <= s_thr[node]) ? s_left[node] : s_right[node];
                acc += s_p1[node];
            }
        }
    }
    if (active) {
        const mc_model &m = sel ? m1 : m0;
        const double p = acc / (double)m.n_trees;
        calls[i].prob = p;
        calls[i].label = (uint8_t)(p >= 0.5);
    }
}

// ---- stage 7 (K4): per-site histogram (make_bed.py:86-96) ----------------------------------------------------------
__global__ void __launch_bounds__(256)
k_hist(const mc_call *__restrict__ calls, int64_t n_cap, const unsigned long long *__restrict__ d_n, uint32_t *__restrict__ depth,
       uint32_t *__restrict__ meth, unsigned long long *__restrict__ first, int64_t n_sites, const unsigned long long *__restrict__ d_row_base,
       mc_call *__restrict__ d_odd, unsigned long long odd_cap, unsigned long long *__restrict__ d_n_odd,
       const unsigned long long *__restrict__ d_abort) {
    if (d_abort && *d_abort) return;                          // a buffer overflowed earlier in this chunk: the host redoes it
    const int64_t n = mc_dev_count(d_n, n_cap);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const mc_call &c = calls[i];
    if (c.kind != MC_CALL || c.close_rec == 0xFFFFFFFFu || c.err) return;     // other kinds, pending rows, error rows (the host raises)
    const unsigned long long row = *d_row_base + (unsigned long long)i;
    if (c.chrom_contig != c.win_contig || c.site < 0 || c.site >= n_sites) {
        // column 1 names another contig than the site's (reference quirk, :216): keyed by the host
        const unsigned long long slot = atomicAdd(d_n_odd, 1ull);
        if (slot < odd_cap) {
            mc_call o = c;
            o.pad1 = (uint32_t)(row & 0xFFFFFFFFull);
            o.pad2 = (uint32_t)(row >> 32);
            d_odd[slot] = o;
        }
        return;
    }
    atomicAdd(depth + c.site, 1u);
    if (c.label) atomicAdd(meth + c.site, 1u);
    atomicMin(first + c.site, row);
}
__global__ void k_advance_base(unsigned long long *d_row_base, const unsigned long long *d_n, const unsigned long long *d_abort) {
    if (d_abort && *d_abort) return;
    *d_row_base += *d_n;
}
// any overflow of the chunk's buffers so far -> d_abort[0] = 1 (the stages that change state across chunks then do nothing)
__global__ void k_chunk_guard(const unsigned long long *__restrict__ counters, unsigned long long rec_cap,
                              const unsigned long long *__restrict__ d_n_records, unsigned long long rec_out_cap,
                              const unsigned long long *__restrict__ d_nseg, unsigned long long seg_cap,
                              const unsigned long long *__restrict__ d_ncalls, unsigned long long call_cap,
                              unsigned long long *__restrict__ d_abort, unsigned long long *__restrict__ d_sticky) {
    const bool bad = counters[MC_C_OVERFLOW] != 0ull || counters[MC_C_RECORDS] > rec_cap || *d_n_records > rec_out_cap ||
                     *d_nseg > seg_cap || d_ncalls[0] > call_cap || d_ncalls[1] != 0ull;
    *d_abort = bad ? 1ull : 0ull;
    if (bad && d_sticky) *d_sticky = 1ull;                        // survives the next chunk's status reset (deferred status reads)
}

// row statistics without a D2H copy of the rows: [0] calls closed in this chunk, [1] calls still pending,
// [2] too-many-skips events closed in this chunk, [3] multi-M events, [4] rows with an error flag, [5] calls labelled
// methylated, [6] too-many-skips events still pending (a window open at the end of the chunk is closed -- and only then
// counted, extract_contexts.py:179/:238 -- by the next kept line of the file; the last one of a file never is)
__global__ void __launch_bounds__(256) k_count_calls(const mc_call *__restrict__ calls, int64_t n_cap, const unsigned long long *__restrict__ d_n,
                                                    unsigned long long *__restrict__ out) {
    __shared__ unsigned int s[7];
    const int64_t n = mc_dev_count(d_n, n_cap);
    if ((int64_t)blockIdx.x * blockDim.x >= n) return;       // block-uniform
    if (threadIdx.x < 7) s[threadIdx.x] = 0u;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const mc_call &c = calls[i];
        if (c.kind == MC_CALL) {
            atomicAdd(&s[c.close_rec == 0xFFFFFFFFu ? 1 : 0], 1u);
            if (c.label && c.close_rec != 0xFFFFFFFFu) atomicAdd(&s[5], 1u);
        } else if (c.kind == MC_TOO_MANY_SKIPS) atomicAdd(&s[c.close_rec == 0xFFFFFFFFu ? 6 : 2], 1u);
        else if (c.kind == MC_MULTI_M) atomicAdd(&s[3], 1u);
        if (c.kind != MC_NONE && c.err) atomicAdd(&s[4], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 7 && s[threadIdx.x]) atomicAdd(out + threadIdx.x, (unsigned long long)s[threadIdx.x]);
}

// check_thresh of make_bed.py:21-28 per site slot: len(list) >= depth_thresh, then np.mean(0/1 list) = meth / depth in float64
// compared with mod_thresh (>= for methylated loci, < with --control)
__global__ void __launch_bounds__(256)
k_bed_select(const uint32_t *__restrict__ depth, const uint32_t *__restrict__ meth, int64_t n_sites, long long depth_thresh,
             double mod_thresh, int control, uint8_t *__restrict__ flags, unsigned long long *__restrict__ d_count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool keep = false;
    if (i < n_sites) {
        const uint32_t d = depth[i];
        if (d > 0u && (long long)d >= depth_thresh) {
            const double frac = __ddiv_rn((double)meth[i], (double)d);
            keep = control ? (frac < mod_thresh) : (frac >= mod_thresh);
        }
        flags[i] = keep ? 1 : 0;
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(d_count, (unsigned long long)__popc(m));
}

// ---- chunk / rank edges: the one window that is still open when the text ends (see mc_carry in the header) -------------------
__device__ __forceinline__ void copy_row(mc_call *dst, const mc_call *src) {
    const uint4 *s4 = reinterpret_cast<const uint4 *>(src);
    uint4 *d4 = reinterpret_cast<uint4 *>(dst);
#pragma unroll
    for (int j = 0; j < 8; ++j) d4[j] = s4[j];
}

// one warp: first kept record of the chunk (first record of the first segment that passes the quality filter, :167)
__global__ void __launch_bounds__(32)
k_carry_rows(mc_call *__restrict__ rows, const unsigned long long *__restrict__ d_ncalls, const mc_record *__restrict__ rec,
             const unsigned long long *__restrict__ d_n_records, const uint32_t *__restrict__ seg_start,
             const unsigned long long *__restrict__ d_nseg, const double *__restrict__ seg_qual, double qual_thresh,
             mc_carry *__restrict__ carry, unsigned long long *__restrict__ d_nrows_out, const unsigned long long *__restrict__ d_abort) {
    const int lane = threadIdx.x;
    if (d_abort && *d_abort) {                                // overflow earlier in this chunk: leave the carry as it is
        if (lane == 0) *d_nrows_out = 0ull;
        return;
    }
    const unsigned long long n_rows = *d_ncalls, n_rec = *d_n_records, n_seg = *d_nseg;
    long long fk_rec = -1;
    if (n_rec > 0 && n_seg > 0) {
        if (!(qual_thresh > 0.0)) fk_rec = 0;
        else {
            for (unsigned long long s0 = 0; s0 < n_seg && fk_rec < 0; s0 += 32) {
                const unsigned long long sg = s0 + lane;
                const bool ok = sg < n_seg && !(seg_qual[sg] < qual_thresh);
                const uint32_t m = __ballot_sync(0xffffffffu, ok);
                if (m) fk_rec = (long long)seg_start[s0 + (__ffs(m) - 1)];
            }
        }
    }
    if (lane != 0) return;
    int fk_contig = -1;
    if (fk_rec >= 0) fk_contig = (int)rec[fk_rec].contig;
    mc_call *slot0 = rows;
    bool resolved = false;
    if (carry->valid && fk_contig >= 0) {
        copy_row(slot0, &carry->row);
        slot0->chrom_contig = (uint16_t)fk_contig;
        slot0->close_rec = (uint32_t)fk_rec;
        slot0->read_off = -1;
        slot0->seg = 0xFFFFFFFFu;                 // not a segment of this chunk
        carry->valid = 0u;
        resolved = true;
    }
    if (!resolved) {
        mc_call z;
        memset(&z, 0, sizeof(z));
        z.kind = MC_NONE;
        z.site = -1;
        copy_row(slot0, &z);
    }
    // the chunk's own open window: always its last row (the hand-off at the end of the last read that passed the filter)
    if (n_rows > 0) {
        const mc_call *last = rows + n_rows;      // rows[1 .. n_rows] hold the chunk's rows
        if (last->close_rec == 0xFFFFFFFFu && (last->kind == MC_CALL || last->kind == MC_TOO_MANY_SKIPS)) {
            copy_row(&carry->row, last);
            carry->valid = 1u;
        }
    }
    if (carry->first_kept_contig < 0 && fk_contig >= 0) carry->first_kept_contig = fk_contig;
    carry->chunks += 1ull;
    *d_nrows_out = n_rows + 1ull;
}

__global__ void k_carry_reset(mc_carry *carry) {
    memset(carry, 0, sizeof(*carry));
    carry->first_kept_contig = -1;
    carry->row.kind = MC_NONE;
}

__global__ void k_carry_close(mc_carry *__restrict__ carry, int closing_contig, const long long *__restrict__ d_next, int from, int count,
                              mc_call *__restrict__ out, uint32_t *__restrict__ depth, uint32_t *__restrict__ meth,
                              unsigned long long *__restrict__ first, int64_t n_sites, unsigned long long *__restrict__ d_row_base) {
    const unsigned long long row_index = d_row_base ? *d_row_base : 0ull;
    int cc = closing_contig;
    if (cc < 0 && d_next) {
        for (int j = from; j < count; ++j) {
            if (d_next[j] >= 0) { cc = (int)d_next[j]; break; }
        }
    }
    mc_call z;
    memset(&z, 0, sizeof(z));
    z.kind = MC_NONE;
    z.site = -1;
    if (!carry->valid || cc < 0) {                // nothing open, or nobody closes it (end of the file: dropped, SURVEY.md Q3)
        copy_row(out, &z);
        carry->valid = 0u;
        return;
    }
    copy_row(out, &carry->row);
    out->chrom_contig = (uint16_t)cc;
    out->close_rec = 0u;
    out->read_off = -1;
    out->seg = 0xFFFFFFFFu;
    out->pad1 = (uint32_t)(row_index & 0xFFFFFFFFull);
    out->pad2 = (uint32_t)(row_index >> 32);
    carry->valid = 0u;
    if (out->kind == MC_CALL && !out->err && depth && out->chrom_contig == out->win_contig && out->site >= 0 && out->site < n_sites) {
        atomicAdd(depth + out->site, 1u);
        if (out->label) atomicAdd(meth + out->site, 1u);
        atomicMin(first + out->site, row_index);
    }
    if (d_row_base) *d_row_base = row_index + 1ull;
}

}  // namespace

extern "C" int mc_count_calls(const mc_call *d_calls, const uint64_t *d_nrows, int64_t row_cap, uint64_t *d_out, void *stream) {
    MC_REQUIRE(d_calls && d_nrows && d_out, "null pointer");
    if (row_cap <= 0) return MC_OK;
    k_count_calls<<<(unsigned)((row_cap + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_calls, row_cap, reinterpret_cast<const unsigned long long *>(d_nrows), reinterpret_cast<unsigned long long *>(d_out));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_carry_reset(mc_carry *d_carry, void *stream) {
    MC_REQUIRE(d_carry, "null pointer");
    k_carry_reset<<<1, 1, 0, (cudaStream_t)stream>>>(d_carry);
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_carry_rows(mc_call *d_rows, const uint64_t *d_ncalls, const mc_record *d_rec, const uint64_t *d_n_records,
                             const uint32_t *d_seg_start, const uint64_t *d_nseg, const double *d_seg_qual, double qual_thresh,
                             mc_carry *d_carry, uint64_t *d_nrows_out, const uint64_t *d_abort, void *stream) {
    MC_REQUIRE(d_rows && d_ncalls && d_rec && d_n_records && d_seg_start && d_nseg && d_seg_qual && d_carry && d_nrows_out, "null pointer");
    k_carry_rows<<<1, 32, 0, (cudaStream_t)stream>>>(d_rows, reinterpret_cast<const unsigned long long *>(d_ncalls), d_rec,
                                                     reinterpret_cast<const unsigned long long *>(d_n_records), d_seg_start,
                                                     reinterpret_cast<const unsigned long long *>(d_nseg), d_seg_qual, qual_thresh, d_carry,
                                                     reinterpret_cast<unsigned long long *>(d_nrows_out),
                                                     reinterpret_cast<const unsigned long long *>(d_abort));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_bed_select(const uint32_t *d_depth, const uint32_t *d_meth, int64_t n_sites, int64_t depth_thresh, double mod_thresh,
                             int control, uint8_t *d_flags, uint64_t *d_count, void *stream) {
    MC_REQUIRE(d_depth && d_meth && d_flags && d_count, "null pointer");
    MC_CUDA_CHECK(cudaMemsetAsync(d_count, 0, 8, (cudaStream_t)stream));
    if (n_sites <= 0) return MC_OK;
    k_bed_select<<<(unsigned)((n_sites + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_depth, d_meth, n_sites, (long long)depth_thresh, mod_thresh,
                                                                                      control, d_flags, reinterpret_cast<unsigned long long *>(d_count));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_chunk_guard(const uint64_t *d_counters, int64_t rec_cap, const uint64_t *d_n_records, int64_t rec_out_cap,
                              const uint64_t *d_nseg, int64_t seg_cap, const uint64_t *d_ncalls, int64_t call_cap, uint64_t *d_abort,
                              uint64_t *d_sticky, void *stream) {
    MC_REQUIRE(d_counters && d_n_records && d_nseg && d_ncalls && d_abort, "null pointer");
    k_chunk_guard<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned long long *>(d_counters), (unsigned long long)rec_cap,
                                                    reinterpret_cast<const unsigned long long *>(d_n_records), (unsigned long long)rec_out_cap,
                                                    reinterpret_cast<const unsigned long long *>(d_nseg), (unsigned long long)seg_cap,
                                                    reinterpret_cast<const unsigned long long *>(d_ncalls), (unsigned long long)call_cap,
                                                    reinterpret_cast<unsigned long long *>(d_abort), reinterpret_cast<unsigned long long *>(d_sticky));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_carry_close(mc_carry *d_carry, int closing_contig, const int64_t *d_next_contigs, int from, int count,
                              mc_call *d_row_out, uint32_t *d_depth, uint32_t *d_meth, uint64_t *d_first, int64_t n_sites,
                              uint64_t *d_row_base, void *stream) {
    MC_REQUIRE(d_carry && d_row_out, "null pointer");
    MC_REQUIRE(!d_depth || (d_meth && d_first), "histogram needs depth, meth and first");
    k_carry_close<<<1, 1, 0, (cudaStream_t)stream>>>(d_carry, closing_contig, reinterpret_cast<const long long *>(d_next_contigs), from, count,
                                                    d_row_out, d_depth, d_meth, reinterpret_cast<unsigned long long *>(d_first), n_sites,
                                                    reinterpret_cast<unsigned long long *>(d_row_base));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int64_t mc_classify_workspace_bytes(int64_t row_cap) { return 256 + 4 * (row_cap < 1 ? 1 : row_cap); }

extern "C" int mc_classify(mc_call *d_calls, const uint64_t *d_nrows, int64_t n_calls /* capacity */, const mc_model *models,
                           void *d_ws, void *stream) {
    MC_REQUIRE(d_calls && d_nrows && models && d_ws, "null pointer");
    if (n_calls <= 0) return MC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned long long *dn = reinterpret_cast<const unsigned long long *>(d_nrows);
    const mc_model &m0 = models[0], &m1 = models[1];
    // one kernel serves both models, so they must be of one kind; each is validated on its own
    MC_REQUIRE(m0.kind == m1.kind, "models 0 ('MH') and 1 ('MG') are of different kinds");
    MC_REQUIRE(m0.n_in >= 1 && m0.n_in <= MC_MAXK + 1, "model 0 ('MH') input width out of range");
    MC_REQUIRE(m1.n_in == m0.n_in, "models 0 ('MH') and 1 ('MG') take different input widths");
    switch (m0.kind) {
        case MC_MLP: {
            for (const mc_model *m : {&m0, &m1}) {
                MC_REQUIRE(m->n_layers >= 1 && m->n_layers < 8, "MLP depth out of range");
                MC_REQUIRE(m->sizes[0] == m->n_in, "MLP input layer does not match its input width");
                for (int l = 0; l <= m->n_layers; ++l) MC_REQUIRE(m->sizes[l] >= 1 && m->sizes[l] <= MAX_WIDTH, "MLP layer too wide");
                MC_REQUIRE(m->sizes[m->n_layers] == 1, "MLP must have one logistic output");
            }
            int width = 8;
            for (int l = 0; l <= m0.n_layers; ++l) width = m0.sizes[l] > width ? m0.sizes[l] : width;
            for (int l = 0; l <= m1.n_layers; ++l) width = m1.sizes[l] > width ? m1.sizes[l] : width;
            width = (width + 3) & ~3;
            auto count = [](const mc_model &m, int &nw, int &nb) {
                nw = nb = 0;
                if (m.kind != MC_MLP) return;
                for (int l = 0; l < m.n_layers; ++l) { nw += m.sizes[l] * m.sizes[l + 1]; nb += m.sizes[l + 1]; }
            };
            int nw0, nb0, nw1, nb1;
            count(m0, nw0, nb0);
            count(m1, nw1, nb1);
            const int alias = (m1.kind == MC_MLP && m1.d_weights == m0.d_weights) ? 1 : 0;
            if (alias) nw1 = nb1 = 0;                             // one model given twice: stage it once
            int dev = 0, sms = 0;
            MC_CUDA_CHECK(cudaGetDevice(&dev));
            MC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
            const size_t act_bytes = sizeof(double) * 2 * (size_t)width * WARPS;
            const size_t staged_bytes = act_bytes + sizeof(double) * (size_t)(nw0 + nb0 + nw1 + nb1);
            int64_t blocks = (n_calls + WARPS - 1) / WARPS;
            if (blocks > (int64_t)sms * 8) blocks = (int64_t)sms * 8;           // persistent: warps stride over the calls
            auto one_hidden = [](const mc_model &m) {
                return m.kind == MC_MLP && m.n_layers == 2 && m.sizes[0] <= MLP_MAX_IN && m.sizes[2] == 1;
            };
            const size_t weight_bytes = sizeof(double) * (size_t)(nw0 + nb0 + nw1 + nb1);
            if (one_hidden(m0) && (alias || one_hidden(m1)) && weight_bytes <= 100 * 1024) {
                int64_t b2 = (n_calls + WARPS * 8 - 1) / (WARPS * 8);
                if (b2 > (int64_t)sms * 8) b2 = (int64_t)sms * 8;
                // index list of the MC_CALL rows first: [count (u64, 256-byte slot)][row indices u32]
                unsigned long long *d_nidx = reinterpret_cast<unsigned long long *>(d_ws);
                uint32_t *d_idx = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(d_ws) + 256);
                MC_CUDA_CHECK(cudaMemsetAsync(d_nidx, 0, 8, st));
                k_call_index<<<(unsigned)((n_calls + 255) / 256), 256, 0, st>>>(d_calls, n_calls, dn, d_idx, d_nidx);
                MC_LAUNCH_CHECK();
                MC_CUDA_CHECK(cudaFuncSetAttribute(k_mlp_1hidden, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)weight_bytes));
                k_mlp_1hidden<<<(unsigned)b2, WARPS * 32, weight_bytes, st>>>(d_calls, d_idx, d_nidx, m0, m1, nw0, nb0, nw1, nb1, alias);
            } else if (staged_bytes <= 100 * 1024) {
                MC_CUDA_CHECK(cudaFuncSetAttribute(k_mlp<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)staged_bytes));
                k_mlp<true><<<(unsigned)blocks, WARPS * 32, staged_bytes, st>>>(d_calls, n_calls, dn, m0, m1, width, nw0, nb0, nw1, nb1, alias);
            } else {
                k_mlp<false><<<(unsigned)blocks, WARPS * 32, act_bytes, st>>>(d_calls, n_calls, dn, m0, m1, width, 0, 0, 0, 0, 0);
            }
            break;
        }
        case MC_LR:
        case MC_GNB:
            k_linear<<<(unsigned)((n_calls + 255) / 256), 256, 0, st>>>(d_calls, n_calls, dn, m0, m1);
            break;
        case MC_RF: {
            int mx = m0.max_nodes > m1.max_nodes ? m0.max_nodes : m1.max_nodes;
            MC_REQUIRE(mx >= 1, "RF max_nodes missing");
            const size_t smem = (size_t)mx * (8 + 8 + 4 + 4 + 4);
            MC_REQUIRE(smem <= 200 * 1024, "RF tree too large for shared-memory staging");
            MC_CUDA_CHECK(cudaFuncSetAttribute(k_rf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_rf<<<(unsigned)((n_calls + 255) / 256), 256, smem, st>>>(d_calls, n_calls, dn, m0, m1, mx);
            break;
        }
        default:
            MC_REQUIRE(false, "unknown model kind");
    }
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_hist_accumulate(const mc_call *d_calls, const uint64_t *d_nrows, int64_t row_cap, uint32_t *d_depth, uint32_t *d_meth,
                                  uint64_t *d_first, int64_t n_sites, uint64_t *d_row_base, mc_call *d_odd, int64_t odd_cap,
                                  uint64_t *d_n_odd, const uint64_t *d_abort, void *stream) {
    MC_REQUIRE(d_calls && d_nrows && d_depth && d_meth && d_first && d_row_base && d_odd && d_n_odd, "null pointer");
    if (row_cap <= 0) return MC_OK;
    k_hist<<<(unsigned)((row_cap + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_calls, row_cap, reinterpret_cast<const unsigned long long *>(d_nrows), d_depth, d_meth,
        reinterpret_cast<unsigned long long *>(d_first), n_sites, reinterpret_cast<const unsigned long long *>(d_row_base), d_odd,
        (unsigned long long)odd_cap, reinterpret_cast<unsigned long long *>(d_n_odd), reinterpret_cast<const unsigned long long *>(d_abort));
    MC_LAUNCH_CHECK();
    k_advance_base<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long *>(d_row_base),
                                                      reinterpret_cast<const unsigned long long *>(d_nrows),
                                                      reinterpret_cast<const unsigned long long *>(d_abort));
    MC_LAUNCH_CHECK();
    return MC_OK;
}
