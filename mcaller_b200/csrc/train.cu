// Training of mCaller's MLP models (mCaller --train -c NN): scikit-learn 1.9 MLPClassifier(hidden_layer_sizes=100,
// activation='tanh', solver='adam', batch_size='auto', shuffle=True).fit -- BaseMultilayerPerceptron._fit_stochastic,
// _backprop, AdamOptimizer -- for a binary target, in float64.
//
// One CTA per job (a cross-validation fold or a final fit), persistent over the epochs of a launch.  A step is 200 rows of a
// d-100-1 network: ~0.3 MFLOP on the FP64 pipe, far too narrow for a tensor-core tile, and 1 500 of them per epoch at 300 k
// rows depend on each other through the weights.  So everything lives on chip: parameters, current batch, hidden
// activations and gradient partials in shared memory, the Adam moments in the registers of the thread that owns the
// parameter.  Every reduction runs in an order fixed by the thread layout alone, so a job's result does not depend on
// which jobs share the launch or on the run.  The host draws the initial weights and every epoch's shuffle from
// numpy's RandomState(seed) exactly as scikit-learn does; the kernel never draws a random number.
#include "common.cuh"

namespace {

constexpr int H = MC_TRAIN_HIDDEN;
constexpr int BATCH = MC_TRAIN_BATCH;
constexpr int DMAX = MC_MAXK + 1;
constexpr int THREADS = 512;
constexpr int WARPS = THREADS / 32;
constexpr int NP_MAX = DMAX * H + 2 * H + 1;                  // W0 (d x H), W1 (H), c0 (H), c1
constexpr int OWN = (NP_MAX + THREADS - 1) / THREADS;         // parameters owned (Adam state in registers) per thread
constexpr int GROUPS = 5;                                     // row groups of the gradient partials (GROUPS * H <= THREADS)
static_assert(GROUPS * H <= THREADS, "one thread per (row group, hidden unit)");
static_assert(GROUPS * (DMAX + 2) * H <= BATCH * H, "gradient partials reuse the activation buffer");
constexpr double BETA1 = 0.9, BETA2 = 0.999, ADAM_EPS = 1e-8;  // AdamOptimizer defaults
constexpr double PROB_EPS = 2.220446049250313e-16;            // np.finfo(np.float64).eps, the clip of binary_log_loss

// shared memory, in doubles
constexpr int S_P = 0;                      // parameters [NP]
constexpr int S_X = S_P + NP_MAX;           // batch features [BATCH][d]
constexpr int S_Y = S_X + BATCH * DMAX;     // batch targets
constexpr int S_A = S_Y + BATCH;            // hidden activations [BATCH][H]; then gradient partials [GROUPS][d + 2][H]
constexpr int S_D = S_A + BATCH * H;        // output deltas p - y
constexpr int S_RED = S_D + BATCH;          // per-warp sums: [0] log-likelihood, [1] deltas, [2] squared weights
constexpr int S_TOTAL = S_RED + 3 * WARPS;
constexpr size_t SMEM_BYTES = sizeof(double) * S_TOTAL + 16;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Σ W0² + Σ W1² over the weights this thread owns, summed per warp into red[warp]
__device__ __forceinline__ void weight_sumsq(const double *P, int n_weights, double *red) {
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        const int p = threadIdx.x + q * THREADS;
        if (p < n_weights) s = fma(P[p], P[p], s);
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
}

__device__ __forceinline__ void load_batch(const mc_train_job &J, const int32_t *idx, int b, int d, double *X, double *Y) {
    const int r0 = b * BATCH, nb = min(BATCH, J.n - r0);
    for (int q = threadIdx.x; q < nb * d; q += THREADS) {
        const int r = q / d, i = q - r * d;
        X[q] = __ldg(J.d_x + (int64_t)__ldg(idx + r0 + r) * d + i);
    }
    for (int r = threadIdx.x; r < nb; r += THREADS) Y[r] = __ldg(J.d_y + __ldg(idx + r0 + r));
}

__global__ void __launch_bounds__(256) k_mlp_train_init(mc_train_job *jobs) {
    mc_train_job &J = jobs[blockIdx.x];
    const int np = J.d * H + 2 * H + 1;
    for (int p = threadIdx.x; p < 2 * np; p += blockDim.x) J.d_w[np + p] = 0.0;
    if (threadIdx.x == 0) {
        J.best_loss = __longlong_as_double(0x7ff0000000000000ll);      // +inf
        J.n_iter = 0; J.no_improve = 0; J.stopped = 0; J.pad = 0;
    }
}

// `epochs` epochs of every job that has not stopped.  d_idx + job.idx_off holds the job's [epochs][n] row numbers: epoch e's
// sample order, batches being consecutive slices of it.
__global__ void __launch_bounds__(THREADS, 1) k_mlp_train(mc_train_job *jobs, const int32_t *__restrict__ d_idx, int epochs) {
    extern __shared__ __align__(16) double sm[];
    mc_train_job &Jg = jobs[blockIdx.x];
    const mc_train_job J = Jg;
    if (J.stopped) return;
    const int d = J.d, n = J.n, np = d * H + 2 * H + 1, nw = d * H + H;
    const int nbatch = (n + BATCH - 1) / BATCH;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    double *P = sm + S_P, *X = sm + S_X, *Y = sm + S_Y, *A = sm + S_A, *D = sm + S_D, *red = sm + S_RED;
    const double *W0 = P, *W1 = P + d * H, *c0 = P + nw, *c1 = P + nw + H;

    double m[OWN], v[OWN];
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        const int p = tid + q * THREADS;
        if (p < np) { P[p] = J.d_w[p]; m[q] = J.d_w[np + p]; v[q] = J.d_w[2 * np + p]; }
    }
    __syncthreads();
    weight_sumsq(P, nw, red + 2 * WARPS);
    int n_iter = J.n_iter, no_improve = J.no_improve, stopped = 0;
    double best = J.best_loss;
    __shared__ int s_stop;
    load_batch(J, d_idx + J.idx_off, 0, d, X, Y);

    for (int e = 0; e < epochs && !stopped; ++e) {
        const int32_t *idx = d_idx + J.idx_off + (int64_t)e * n;
        double acc = 0.0;                                           // Σ batch_loss * nb (thread 0)
        for (int b = 0; b < nbatch; ++b) {
            const int nb = min(BATCH, n - b * BATCH);
            __syncthreads();
            // forward: a = tanh(x W0 + c0)  (the dot product first, then the intercept, like x @ W0 += c0)
            for (int q = tid; q < nb * H; q += THREADS) {
                const int r = q / H, j = q - r * H;
                double z = 0.0;
                for (int i = 0; i < d; ++i) z = fma(X[r * d + i], W0[i * H + j], z);
                A[q] = mc_tanh(z + c0[j]);
            }
            __syncthreads();
            // output: p = expit(a W1 + c1), one warp per row; log-likelihood and deltas summed per warp in row order
            {
                double ll = 0.0, ds = 0.0;
                for (int r = warp; r < nb; r += WARPS) {
                    double z = 0.0;
#pragma unroll
                    for (int s = 0; s < (H + 31) / 32; ++s) {
                        const int j = lane + 32 * s;
                        if (j < H) z = fma(A[r * H + j], W1[j], z);
                    }
                    z = warp_sum(z);
                    const double p = mc_expit(z + c1[0]), y = Y[r];
                    const double pc = fmin(fmax(p, PROB_EPS), 1.0 - PROB_EPS);
                    ll += y != 0.0 ? log(pc) : log(1.0 - pc);
                    const double dz = p - y;
                    ds += dz;
                    if (lane == 0) D[r] = dz;
                }
                if (lane == 0) { red[warp] = ll; red[WARPS + warp] = ds; }
            }
            __syncthreads();
            if (tid == 0) {
                double ll = 0.0, sq = 0.0;
                for (int w = 0; w < WARPS; ++w) { ll += red[w]; sq += red[2 * WARPS + w]; }
                const double loss = -ll / nb + (0.5 * J.alpha) * sq / nb;
                acc += loss * nb;
            }
            // backward partials: thread (g, j) sums over its rows  a_j dz, da_j and x_i da_j, da = dz W1_j (1 - a_j^2)
            double gw1 = 0.0, gc0 = 0.0, gx[DMAX];
#pragma unroll
            for (int i = 0; i < DMAX; ++i) gx[i] = 0.0;
            const int g = tid / H, j = tid - g * H;
            if (g < GROUPS) {
                const int per = (nb + GROUPS - 1) / GROUPS, r1 = min(nb, (g + 1) * per);
                const double w1 = W1[j];
                for (int r = g * per; r < r1; ++r) {
                    const double a = A[r * H + j], dz = D[r];
                    gw1 = fma(a, dz, gw1);
                    const double da = (dz * w1) * (1.0 - a * a);
                    gc0 += da;
#pragma unroll
                    for (int i = 0; i < DMAX; ++i)
                        if (i < d) gx[i] = fma(X[r * d + i], da, gx[i]);
                }
            }
            __syncthreads();
            double *part = A;                                       // [GROUPS][d + 2][H]
            if (g < GROUPS) {
#pragma unroll
                for (int i = 0; i < DMAX; ++i)
                    if (i < d) part[(g * (d + 2) + i) * H + j] = gx[i];
                part[(g * (d + 2) + d) * H + j] = gw1;
                part[(g * (d + 2) + d + 1) * H + j] = gc0;
            }
            __syncthreads();
            // Adam on the parameters this thread owns: grad = (Σ + alpha W) / nb for weights, Σ / nb for intercepts
            const double t = (double)((int64_t)n_iter * nbatch + b + 1);
            const double lr_t = J.lr * sqrt(1.0 - pow(BETA2, t)) / (1.0 - pow(BETA1, t));
#pragma unroll
            for (int q = 0; q < OWN; ++q) {
                const int p = tid + q * THREADS;
                if (p >= np) continue;
                int row, col;                                       // row of the partials, hidden unit
                if (p < d * H) { row = p / H; col = p - row * H; }
                else if (p < nw) { row = d; col = p - d * H; }
                else if (p < nw + H) { row = d + 1; col = p - nw; }
                else { row = -1; col = 0; }
                double s = 0.0;
                if (row >= 0) {
                    for (int gg = 0; gg < GROUPS; ++gg) s += part[(gg * (d + 2) + row) * H + col];
                } else {
                    for (int w = 0; w < WARPS; ++w) s += red[WARPS + w];
                }
                const double grad = p < nw ? (s + J.alpha * P[p]) / nb : s / nb;
                m[q] = BETA1 * m[q] + (1.0 - BETA1) * grad;
                v[q] = BETA2 * v[q] + (1.0 - BETA2) * (grad * grad);
                P[p] += (-lr_t * m[q]) / (sqrt(v[q]) + ADAM_EPS);
            }
            weight_sumsq(P, nw, red + 2 * WARPS);
            // the next batch of this launch (X and Y are not read by the update above)
            if (b + 1 < nbatch) load_batch(J, idx, b + 1, d, X, Y);
            else if (e + 1 < epochs) load_batch(J, idx + n, 0, d, X, Y);
        }
        // end of epoch: loss curve and the no-improvement rule of _update_no_improvement_count.  Every thread counts the
        // epoch: n_iter gives the Adam step of the next epoch's updates.
        if (tid == 0) J.d_loss_curve[n_iter] = acc / n;
        ++n_iter;
        if (tid == 0) {
            const double loss = acc / n;
            no_improve = loss > best - J.tol ? no_improve + 1 : 0;
            if (loss < best) best = loss;
            s_stop = no_improve > J.n_iter_no_change ? 1 : (n_iter >= J.max_iter ? 2 : 0);
        }
        __syncthreads();
        stopped = s_stop;
    }
#pragma unroll
    for (int q = 0; q < OWN; ++q) {
        const int p = tid + q * THREADS;
        if (p < np) { J.d_w[p] = P[p]; J.d_w[np + p] = m[q]; J.d_w[2 * np + p] = v[q]; }
    }
    if (tid == 0) {
        Jg.n_iter = n_iter; Jg.no_improve = no_improve; Jg.best_loss = best; Jg.stopped = stopped;
    }
}

}  // namespace

extern "C" int mc_mlp_train_init(mc_train_job *d_jobs, int32_t n_jobs, void *stream) {
    MC_REQUIRE(d_jobs && n_jobs > 0, "bad argument");
    k_mlp_train_init<<<n_jobs, 256, 0, (cudaStream_t)stream>>>(d_jobs);
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_mlp_train_epochs(mc_train_job *d_jobs, int32_t n_jobs, const int32_t *d_idx, int32_t epochs, void *stream) {
    MC_REQUIRE(d_jobs && d_idx && n_jobs > 0 && epochs > 0, "bad argument");
    MC_CUDA_CHECK(cudaFuncSetAttribute(k_mlp_train, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
    k_mlp_train<<<n_jobs, THREADS, SMEM_BYTES, (cudaStream_t)stream>>>(d_jobs, d_idx, epochs);
    MC_LAUNCH_CHECK();
    return MC_OK;
}
