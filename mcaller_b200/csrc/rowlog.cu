// Row log of the multi-GPU product path: make_bed.py's per-read summaries (--vo :96-97/:147-159, -p :115-127) from the
// device rows.  Each rank appends the rows its histogram counts (mc_rowlog_append, one launch per chunk after the
// classifier); rank 0 groups the gathered entries by locus (mc_rowlog_group): a counting scatter over the exclusive scan of
// the per-locus depths, then a merge sort of each locus's segment on the global row index, because the scatter's atomics
// leave the order inside a segment undefined.  Row indices are unique, so each merge step places an entry at its own index
// in its run plus the number of smaller keys in the partner run (one binary search): no per-locus size limit.
#include "common.cuh"

namespace {

constexpr int64_t ENTRY_BYTES = (int64_t)sizeof(mc_row_entry);

__device__ __forceinline__ mc_row_entry *entry_at(uint8_t *log, int64_t stride, unsigned long long i) {
    return reinterpret_cast<mc_row_entry *>(log + (int64_t)i * stride);
}
__device__ __forceinline__ const mc_row_entry *entry_at(const uint8_t *log, int64_t stride, int64_t i) {
    return reinterpret_cast<const mc_row_entry *>(log + i * stride);
}

__global__ void __launch_bounds__(256)
k_rowlog_append(const mc_call *__restrict__ calls, int64_t n_cap, const unsigned long long *__restrict__ d_n,
                const unsigned long long *__restrict__ d_row_base, const uint8_t *__restrict__ site_flags, int64_t n_sites, int n_feat,
                uint8_t *__restrict__ log, int64_t stride, unsigned long long log_cap, unsigned long long *__restrict__ d_n_log,
                unsigned long long *__restrict__ d_n_added, const unsigned long long *__restrict__ d_abort) {
    if (d_abort && *d_abort) return;                          // the chunk is run again with larger buffers
    const int64_t n = d_n ? mc_dev_count(d_n, n_cap) : n_cap;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool keep = false, odd = false;
    if (i < n) {
        const mc_call &c = calls[i];
        // the rows k_hist counts (or sends to the odd-row list)
        keep = c.kind == MC_CALL && c.close_rec != 0xFFFFFFFFu && !c.err;
        odd = c.chrom_contig != c.win_contig || c.site < 0 || c.site >= n_sites;
        if (keep && odd && !d_row_base) keep = false;            // k_carry_close keeps such a row out of the histogram
        if (keep && !odd && site_flags && !site_flags[c.site]) keep = false;
    }
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (!m) return;
    const int lane = threadIdx.x & 31, leader = __ffs(m) - 1;
    unsigned long long base = 0ull;
    if (lane == leader) {
        base = atomicAdd(d_n_log, (unsigned long long)__popc(m));
        if (d_n_added) atomicAdd(d_n_added, (unsigned long long)__popc(m));
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    if (!keep) return;
    const unsigned long long slot = base + (unsigned long long)__popc(m & ((1u << lane) - 1u));
    if (slot >= log_cap) return;
    const mc_call &c = calls[i];
    mc_row_entry *e = entry_at(log, stride, slot);
    e->row = d_row_base ? *d_row_base + (unsigned long long)i : ((unsigned long long)c.pad2 << 32) | (unsigned long long)c.pad1;
    e->site = odd ? -1 : c.site;
    e->pad = 0u;
    e->prob = c.prob;
    double *f = reinterpret_cast<double *>(e + 1);
    for (int j = 0; j < n_feat; ++j) f[j] = ((c.empty_mask >> j) & 1u) ? 0.0 : c.feat[j];     // an empty column prints as 0
}

// entry -> its locus, and a place in that locus's segment (unordered inside it)
__global__ void __launch_bounds__(256)
k_rowlog_scatter(const uint8_t *__restrict__ log, int64_t stride, int64_t n, const int32_t *__restrict__ locus_of_site, int64_t n_sites,
                 const unsigned long long *__restrict__ odd_rows, const int32_t *__restrict__ odd_locus, int64_t n_odd,
                 const uint32_t *__restrict__ locus_off, uint32_t *__restrict__ fill, unsigned long long *__restrict__ key,
                 uint32_t *__restrict__ idx, unsigned long long *__restrict__ counters) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const mc_row_entry e = *entry_at(log, stride, i);
    int32_t l = -1;
    if (e.site >= 0) {
        if (e.site < n_sites) l = locus_of_site[e.site];
    } else {
        int64_t lo = 0, hi = n_odd;                               // first odd row index >= e.row
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (odd_rows[mid] < e.row) lo = mid + 1; else hi = mid;
        }
        if (lo < n_odd && odd_rows[lo] == e.row) l = odd_locus[lo];
    }
    if (l < 0) { atomicAdd(&counters[0], 1ull); return; }
    const uint32_t a = locus_off[l], r = atomicAdd(&fill[l], 1u);
    if (r >= locus_off[l + 1] - a) { atomicAdd(&counters[1], 1ull); return; }
    key[a + r] = e.row;
    idx[a + r] = (uint32_t)i;
}

// number of keys in [p, p + n) smaller than k (ascending, unique)
__device__ __forceinline__ int64_t count_below(const unsigned long long *__restrict__ p, int64_t n, unsigned long long k) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (p[mid] < k) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// one block per locus: bottom-up merge sort of the segment on the row index, ping-ponging between (key_a, idx_a) and
// (key_b, idx_b); the final entry order goes to `order`
__global__ void __launch_bounds__(128)
k_rowlog_segsort(const uint32_t *__restrict__ locus_off, int64_t n_loci, unsigned long long *key_a, uint32_t *idx_a,
                 unsigned long long *key_b, uint32_t *idx_b, uint32_t *__restrict__ order) {
    for (int64_t l = blockIdx.x; l < n_loci; l += gridDim.x) {
        const int64_t a0 = locus_off[l], n = (int64_t)locus_off[l + 1] - a0;
        unsigned long long *sk = key_a + a0, *dk = key_b + a0;
        uint32_t *si = idx_a + a0, *di = idx_b + a0;
        for (int64_t w = 1; w < n; w *= 2) {
            for (int64_t t = threadIdx.x; t < n; t += blockDim.x) {
                const int64_t base = (t / (2 * w)) * (2 * w);
                const int64_t mid = min(base + w, n), end = min(base + 2 * w, n);
                const unsigned long long k = sk[t];
                const int64_t pos = t < mid ? t + count_below(sk + mid, end - mid, k)
                                            : base + (t - mid) + count_below(sk + base, mid - base, k);
                dk[pos] = k;
                di[pos] = si[t];
            }
            __syncthreads();
            unsigned long long *tk = sk; sk = dk; dk = tk;
            uint32_t *ti = si; si = di; di = ti;
        }
        for (int64_t t = threadIdx.x; t < n; t += blockDim.x) order[a0 + t] = si[t];
        __syncthreads();
    }
}

// grouped order -> probabilities and (for the t-tests) the feature rows in mc_colstats's layout
__global__ void __launch_bounds__(256)
k_rowlog_gather(const uint8_t *__restrict__ log, int64_t stride, int n_feat, const uint32_t *__restrict__ order, int64_t n_rows,
                double *__restrict__ prob, double *__restrict__ vals, uint32_t *__restrict__ ncol) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_rows) return;
    const mc_row_entry *e = entry_at(log, stride, (int64_t)order[j]);
    prob[j] = e->prob;
    if (vals) {
        const double *f = reinterpret_cast<const double *>(e + 1);
        for (int c = 0; c < n_feat; ++c) vals[j * (MC_MAXK + 1) + c] = f[c];
        ncol[j] = (uint32_t)n_feat;
    }
}

inline int64_t up256(int64_t b) { return ((b + 255) / 256) * 256; }

}  // namespace

extern "C" int64_t mc_rowlog_stride(int32_t n_feat) { return ENTRY_BYTES + 8 * (int64_t)(n_feat > 0 ? n_feat : 0); }

extern "C" int mc_rowlog_append(const mc_call *d_calls, const uint64_t *d_nrows, int64_t row_cap, const uint64_t *d_row_base,
                                const uint8_t *d_site_flags, int64_t n_sites, int32_t n_feat, void *d_log, int64_t log_cap,
                                uint64_t *d_n_log, uint64_t *d_n_added, const uint64_t *d_abort, void *stream) {
    MC_REQUIRE(d_calls && d_log && d_n_log, "null pointer");
    MC_REQUIRE(n_feat >= 0 && n_feat <= MC_MAXK, "feature count out of range");
    MC_REQUIRE(log_cap >= 0, "negative capacity");
    if (row_cap <= 0) return MC_OK;
    k_rowlog_append<<<(unsigned)((row_cap + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_calls, row_cap, reinterpret_cast<const unsigned long long *>(d_nrows), reinterpret_cast<const unsigned long long *>(d_row_base),
        d_site_flags, n_sites, n_feat, reinterpret_cast<uint8_t *>(d_log), mc_rowlog_stride(n_feat), (unsigned long long)log_cap,
        reinterpret_cast<unsigned long long *>(d_n_log), reinterpret_cast<unsigned long long *>(d_n_added),
        reinterpret_cast<const unsigned long long *>(d_abort));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

// workspace: [fill u32 n_loci][key_a u64][key_b u64][idx_a u32][idx_b u32][order u32] (n_rows each) [scan sums]
extern "C" int64_t mc_rowlog_group_workspace_bytes(int64_t n_rows, int64_t n_loci) {
    if (n_rows < 1) n_rows = 1;
    if (n_loci < 1) n_loci = 1;
    return up256(4 * n_loci) + 2 * up256(8 * n_rows) + 3 * up256(4 * n_rows) + mc_exscan_ws_bytes(n_loci + 1) + 256;
}

extern "C" int mc_rowlog_group(const void *d_log, int64_t n_entries, int32_t n_feat, const int32_t *d_locus_of_site, int64_t n_sites,
                               const uint64_t *d_odd_rows, const int32_t *d_odd_locus, int64_t n_odd, const uint32_t *d_depth,
                               int64_t n_loci, int64_t n_rows, uint32_t *d_locus_off, double *d_prob, double *d_vals, uint32_t *d_ncol,
                               void *d_ws, uint64_t *d_counters, void *stream) {
    MC_REQUIRE(d_depth && d_locus_off && d_ws && d_counters, "null pointer");
    MC_REQUIRE(n_entries == 0 || d_log, "null log");
    MC_REQUIRE(n_sites == 0 || d_locus_of_site, "null site map");
    MC_REQUIRE(n_odd == 0 || (d_odd_rows && d_odd_locus), "null odd-row map");
    MC_REQUIRE(n_rows == 0 || d_prob, "null probability output");
    MC_REQUIRE(!d_vals || (d_ncol && n_feat >= 1 && n_feat <= MC_MAXK), "feature output needs d_ncol and 1 <= n_feat <= MC_MAXK");
    MC_REQUIRE(n_loci >= 0 && n_rows >= 0 && n_rows < (1ll << 32) && n_entries < (1ll << 32), "count out of range");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t *ws = reinterpret_cast<uint8_t *>(d_ws);
    const int64_t nr = n_rows < 1 ? 1 : n_rows, nl = n_loci < 1 ? 1 : n_loci;
    uint32_t *fill = reinterpret_cast<uint32_t *>(ws);
    ws += up256(4 * nl);
    unsigned long long *key_a = reinterpret_cast<unsigned long long *>(ws), *key_b = key_a + (up256(8 * nr) / 8);
    ws += 2 * up256(8 * nr);
    uint32_t *idx_a = reinterpret_cast<uint32_t *>(ws), *idx_b = idx_a + up256(4 * nr) / 4, *order = idx_b + up256(4 * nr) / 4;
    ws += 3 * up256(4 * nr);
    MC_CUDA_CHECK(cudaMemsetAsync(d_counters, 0, 16, st));
    int rc = mc_exscan_u32(d_depth, d_locus_off, n_loci + 1, nullptr, nullptr, ws, st);    // entry n_loci (count 0) = the total
    if (rc) return rc;
    if (n_entries == 0) return MC_OK;
    MC_CUDA_CHECK(cudaMemsetAsync(fill, 0, 4 * (size_t)nl, st));           // with no locus every entry counts as unplaced
    // a locus the log holds fewer rows of than its depth (the host raises) still sorts and gathers inside the buffers
    MC_CUDA_CHECK(cudaMemsetAsync(key_a, 0, 8 * (size_t)nr, st));
    MC_CUDA_CHECK(cudaMemsetAsync(idx_a, 0, 4 * (size_t)nr, st));
    const int64_t stride = mc_rowlog_stride(n_feat);
    k_rowlog_scatter<<<(unsigned)((n_entries + 255) / 256), 256, 0, st>>>(
        reinterpret_cast<const uint8_t *>(d_log), stride, n_entries, d_locus_of_site, n_sites,
        reinterpret_cast<const unsigned long long *>(d_odd_rows), d_odd_locus, n_odd, d_locus_off, fill, key_a, idx_a,
        reinterpret_cast<unsigned long long *>(d_counters));
    MC_LAUNCH_CHECK();
    if (n_rows == 0) return MC_OK;
    int dev = 0, sms = 0;
    MC_CUDA_CHECK(cudaGetDevice(&dev));
    MC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int64_t blocks = n_loci < (int64_t)sms * 16 ? n_loci : (int64_t)sms * 16;
    k_rowlog_segsort<<<(unsigned)blocks, 128, 0, st>>>(d_locus_off, n_loci, key_a, idx_a, key_b, idx_b, order);
    MC_LAUNCH_CHECK();
    k_rowlog_gather<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(reinterpret_cast<const uint8_t *>(d_log), stride, n_feat, order,
                                                                      n_rows, d_prob, d_vals, d_ncol);
    MC_LAUNCH_CHECK();
    return MC_OK;
}
