// Stages 2-4: file-order gather of the stage-1 records, read segmentation, per-read quality lookup,
// plus the generic exclusive scan they (and the window builder) share.
#include "parse.cuh"

namespace {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_IPT = 8;
constexpr int SCAN_BLOCK = SCAN_THREADS * SCAN_IPT;

// ---- generic exclusive scan over uint32 -----------------------------------------------------------------
// the item count may live on the device (d_n != nullptr): n_cap is then only the capacity the grid was sized for
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_reduce(const uint32_t *__restrict__ in, int64_t n_cap,
                                                            const unsigned long long *__restrict__ d_n,
                                                            unsigned long long *__restrict__ block_sums) {
    __shared__ int s_warp[SCAN_THREADS / 32 + 1];
    const int64_t n = d_n ? mc_dev_count(d_n, n_cap) : n_cap;
    const int64_t base = (int64_t)blockIdx.x * SCAN_BLOCK;
    unsigned long long acc = 0ull;
#pragma unroll
    for (int j = 0; j < SCAN_IPT; ++j) {
        const int64_t i = base + (int64_t)j * SCAN_THREADS + threadIdx.x;
        if (i < n) acc += in[i];
    }
    // block reduce (64-bit)
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
    __shared__ unsigned long long s_sum[SCAN_THREADS / 32];
    if ((threadIdx.x & 31) == 0) s_sum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0ull;
        for (int w = 0; w < SCAN_THREADS / 32; ++w) t += s_sum[w];
        block_sums[blockIdx.x] = t;
    }
    (void)s_warp;
}

__global__ void __launch_bounds__(1024) k_scan_sums(unsigned long long *__restrict__ block_sums, int64_t nb,
                                                   unsigned long long *__restrict__ d_total) {
    __shared__ unsigned long long s_w[33];
    __shared__ unsigned long long s_carry;
    if (threadIdx.x == 0) s_carry = 0ull;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int64_t c0 = 0; c0 < nb; c0 += 1024) {
        const int64_t i = c0 + threadIdx.x;
        const unsigned long long v = (i < nb) ? block_sums[i] : 0ull;
        unsigned long long inc = v;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) s_w[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            unsigned long long x = s_w[lane], xi = x;
            for (int d = 1; d < 32; d <<= 1) {
                unsigned long long t = __shfl_up_sync(0xffffffffu, xi, d);
                if (lane >= d) xi += t;
            }
            s_w[lane] = xi - x;
            if (lane == 31) s_w[32] = xi;
        }
        __syncthreads();
        const unsigned long long carry = s_carry;
        if (i < nb) block_sums[i] = carry + s_w[wid] + inc - v;
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + s_w[32];
        __syncthreads();
    }
    if (threadIdx.x == 0 && d_total) *d_total = s_carry;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_down(const uint32_t *__restrict__ in, int64_t n_cap,
                                                          const unsigned long long *__restrict__ d_n,
                                                          const unsigned long long *__restrict__ block_sums,
                                                          uint32_t *__restrict__ out) {
    __shared__ int s_warp[SCAN_THREADS / 32 + 1];
    const int64_t n = d_n ? mc_dev_count(d_n, n_cap) : n_cap;
    if ((int64_t)blockIdx.x * SCAN_BLOCK >= n) return;           // whole block beyond the count (block-uniform)
    // thread owns SCAN_IPT consecutive items so the scan order is the index order
    const int64_t base = (int64_t)blockIdx.x * SCAN_BLOCK + (int64_t)threadIdx.x * SCAN_IPT;
    uint32_t v[SCAN_IPT];
    int sum = 0;
#pragma unroll
    for (int j = 0; j < SCAN_IPT; ++j) {
        const int64_t i = base + j;
        v[j] = (i < n) ? in[i] : 0u;
        sum += (int)v[j];
    }
    int total;
    int off = mc_block_exscan<SCAN_THREADS>(sum, s_warp, total);
    uint32_t run = (uint32_t)block_sums[blockIdx.x] + (uint32_t)off;
#pragma unroll
    for (int j = 0; j < SCAN_IPT; ++j) {
        const int64_t i = base + j;
        if (i < n) out[i] = run;
        run += v[j];
    }
}

}  // namespace

int64_t mc_exscan_ws_bytes(int64_t n) { return ((n + SCAN_BLOCK - 1) / SCAN_BLOCK + 1) * 8 + 256; }

int mc_exscan_u32(const uint32_t *d_in, uint32_t *d_out, int64_t n_cap, const uint64_t *d_n, uint64_t *d_total, void *d_ws,
                  cudaStream_t st) {
    if (n_cap <= 0) {
        if (d_total) MC_CUDA_CHECK(cudaMemsetAsync(d_total, 0, 8, st));
        return MC_OK;
    }
    const int64_t nb = (n_cap + SCAN_BLOCK - 1) / SCAN_BLOCK;
    unsigned long long *sums = reinterpret_cast<unsigned long long *>(d_ws);
    const unsigned long long *dn = reinterpret_cast<const unsigned long long *>(d_n);
    k_scan_reduce<<<(unsigned)nb, SCAN_THREADS, 0, st>>>(d_in, n_cap, dn, sums);
    MC_LAUNCH_CHECK();
    k_scan_sums<<<1, 1024, 0, st>>>(sums, nb, reinterpret_cast<unsigned long long *>(d_total));
    MC_LAUNCH_CHECK();
    k_scan_down<<<(unsigned)nb, SCAN_THREADS, 0, st>>>(d_in, n_cap, dn, sums, d_out);
    MC_LAUNCH_CHECK();
    return MC_OK;
}

// workspace layout used by the stages: [A: uint32 n][B: uint32 n][scan sums]
extern "C" int64_t mc_windows_workspace_bytes(int64_t rec_cap);
extern "C" int64_t mc_workspace_bytes(int64_t n) {
    if (n < 1) n = 1;
    const int64_t a = ((n * 4 + 255) / 256) * 256;
    const int64_t mine = 2 * a + mc_exscan_ws_bytes(n) + 512;
    const int64_t win = mc_windows_workspace_bytes(n);             // unit counts, first-'M' indices, block totals, tags (windows.cu)
    return mine > win ? mine : win;
}
static inline uint32_t *ws_a(void *ws) { return reinterpret_cast<uint32_t *>(ws); }
static inline uint32_t *ws_b(void *ws, int64_t n) { return reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(ws) + ((n * 4 + 255) / 256) * 256); }
static inline void *ws_s(void *ws, int64_t n) { return reinterpret_cast<uint8_t *>(ws) + 2 * (((n * 4 + 255) / 256) * 256); }

namespace {

// ---- stage 2: gather records into file order ----------------------------------------------------------------
// Stage 1 hands over two tables: per chunk {first record slot, count | filler flag << 16 | state << 17} and per RUN of
// consecutive chunks (one warp parsed them in order) {records of the run, filler flag | state of the run's last kept
// line << 1}.  The order of the records is fixed run by run: only the ~n_chunks / 128 run entries are prefix-summed, a
// warp then walks its run's chunk entries (most are empty in sparse mode) and copies the records.
//
// Stage 1 records the first kept line of a run blindly because the line before it belongs to another warp.  With all
// runs done the predecessor is known (every run reports the state of its last kept line): the record is dropped unless
// the previous kept line was a candidate (or there is none, so the first kept line of the text stays: it may close a
// window handed over by the caller).
__global__ void __launch_bounds__(256) k_run_resolve(uint32_t *__restrict__ run_tab, int64_t n_runs, uint32_t *__restrict__ cnt_clean,
                                                    const unsigned long long *__restrict__ scan_counters, unsigned long long rec_in_cap) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_runs) return;
    // stage 1 ran out of record slots: its buffer has unwritten records.  Nothing is ordered (zero records come out), the
    // caller sees the overflow in the counters and runs the chunk again with a larger buffer.
    if (scan_counters && (scan_counters[MC_C_OVERFLOW] != 0ull || scan_counters[MC_C_RECORDS] > rec_in_cap)) {
        cnt_clean[r] = 0u;
        return;
    }
    uint32_t count = run_tab[2 * r];
    const uint32_t v = run_tab[2 * r + 1];
    if (v & 1u) {
        int64_t p = r - 1;
        uint32_t st = 0u;
        while (p >= 0 && (st = (run_tab[2 * p + 1] >> 1) & 3u) == 0u) --p;
        if (p >= 0 && st == 1u && count > 0u) {
            run_tab[2 * r + 1] = v | 0x80000000u;           // the gather skips the filler (first record of its chunk)
            --count;
        }
    }
    cnt_clean[r] = count;
}

// A warp owns a run: it reads the run's chunk entries (lane j <-> j-th chunk, 32 at a time), prefix-sums their counts and
// then takes the run's records 32 at a time, ONE LANE PER RECORD: the raw record is fetched from stage 1's buffer,
// finished (mc_finish_record_win, parse.cuh: columns from the field-start bits stage 1 left in the record, event index,
// np.round(event_mean - model_mean, 4), k-mer equality, read-name span), given the target bits of its k-mer on both
// strands (meth_ref[pos:pos+k], extract_contexts.py:176) and the read-change flag against the record before it in the
// run (MC_RF_NEWREAD: one shuffle, both lines still in L1), and written to its place in file order.  The first record of
// a run leaves the flag to stage 3 (its predecessor belongs to another warp).
__global__ void __launch_bounds__(256, 4) k_gather_finish(const uint8_t *__restrict__ text, int64_t limit, mc_refindex R,
                                                      const uint32_t *__restrict__ tile_tab, const uint32_t *__restrict__ run_tab,
                                                      const uint32_t *__restrict__ run_dst, int64_t n_tiles, int64_t n_runs, int run_len,
                                                      const mc_record *__restrict__ in, unsigned long long in_cap, mc_record *__restrict__ out,
                                                      unsigned long long out_cap, uint32_t *__restrict__ seg_flags,
                                                      uint32_t *__restrict__ run_first) {
    const int lane = threadIdx.x & 31;
    // warps stride over the runs (a resident grid): a warp whose run is empty moves on to its next run at once instead of
    // leaving a hole in its CTA until the CTA's longest run is done
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t run = warp0; run < n_runs; run += n_warps) {
    const uint32_t rv = __ldg(run_tab + 2 * run + 1);
    const bool empty_run = __ldg(run_dst + run) == __ldg(run_dst + run + 1);       // after the filler drop
    if (run_first && lane == 0) run_first[run] = empty_run ? 0xFFFFFFFFu : __ldg(run_dst + run);
    if (__ldg(run_tab + 2 * run) == 0u) continue;                // nothing recorded in this run
    const bool drop = (rv >> 31) != 0u;
    unsigned long long d_run = __ldg(run_dst + run);
    const int64_t c0 = run * run_len, c1 = min(c0 + (int64_t)run_len, n_tiles);
    long long carry_line = -1;                                   // line / name span of the last record written (-1: none yet)
    uint32_t carry_span = 0u;
    for (int64_t cb = c0; cb < c1; cb += 32) {
        const int64_t c = cb + lane;
        unsigned long long src = 0ull;
        uint32_t cnt = 0u;
        if (c < c1) {
            const uint2 e = __ldg(reinterpret_cast<const uint2 *>(tile_tab) + c);
            src = e.x;
            cnt = e.y & 0xFFFFu;
            if (drop && ((e.y >> 16) & 1u) && cnt > 0u) { src += 1ull; --cnt; }     // the filler is the first record of its chunk
        }
        uint32_t incl = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        const uint32_t excl = incl - cnt, tot = __shfl_sync(0xffffffffu, incl, 31);
        for (uint32_t k0 = 0; k0 < tot; k0 += 32) {
            const uint32_t idx = k0 + lane;
            const bool act = idx < tot;
            // owning chunk: the last lane whose exclusive prefix is <= idx (empty chunks share the prefix of the next
            // non-empty one and come before it, trailing ones have prefix == tot)
            int lo = 0, hi = 31;
#pragma unroll
            for (int st = 0; st < 5; ++st) {
                const int mid = (lo + hi + 1) >> 1;
                const uint32_t e_mid = __shfl_sync(0xffffffffu, excl, mid);
                if (e_mid <= idx) lo = mid; else hi = mid - 1;
            }
            const unsigned long long s_own = __shfl_sync(0xffffffffu, src, lo);
            const uint32_t e_own = __shfl_sync(0xffffffffu, excl, lo);
            const unsigned long long slot = s_own + (idx - e_own), dst = d_run + idx;
            const bool ok = act && slot < in_cap && dst < out_cap;     // else: dropped by a capacity overflow (redone by the host)
            alignas(16) mc_record r;
            long long line = -1;
            uint32_t span = 0u;
            if (ok) {
                const uint4 *sp = reinterpret_cast<const uint4 *>(in + slot);
                uint4 *dr = reinterpret_cast<uint4 *>(&r);
                dr[0] = __ldg(sp);
                dr[1] = __ldg(sp + 1);
                if (r.flags & MC_RF_RAW) mc_finish_record_win(text, limit, r);
                if (r.flags & MC_RF_CAND) {
                    const int cid = r.contig;
                    if (r.pos < __ldg(R.d_len + cid)) {
                        const int64_t g = __ldg(R.d_base + cid) + r.pos;
                        r.kbits_fwd = (uint8_t)mc_kmer_bits(R.d_site_fwd, g, R.k);
                        r.kbits_rev = (uint8_t)mc_kmer_bits(R.d_site_rev, g, R.k);
                    }
                }
                line = mc_rec_line(r);
                span = (uint32_t)r.name_off | ((uint32_t)r.name_len << 16);
            }
            // read name against the previous record of the run (same read <=> equal bytes, extract_contexts.py:161)
            long long pl = __shfl_up_sync(0xffffffffu, line, 1);
            uint32_t ps = __shfl_up_sync(0xffffffffu, span, 1);
            if (lane == 0) { pl = carry_line; ps = carry_span; }
            if (ok) {
                uint32_t sf = 1u;                                      // read-change flag for stage 3 (the first record of a run is
                                                                       // listed in run_first and decided there)
                if (pl >= 0) {
                    uint32_t fl = r.flags | MC_RF_SEGKNOWN;
                    sf = 0u;
                    if ((ps >> 16) != r.name_len || bytes_differ(text + pl + (ps & 0xFFFFu), text + line + r.name_off, r.name_len)) {
                        fl |= MC_RF_NEWREAD;
                        sf = 1u;
                    }
                    r.flags = (uint8_t)fl;
                }
                if (seg_flags) seg_flags[dst] = sf;
                uint4 *dp = reinterpret_cast<uint4 *>(out + dst);
                const uint4 *sr = reinterpret_cast<const uint4 *>(&r);
                dp[0] = sr[0];
                dp[1] = sr[1];
            }
            const int last = (int)min(tot - k0, 32u) - 1;
            carry_line = __shfl_sync(0xffffffffu, line, last);
            carry_span = __shfl_sync(0xffffffffu, span, last);
        }
        d_run += tot;
    }
    }
}

// ---- stage 3: read segmentation ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_seg_flags(const uint8_t *__restrict__ text, mc_record *__restrict__ rec, int64_t n_cap,
                                                  const unsigned long long *__restrict__ d_n, uint32_t *__restrict__ flags,
                                                  const uint32_t *__restrict__ known) {
    const int64_t n = mc_dev_count(d_n, n_cap);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (known) {                                                  // stage 2 left the answer for all but the first record of a run
        const uint32_t kf = known[i];
        if (kf < 2u) { flags[i] = kf; return; }
    }
    uint32_t f = 1u;
    const mc_record b = rec[i];
    if (b.flags & MC_RF_SEGKNOWN) {
        f = (b.flags & MC_RF_NEWREAD) ? 1u : 0u;                  // stage 1 compared the names while both lines were staged
    } else {
        // first record of a scan pass, neighbour of a raw record, or records that did not come through stage 1: compare the
        // read names in the text, and leave the answer in the record (the window builder reads it there).  Only the flag
        // byte of the own record is written; neighbours read this record's name span and line offset, never its flags.
        if (i > 0) {
            const mc_record a = rec[i - 1];
            if (a.name_len == b.name_len)
                f = bytes_differ(text + mc_rec_line(a) + a.name_off, text + mc_rec_line(b) + b.name_off, a.name_len) ? 1u : 0u;
        }
        rec[i].flags = (uint8_t)(b.flags | MC_RF_SEGKNOWN | (f ? MC_RF_NEWREAD : 0u));
    }
    flags[i] = f;
}

// With the flags of stage 2: only the first record of every run is still undecided (its predecessor was finished by
// another warp); one thread per run compares the two read names in the text and settles flag and record.
__global__ void __launch_bounds__(256) k_seg_fix(const uint8_t *__restrict__ text, mc_record *__restrict__ rec, const unsigned long long *__restrict__ d_n,
                                                int64_t n_cap, const uint32_t *__restrict__ run_first, int64_t n_runs, uint32_t *__restrict__ flags) {
    const int64_t run = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (run >= n_runs) return;
    const uint32_t i = run_first[run];
    if (i == 0xFFFFFFFFu || (int64_t)i >= mc_dev_count(d_n, n_cap)) return;
    uint32_t f = 1u;
    const mc_record b = rec[i];
    if (i > 0u) {
        const mc_record a = rec[i - 1];
        if (a.name_len == b.name_len)
            f = bytes_differ(text + mc_rec_line(a) + a.name_off, text + mc_rec_line(b) + b.name_off, a.name_len) ? 1u : 0u;
    }
    rec[i].flags = (uint8_t)(b.flags | MC_RF_SEGKNOWN | (f ? MC_RF_NEWREAD : 0u));
    flags[i] = f;
}

__global__ void __launch_bounds__(256) k_seg_starts(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ excl, int64_t n_cap,
                                                   const unsigned long long *__restrict__ d_n, uint32_t *__restrict__ seg_start,
                                                   const unsigned long long *__restrict__ d_nseg) {
    const int64_t n = mc_dev_count(d_n, n_cap);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && flags[i]) seg_start[excl[i]] = (uint32_t)i;
    if (i == 0) seg_start[*d_nseg] = (uint32_t)n;
}

// ---- stage 4: quality lookup -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_seg_quality(const uint8_t *__restrict__ text, const mc_record *__restrict__ rec,
                                                    const uint32_t *__restrict__ seg_start, int64_t seg_cap,
                                                    const unsigned long long *__restrict__ d_nseg,
                                                    const mc_qual_entry *__restrict__ table, unsigned long long mask,
                                                    double *__restrict__ seg_qual, unsigned long long *__restrict__ d_err) {
    const int64_t n_seg = mc_dev_count(d_nseg, seg_cap);
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const mc_record r = rec[seg_start[s]];
    const mc_read_key key = mc_read_key_of(text + mc_rec_line(r) + r.name_off, r.name_len);
    double q = __longlong_as_double(0x7ff8000000000000ll);   // NaN = missing
    unsigned long long slot = key.hash & mask;
    for (unsigned long long probe = 0; probe <= mask; ++probe) {
        const mc_qual_entry e = table[slot];
        if (e.hash == 0ull) break;
        if (e.hash == key.hash && e.check == key.check && e.len == key.len) { q = e.qual; break; }
        slot = (slot + 1) & mask;
    }
    if (q != q) atomicAdd(d_err, 1ull);
    seg_qual[s] = q;
}

}  // namespace

extern "C" int mc_order_records(const uint8_t *d_text, int64_t nbytes, const mc_refindex *ref, const uint32_t *d_tile_tab, int64_t n_tiles,
                                uint32_t *d_run_tab, int run_len, const mc_record *d_rec_in, int64_t rec_in_cap,
                                const uint64_t *d_scan_counters, mc_record *d_rec_out, int64_t rec_out_cap, uint64_t *d_n_out,
                                uint32_t *d_seg_flags, uint32_t *d_run_first, void *d_ws, void *stream) {
    MC_REQUIRE(!d_seg_flags == !d_run_first, "d_seg_flags and d_run_first go together");
    MC_REQUIRE(d_text && ref && d_tile_tab && d_run_tab && d_rec_in && d_rec_out && d_n_out && d_ws, "null pointer");
    MC_REQUIRE(run_len >= 1, "run length must be >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_tiles <= 0) {
        MC_CUDA_CHECK(cudaMemsetAsync(d_n_out, 0, 8, st));
        return MC_OK;
    }
    const int64_t n_runs = (n_tiles + run_len - 1) / run_len;
    uint32_t *cnt = ws_a(d_ws), *dst = ws_b(d_ws, n_runs + 1);
    MC_CUDA_CHECK(cudaMemsetAsync(cnt + n_runs, 0, 4, st));
    k_run_resolve<<<(unsigned)((n_runs + 255) / 256), 256, 0, st>>>(d_run_tab, n_runs, cnt, reinterpret_cast<const unsigned long long *>(d_scan_counters),
                                                                   (unsigned long long)rec_in_cap);
    MC_LAUNCH_CHECK();
    int rc = mc_exscan_u32(cnt, dst, n_runs + 1, nullptr, d_n_out, ws_s(d_ws, n_runs + 1), st);     // entry n_runs (count 0) = the total
    if (rc) return rc;
    int64_t gf_blocks = (n_runs * 32 + 255) / 256;
    {
        int dev = 0, sms = 0;
        MC_CUDA_CHECK(cudaGetDevice(&dev));
        MC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        const int64_t resident = (int64_t)sms * 4;                 // __launch_bounds__(256, 4)
        if (gf_blocks > resident) gf_blocks = resident;
    }
    k_gather_finish<<<(unsigned)gf_blocks, 256, 0, st>>>(d_text, nbytes + MC_TEXT_PAD - 64, *ref, d_tile_tab, d_run_tab, dst, n_tiles,
                                                                          n_runs, run_len, d_rec_in, (unsigned long long)rec_in_cap, d_rec_out,
                                                                          (unsigned long long)rec_out_cap, d_seg_flags, d_run_first);
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_segment_reads(const uint8_t *d_text, mc_record *d_rec, const uint64_t *d_n_records, int64_t rec_cap,
                                uint32_t *d_seg_flags, const uint32_t *d_run_first, int64_t n_runs, uint32_t *d_seg_start, uint64_t *d_nseg,
                                void *d_ws, void *stream) {
    MC_REQUIRE(d_text && d_rec && d_n_records && d_seg_start && d_nseg && d_ws, "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (rec_cap <= 0) {
        MC_CUDA_CHECK(cudaMemsetAsync(d_nseg, 0, 8, st));
        MC_CUDA_CHECK(cudaMemsetAsync(d_seg_start, 0, 4, st));
        return MC_OK;
    }
    uint32_t *flags = ws_a(d_ws), *excl = ws_b(d_ws, rec_cap);
    const unsigned nb = (unsigned)((rec_cap + 255) / 256);
    const unsigned long long *dn = reinterpret_cast<const unsigned long long *>(d_n_records);
    if (d_seg_flags && d_run_first) {
        // stage 2 decided every record but the first of each run: settle those, the flag array is then complete
        flags = d_seg_flags;
        if (n_runs > 0) k_seg_fix<<<(unsigned)((n_runs + 255) / 256), 256, 0, st>>>(d_text, d_rec, dn, rec_cap, d_run_first, n_runs, flags);
    } else {
        k_seg_flags<<<nb, 256, 0, st>>>(d_text, d_rec, rec_cap, dn, flags, nullptr);
    }
    MC_LAUNCH_CHECK();
    int rc = mc_exscan_u32(flags, excl, rec_cap, d_n_records, d_nseg, ws_s(d_ws, rec_cap), st);
    if (rc) return rc;
    k_seg_starts<<<nb, 256, 0, st>>>(flags, excl, rec_cap, dn, d_seg_start, reinterpret_cast<const unsigned long long *>(d_nseg));
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_segment_quality(const uint8_t *d_text, const mc_record *d_rec, const uint32_t *d_seg_start, const uint64_t *d_nseg,
                                  int64_t seg_cap, const mc_qual_entry *d_table, int64_t table_size, double *d_seg_qual,
                                  uint64_t *d_err, void *stream) {
    MC_REQUIRE(d_text && d_rec && d_seg_start && d_nseg && d_table && d_seg_qual && d_err, "null pointer");
    MC_REQUIRE(table_size > 0 && (table_size & (table_size - 1)) == 0, "table size must be a power of two");
    if (seg_cap <= 0) return MC_OK;
    k_seg_quality<<<(unsigned)((seg_cap + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        d_text, d_rec, d_seg_start, seg_cap, reinterpret_cast<const unsigned long long *>(d_nseg), d_table,
        (unsigned long long)(table_size - 1), d_seg_qual, reinterpret_cast<unsigned long long *>(d_err));
    MC_LAUNCH_CHECK();
    return MC_OK;
}
