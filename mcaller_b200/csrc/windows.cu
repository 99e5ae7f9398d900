// Stage 5 (K2): context-window builder -- the state machine of the reference's extract_features
// (extract_contexts.py:169-291) run per read segment over the stage-1 records.
//
// Why this is enough: a kept line whose k-mer holds no 'M' leaves the reference's state machine closed and
// empty (:242-245 / :289-291), and stage 1 records every line that can hold an 'M' on either strand plus the
// kept line that follows it (the line that closes an open window, :179).  Unrecorded lines are therefore no-ops
// and the state machine can run on the records alone.  State never crosses a read boundary except for the one
// still-open window of the previous read, which the first record of the next read closes (:179, `read_name !=
// last_read`); that hand-off is resolved here by looking at the first record of the next segment.
//
// Parallel decomposition: a read is cut into UNITS.  A record that is not a candidate (its k-mer touches no target on
// either strand) leaves the state machine closed and empty (:242-245, :289-291), so the records from the first candidate
// after such a record up to and including the next non-candidate record (the closer) can be processed on their own; the
// only read-level state they need is `last_read` / `first_read_ind` (:161-174), i.e. the read's first line with an 'M',
// which k_first_m finds per read beforehand.  Reads whose first record lies within k of the contig start stay one unit:
// a window at position 0 never closes (`if mpos and`, :179) and keeps its columns across non-candidate lines.
//
// A block of 256 threads owns WIN_RECS consecutive records.  It STAGES them in shared memory with coalesced loads (the
// fields the state machine reads: position, event index, flags, the k-mer's target bits on both strands that stage 1
// left in the record, contig; the write pass also the float64 deviation), compacts the unit starts among them and runs
// one thread per unit through the literal state machine -- every per-record step is then a shared-memory read instead of
// a dependent global load.  Two passes (count rows / write rows) so rows land in file order.
//
// Column sums follow numpy (np.mean -> add.reduce) bit for bit.  Below 8 values numpy adds left to right, which is an
// online running sum: one float64 per column slot and thread in shared memory, updated as the lines go by (99 % of the
// columns).  The state machine also tags every fed record with the column slot it went to; a column that reaches 8 values
// (8 running lanes + tail up to 128, recursive halving above) is re-read from the staged records in file order when its
// window closes, so ANY number of events per column is handled; nothing lives in local memory.
#include "common.cuh"

namespace {

#ifndef MC_WIN_ITEMS
#define MC_WIN_ITEMS 12
#endif
#ifndef MC_WIN_THREADS
#define MC_WIN_THREADS 128
#endif
#ifndef MC_WIN_BLOCKS
#define MC_WIN_BLOCKS 4
#endif
constexpr int WIN_THREADS = MC_WIN_THREADS, WIN_ITEMS = MC_WIN_ITEMS, WIN_RECS = WIN_THREADS * WIN_ITEMS;   // 1536 records per block: ~115 units
constexpr int WIN_UNITS = WIN_RECS / 2 + 2;       // a unit holds a candidate and is followed by a non-candidate: <= ceil(n/2) units
static_assert(WIN_RECS < 65536, "unit / read counts of a block are packed in 16 bits");
constexpr uint32_t TAG_NONE = 0xFu;               // record fed no column

// ---- staged record: {pos, event_idx, flags | kbits_fwd << 8 | kbits_rev << 16 | tag << 24, contig} -----------------------
__device__ __forceinline__ uint4 stage_word(const mc_record *p) {
    const uint4 a = __ldg(reinterpret_cast<const uint4 *>(p)), b = __ldg(reinterpret_cast<const uint4 *>(p) + 1);
    return make_uint4(a.z, a.w, (b.w & 0x00FFFFFFu) | (TAG_NONE << 24), b.z >> 16);
}
__device__ __forceinline__ double stage_diff(const mc_record *p) {
    const uint4 b = __ldg(reinterpret_cast<const uint4 *>(p) + 1);
    return __longlong_as_double((long long)(((unsigned long long)b.y << 32) | b.x));
}

// events per column slot: 8 x 16 bits in two registers (slots 0-3 / 4-7), saturating at 65535 (flagged as MC_CE_COLUMN)
struct Counts {
    unsigned long long lo, hi;
};
__device__ __forceinline__ int cnt_get(const Counts &q, int c) { return (int)(((c < 4 ? q.lo : q.hi) >> (16 * (c & 3))) & 0xFFFFull); }
__device__ __forceinline__ void cnt_inc(Counts &q, int c) {
    if (cnt_get(q, c) < 65535) {
        const unsigned long long one = 1ull << (16 * (c & 3));
        if (c < 4) q.lo += one; else q.hi += one;
    }
}
__device__ __forceinline__ void cnt_clear(Counts &q, int c) {
    const unsigned long long m = ~(0xFFFFull << (16 * (c & 3)));
    if (c < 4) q.lo &= m; else q.hi &= m;
}
__device__ __forceinline__ int map_get(uint32_t mp, int c) { return (int)((mp >> (4 * c)) & 0xFu); }

__device__ __forceinline__ mc_record load_rec(const mc_record *p) {
    mc_record r;
    const uint4 *s = reinterpret_cast<const uint4 *>(p);
    uint4 a = __ldg(s), b = __ldg(s + 1);
    uint4 *d = reinterpret_cast<uint4 *>(&r);
    d[0] = a;
    d[1] = b;
    return r;
}

__device__ __forceinline__ uint8_t comp_base(uint8_t c) {
    switch (c) {
        case 'A': return 'T';
        case 'C': return 'G';
        case 'G': return 'C';
        case 'T': return 'A';
        case 'N': return 'N';
        default: return 0;
    }
}

// first line of each read with an 'M' under the per-line strand guess (:169-176): record index and event index
__global__ void __launch_bounds__(128) k_first_m(const mc_record *__restrict__ rec, const uint32_t *__restrict__ seg_start, int64_t seg_cap,
                                                const unsigned long long *__restrict__ d_nseg, uint32_t *__restrict__ first_idx,
                                                int32_t *__restrict__ first_ind) {
    const int64_t n_seg = mc_dev_count(d_nseg, seg_cap);
    const int64_t seg = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (seg >= n_seg) return;
    const uint32_t b = seg_start[seg], e = seg_start[seg + 1];
    uint32_t fi = 0xFFFFFFFFu;
    int32_t ev = 0;
    for (uint32_t i = b; i < e; ++i) {
        const uint4 c = __ldg(reinterpret_cast<const uint4 *>(rec + i) + 1);
        const uint32_t fl = c.w & 0xFFu;
        if (!(fl & MC_RF_CAND)) continue;
        const int rev = !(fl & MC_RF_EQ);
        const uint32_t bits = rev ? ((c.w >> 16) & 0xFFu) : ((c.w >> 8) & 0xFFu);      // 'M's of the k-mer on that strand (stage 1)
        if (bits) { fi = i; ev = (int32_t)__ldg(reinterpret_cast<const uint4 *>(rec + i)).w; break; }
    }
    first_idx[seg] = fi;
    first_ind[seg] = ev;
}

// spill arena for columns with more than 128 events (numpy's recursive halving needs random access to the values)
struct Spill {
    double *buf;
    unsigned long long cap;
    unsigned long long *cursor;
};

// where a unit finds the staged fields of record i: this block's shared memory, or global memory past the block's range
struct ColSrc {
    const uint4 *s_rec;
    const double *s_diff;
    const mc_record *rec;
    const uint8_t *g_tag;
    int64_t base;
};
__device__ __forceinline__ uint32_t cs_tag(const ColSrc &S, uint32_t i) {
    const int64_t j = (int64_t)i - S.base;
    return (j >= 0 && j < WIN_RECS) ? (S.s_rec[j].z >> 24) : (uint32_t)S.g_tag[i];
}
__device__ __forceinline__ double cs_diff(const ColSrc &S, uint32_t i) {
    const int64_t j = (int64_t)i - S.base;
    return (j >= 0 && j < WIN_RECS) ? S.s_diff[j] : stage_diff(S.rec + i);
}
// np.add.reduce of a column with 8 or more values (rare: P(8+ events on one position) < 1 %), kept out of line so the
// common path stays small: 8 running lanes + sequential tail up to 128 values, recursive halving above
__device__ __noinline__ double col_sum_big(const ColSrc S, uint32_t src, uint32_t unit_b, uint32_t upto, int n, Spill spill, uint32_t *err) {
    // the column's current contents are the last n records before `upto` that carry its tag (older ones with the same tag
    // belong to an earlier window whose column was cleared since)
    uint32_t f0 = upto;
    for (int need = n; need > 0 && f0 > unit_b;) {
        --f0;
        if (cs_tag(S, f0) == src) --need;
    }
    if (n >= 65535) { *err |= MC_CE_COLUMN; return 0.0; }          // counter saturated: the span is not known
    double res = 0.0;
    if (n <= 128) {
        double r[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) r[q] = 0.0;
        const int full = n - (n % 8);
        int t = 0;
        uint32_t j = f0;
        for (; j < upto && t < full; ++j) {
            if (cs_tag(S, j) != src) continue;
            const double v = cs_diff(S, j);
            // element t of the column goes to running lane t % 8 (the first eight start the lanes)
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if ((t & 7) == q) r[q] = t < 8 ? v : __dadd_rn(r[q], v);
            ++t;
        }
        res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
        for (; j < upto; ++j)
            if (cs_tag(S, j) == src) res = __dadd_rn(res, cs_diff(S, j));
        return res;
    }
    // more than 128 events in one column (a stalled read): numpy halves recursively, which needs the values side by side
    // -> gather them into the spill arena
    const unsigned long long at = atomicAdd(spill.cursor, (unsigned long long)n);
    if (at + (unsigned long long)n > spill.cap) { *err |= MC_CE_COLUMN; return 0.0; }
    double *a = spill.buf + at;
    int t = 0;
    for (uint32_t j = f0; j < upto; ++j)
        if (cs_tag(S, j) == src) a[t++] = cs_diff(S, j);
    return mc_pairwise_sum([a](int64_t q) { return a[q]; }, 0, n);
}

template <bool WRITE>
__global__ void __launch_bounds__(WIN_THREADS, MC_WIN_BLOCKS)
k_windows(const mc_record *__restrict__ rec, int64_t rec_cap, const unsigned long long *__restrict__ d_n_records,
          const uint32_t *__restrict__ seg_start, int64_t seg_cap, const unsigned long long *__restrict__ d_nseg,
          const double *__restrict__ seg_qual, const uint32_t *__restrict__ first_idx, const int32_t *__restrict__ first_ind_arr,
          mc_refindex R, int skip_thresh, double qual_thresh, int two_models, mc_call *__restrict__ calls,
          unsigned long long call_cap, uint32_t *__restrict__ unit_cnt /* [n_records], written at unit starts */,
          uint32_t *__restrict__ blk_tot, const uint32_t *__restrict__ blk_off, uint8_t *__restrict__ g_tag /* [n_records] */, Spill spill) {
    __shared__ uint32_t s_unit[WIN_UNITS];        // record index of each unit start of the block, in record order
    __shared__ uint32_t s_off[WIN_UNITS];         // write pass: row offset of each unit
    __shared__ uint16_t s_seg[WIN_UNITS];         // read segment of each unit, relative to the block's first record's
    __shared__ int s_warp[WIN_THREADS / 32 + 1];
    __shared__ int64_t s_seg0;
    // [WIN_RECS] staged records, then (write pass) [WIN_RECS] float64 deviations and [MC_MAXK][WIN_THREADS] running column sums
    extern __shared__ __align__(16) uint4 s_dyn[];
    uint4 *s_rec = s_dyn;
    double *s_diff = reinterpret_cast<double *>(s_dyn + WIN_RECS);
    double *s_seq = s_diff + WIN_RECS + threadIdx.x;              // this thread's slice: element [slot] at s_seq[slot * WIN_THREADS]
    const int k = R.k;
    // the record / segment counts live on the device; the grid was sized for rec_cap records
    const int64_t n_records = mc_dev_count(d_n_records, rec_cap), n_seg = mc_dev_count(d_nseg, seg_cap);
    const int64_t base = (int64_t)blockIdx.x * WIN_RECS;
    if (base >= n_records || n_seg <= 0) {                        // block-uniform
        if (!WRITE && threadIdx.x == 0) blk_tot[blockIdx.x] = 0u;
        return;
    }
    // ---- stage the block's records (coalesced: a warp reads 32 consecutive records) ------------------------------------------
    for (int j = threadIdx.x; j < WIN_RECS; j += WIN_THREADS) {
        const int64_t i = base + j;
        if (i < n_records) {
            s_rec[j] = stage_word(rec + i);
            if (WRITE) s_diff[j] = stage_diff(rec + i);
        } else {
            s_rec[j] = make_uint4(0u, 0u, TAG_NONE << 24, 0u);
        }
    }
    if (threadIdx.x == 0) {                       // segment of the block's first record: last segment starting at or before it
        int64_t lo = 0, hi = n_seg - 1;
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if ((int64_t)__ldg(seg_start + mid) <= base) lo = mid; else hi = mid - 1;
        }
        s_seg0 = lo;
    }
    __syncthreads();
    // staged view of record i (this block's range) or a global read (a unit that runs past the block's last record)
    auto rec_word = [&](uint32_t i) -> uint4 {
        const int64_t j = (int64_t)i - base;
        return (j >= 0 && j < WIN_RECS) ? s_rec[j] : stage_word(rec + i);
    };
    auto rec_diff = [&](uint32_t i) -> double {
        const int64_t j = (int64_t)i - base;
        return (WRITE && j >= 0 && j < WIN_RECS) ? s_diff[j] : stage_diff(rec + i);
    };
    auto tag_set = [&](uint32_t i, uint32_t t) {
        const int64_t j = (int64_t)i - base;
        if (j >= 0 && j < WIN_RECS) s_rec[j].z = (s_rec[j].z & 0x00FFFFFFu) | (t << 24);
        else g_tag[i] = (uint8_t)t;
    };
    auto tag_get = [&](uint32_t i) -> uint32_t {
        const int64_t j = (int64_t)i - base;
        return (j >= 0 && j < WIN_RECS) ? (s_rec[j].z >> 24) : (uint32_t)g_tag[i];
    };
    // ---- unit starts among this block's records, compacted in record order ------------------------------------------------
    int nu;
    {
        const int j0 = threadIdx.x * WIN_ITEMS;
        const int64_t i0 = base + j0;
        uint32_t prev_cand = 0u;
        if (i0 > 0 && i0 <= n_records)
            prev_cand = (j0 > 0 ? s_rec[j0 - 1].z : __ldg(reinterpret_cast<const uint4 *>(rec + i0 - 1) + 1).w) & MC_RF_CAND;
        uint32_t umask = 0u, nmask = 0u;          // unit starts / read starts among this thread's records
#pragma unroll
        for (int j = 0; j < WIN_ITEMS; ++j) {
            const int64_t i = i0 + j;
            if (i < n_records) {
                const uint4 w = s_rec[j0 + j];
                const uint32_t fl = w.z & 0xFFu;
                const uint32_t cand = fl & MC_RF_CAND;
                bool u;
                if (i == 0 || (fl & MC_RF_NEWREAD)) {
                    if (i != base) nmask |= 1u << j;
                    u = cand != 0u;
                    if (!u) u = (int)w.x < k;                     // whole-read unit (see above)
                } else {
                    u = cand != 0u && prev_cand == 0u;
                }
                if (u) umask |= 1u << j;
                prev_cand = cand;
            }
        }
        int total;
        const int off = mc_block_exscan<WIN_THREADS>(__popc(umask) | (__popc(nmask) << 16), s_warp, total);
        int ou = off & 0xFFFF;
        const int on = off >> 16;
        for (uint32_t m = umask; m; m &= m - 1u) {
            const int j = __ffs(m) - 1;
            if (ou < WIN_UNITS) {
                s_unit[ou] = (uint32_t)(i0 + j);
                s_seg[ou] = (uint16_t)(on + __popc(nmask & ((2u << j) - 1u)));
            }
            ++ou;
        }
        nu = total & 0xFFFF;
        if (nu > WIN_UNITS) nu = WIN_UNITS;       // cannot happen (see WIN_UNITS)
        __syncthreads();
    }
    if (WRITE) {
        // row offsets of the block's units: counts of the first pass -> exclusive prefix in shared memory
        constexpr int UPT = (WIN_UNITS + WIN_THREADS - 1) / WIN_THREADS;          // units per thread in the prefix
        uint32_t v[UPT];
        int sum = 0;
#pragma unroll
        for (int j = 0; j < UPT; ++j) {
            const int u = threadIdx.x * UPT + j;
            v[j] = u < nu ? unit_cnt[s_unit[u]] : 0u;
            sum += (int)v[j];
        }
        int total;
        uint32_t run = blk_off[blockIdx.x] + (uint32_t)mc_block_exscan<WIN_THREADS>(sum, s_warp, total);
#pragma unroll
        for (int j = 0; j < UPT; ++j) {
            const int u = threadIdx.x * UPT + j;
            if (u < WIN_UNITS) s_off[u] = run;
            run += v[j];
        }
        __syncthreads();
    }
    int my_rows = 0;
    for (int un = threadIdx.x; un < nu; un += WIN_THREADS) {
    const uint32_t b = s_unit[un];
    const int64_t seg = s_seg0 + s_seg[un];
    const uint32_t seg_b = __ldg(seg_start + seg), e_read = __ldg(seg_start + seg + 1);
    const bool whole = (int)rec_word(seg_b).x < k;             // the read is one unit
    uint32_t n_out = 0;
    const double myq = seg_qual[seg];
    if (myq < qual_thresh || (whole && b != seg_b)) {          // whole read dropped (:167) / unit covered by the whole-read unit
        if (!WRITE) unit_cnt[b] = 0u;
        continue;
    }
    uint32_t e = e_read;
    uint32_t out_pos = WRITE ? s_off[un] : 0u;
    const uint32_t fidx = __ldg(first_idx + seg);

    Counts cnts{0ull, 0ull};                       // events per column slot
    uint32_t mp = 0x76543210u;                     // window column -> column slot (the multi-M carry permutes it)
    bool started = b > fidx;     // read_name == last_read  (this read already had a line with 'M')
    bool has_mpos = false;
    int mpos = 0, first_ind = started ? __ldg(first_ind_arr + seg) : 0, last_rev = 0, last_cid = 0;
    uint32_t name_rec = b;
    uint32_t sticky_err = 0u;

#define MPOS_TRUTHY (has_mpos && mpos != 0)

    // np.mean of the values that column slot `src` holds when the window closes at record `upto` (exclusive), summed like
    // numpy's add.reduce
    auto col_mean = [&](int src, uint32_t upto, uint32_t &err) -> double {
        const int n = cnt_get(cnts, src);
        double res;
        if (n < 8) res = s_seq[src * WIN_THREADS];                 // numpy adds fewer than 8 values left to right: the running sum
        else {
            const ColSrc S{s_rec, s_diff, rec, g_tag, base};
            res = col_sum_big(S, (uint32_t)src, b, upto, n, spill, &err);
        }
        return __ddiv_rn(res, (double)n);
    };

    // emits the row(s) for the open window; `close_idx` = ordered index of the closing record (or ~0u); the window holds the
    // records before `upto`
    auto emit_window = [&](uint32_t close_idx, int chrom_cid, uint32_t upto) {
        int n_empty = 0;
        for (int c = 0; c < k; ++c) n_empty += (cnt_get(cnts, map_get(mp, c)) == 0);
        if (WRITE) {
            if (out_pos < call_cap) {
                mc_call &o = calls[out_pos];
                const mc_record nr = load_rec(rec + name_rec);
                o.read_off = mc_rec_line(nr) + nr.name_off;
                o.read_len = nr.name_len;
                o.prob = 0.0;
                o.mpos = mpos;
                o.close_rec = close_idx;
                o.win_contig = (uint16_t)last_cid;
                o.chrom_contig = (uint16_t)(chrom_cid < 0 ? 0xFFFF : chrom_cid);
                o.rev = (uint8_t)last_rev;
                o.n_empty = (uint8_t)n_empty;
                o.label = 0;
                o.pad0 = 0;
                o.seg = (uint32_t)seg;
                o.pad1 = 0;
                o.pad2 = 0;
                uint32_t err = sticky_err;
                uint32_t empty_mask = 0u;
                const int64_t g = __ldg(R.d_base + last_cid) + mpos;
                // dense site slot = rank of the target among the strand's sites
                {
                    const uint32_t *bm = last_rev ? R.d_site_rev : R.d_site_fwd;
                    const uint32_t *rk = last_rev ? R.d_rank_rev : R.d_rank_fwd;
                    const uint32_t wbits = __ldg(bm + (g >> 5));
                    o.site = (int32_t)(__ldg(rk + (g >> 5)) + __popc(wbits & ((1u << (g & 31)) - 1u)));
                }
                if (n_empty <= skip_thresh) {
                    o.kind = MC_CALL;
                    for (int c = 0; c < k; ++c) {                 // :186-188 (forward reads are flipped)
                        const int src = map_get(mp, last_rev ? c : (k - 1 - c));
                        if (cnt_get(cnts, src) == 0) { o.feat[c] = 0.0; empty_mask |= 1u << c; }
                        else o.feat[c] = col_mean(src, upto, err);
                    }
                    o.feat[k] = myq;                              // :189-193
                    for (int c = k + 1; c <= MC_MAXK; ++c) o.feat[c] = 0.0;
                    // context bounds (:194-195) and base after the target (:197, base_models :99-106)
                    const int clen = __ldg(R.d_len + last_cid);
                    uint8_t nextb = 0;
                    if (mpos - k + 1 < 0 || mpos + k > clen) err |= MC_CE_CONTEXT;
                    else if (k < 2) {
                        // the key context[k-1:k+1] of a one-letter context has one letter: KeyError in base_models
                        // (nextb stays 0, which the check below flags as MC_CE_MODELKEY)
                    } else if (!last_rev) {
                        const int64_t gn = g + 1;
                        nextb = ((__ldg(R.d_site_fwd + (gn >> 5)) >> (gn & 31)) & 1u) ? 'M' : __ldg(R.d_bases + gn);
                    } else {
                        const int64_t gn = g - 1;
                        nextb = ((__ldg(R.d_site_rev + (gn >> 5)) >> (gn & 31)) & 1u) ? 'M' : comp_base(__ldg(R.d_bases + gn));
                    }
                    if (!(err & MC_CE_CONTEXT) &&
                        !(nextb == 'A' || nextb == 'C' || nextb == 'G' || nextb == 'T' || nextb == 'M'))
                        err |= MC_CE_MODELKEY;
                    o.model_sel = (uint8_t)((two_models && nextb == 'G') ? 1 : 0);
                } else {
                    o.kind = MC_TOO_MANY_SKIPS;                   // :238-239
                    for (int c = 0; c <= MC_MAXK; ++c) o.feat[c] = 0.0;
                    o.model_sel = 0;
                }
                o.empty_mask = (uint8_t)empty_mask;
                o.err = (uint8_t)err;
            }
            ++out_pos;
        }
        ++n_out;
    };
    auto emit_multi = [&]() {
        if (WRITE) {
            if (out_pos < call_cap) {
                mc_call &o = calls[out_pos];
                const mc_record nr = load_rec(rec + name_rec);
                o.read_off = mc_rec_line(nr) + nr.name_off;
                o.read_len = nr.name_len;
                o.prob = 0.0;
                for (int c = 0; c <= MC_MAXK; ++c) o.feat[c] = 0.0;
                o.mpos = mpos;
                o.site = -1;
                o.close_rec = 0u;
                o.win_contig = (uint16_t)last_cid;
                o.chrom_contig = (uint16_t)last_cid;
                o.kind = MC_MULTI_M;
                o.rev = (uint8_t)last_rev;
                o.n_empty = 0; o.empty_mask = 0; o.model_sel = 0; o.label = 0; o.err = 0; o.pad0 = 0;
                o.seg = (uint32_t)seg;
                o.pad1 = 0;
                o.pad2 = 0;
            }
            ++out_pos;
        }
        ++n_out;
    };
    auto reset_cols = [&]() { cnts.lo = 0ull; cnts.hi = 0ull; };

    // The row-producing code (column means, divisions, context look-ups) is by far the heaviest path and a lane needs it
    // only once per ~20 records.  Run in rounds so the warp executes it together: each lane advances through its records
    // until it reaches a window close (or its end-of-read hand-off), then all lanes that have one emit, then the next round.
    // a record the unit steps over beyond the block's staged range has its tag in global memory: start it as 'fed no column'
    auto tag_init = [&](uint32_t q) {
        if (WRITE && (int64_t)q - base >= WIN_RECS) g_tag[q] = (uint8_t)TAG_NONE;
    };
    uint32_t i = b;
    uint4 r = (b < e) ? rec_word(b) : make_uint4(0u, 0u, 0u, 0u);
    if (b < e) tag_init(b);
    auto advance = [&]() {
        ++i;
        if (i < e) { r = rec_word(i); tag_init(i); }
    };
    int rev = 0, first_m = -1, cid = 0, pos = 0;
    bool pending_close = false, handoff_done = false;
    // part of a record's processing after the close decision: feed or reset (:269-291)
    auto feed = [&]() {
        if (first_m >= 0) {                                        // :269-287
            if (MPOS_TRUTHY && rev != last_rev) has_mpos = false;  // columns kept (:276-277)
            if (!MPOS_TRUTHY) { has_mpos = true; mpos = pos + first_m; }
            started = true;
            last_rev = rev;
            last_cid = cid;
            name_rec = i;
            if (r.z & MC_RF_BADNUM) sticky_err |= MC_CE_BADNUM;
            const int slot = map_get(mp, first_m);
            if (WRITE) {
                // running left-to-right sum of the column (numpy starts from 0.0, which also turns a leading -0.0 into 0.0)
                const double v = rec_diff(i);
                double *q = s_seq + slot * WIN_THREADS;
                *q = __dadd_rn(cnt_get(cnts, slot) == 0 ? 0.0 : *q, v);
                tag_set(i, (uint32_t)slot);
            }
            cnt_inc(cnts, slot);
        } else if (MPOS_TRUTHY) {                                  // :289-291
            has_mpos = false;
            reset_cols();
        }
    };
    for (;;) {
        // ---- phase 1: advance to the next emission point ---------------------------------------------------------------
        while (!pending_close && i < e) {
            const uint32_t fl = r.z & 0xFFu;
            if (!whole && !(fl & MC_RF_CAND)) e = i + 1;           // the closer ends the unit
            const bool same_read = started;
            if (!same_read) {                                      // :161-162
                first_ind = (int)r.y;
                if (fl & MC_RF_BADIDX) sticky_err |= MC_CE_BADNUM;
            }
            if (!same_read) rev = !(fl & MC_RF_EQ);                // :169-174
            else {
                if (fl & MC_RF_BADIDX) sticky_err |= MC_CE_BADNUM;
                rev = !((int)r.y > first_ind);
            }
            cid = (int)r.w;
            pos = (int)r.x;
            const uint32_t bits = rev ? ((r.z >> 16) & 0xFFu) : ((r.z >> 8) & 0xFFu);   // 'M's of meth_ref[pos:pos+k] (:176), from stage 1
            first_m = bits ? (__ffs(bits) - 1) : -1;
            if (MPOS_TRUTHY && pos >= mpos + 1 && same_read) {     // :179 (the other-read case is the segment hand-off below)
                pending_close = true;
                break;
            }
            feed();
            advance();
        }
        // hand-off: a window still open at the end of the read is closed by the next kept line of the file, i.e. the
        // first record of the next segment that passes the quality filter (:179, read_name != last_read)
        const bool pending_handoff = !pending_close && i >= e && !handoff_done && MPOS_TRUTHY;
        if (!pending_close && !pending_handoff) break;
        // ---- phase 2: the lanes that reached an emission point emit together --------------------------------------------
        uint32_t close_idx = i;
        int chrom = cid;
        if (pending_handoff) {
            int64_t j = seg + 1;
            while (j < n_seg && seg_qual[j] < qual_thresh) ++j;
            if (j < n_seg) {
                close_idx = seg_start[j];
                chrom = load_rec(rec + close_idx).contig;
            } else {
                close_idx = 0xFFFFFFFFu;                           // pending: resolved by the next chunk, dropped at EOF
                chrom = -1;
            }
        }
        emit_window(close_idx, chrom, i);
        if (pending_handoff) {
            handoff_done = true;
            continue;
        }
        if (first_m < 0 || pos > mpos + skip_thresh + 1) {         // :242-245
            reset_cols();
            has_mpos = false;
        } else {                                                   // :246-256 multi-M carry
            if (first_m != 0) emit_multi();
            const int last_mpos = mpos;
            mpos = pos + first_m;
            int sp = mpos - last_mpos;
            if (sp > k) sp = k;
            if (sp <= 0) { sticky_err |= MC_CE_SPACING; sp = k; }
            uint32_t nmp = 0u;
            for (int c = 0; c < k; ++c) {
                int slot;
                if (c < sp) { slot = map_get(mp, k - sp + c); cnt_clear(cnts, slot); }
                else slot = map_get(mp, c - sp);
                nmp |= (uint32_t)slot << (4 * c);
            }
            mp = nmp | (mp & ~((k < 8) ? ((1u << (4 * k)) - 1u) : 0xFFFFFFFFu));
        }
        pending_close = false;
        feed();
        advance();
    }
    if (!WRITE) unit_cnt[b] = n_out;
    my_rows += (int)n_out;
#undef MPOS_TRUTHY
    }
    if (!WRITE) {
        __syncthreads();
        int total;
        (void)mc_block_exscan<WIN_THREADS>(my_rows, s_warp, total);
        if (threadIdx.x == 0) blk_tot[blockIdx.x] = (uint32_t)total;
    }
}

__global__ void k_check_cap(const unsigned long long *d_ncalls, unsigned long long cap, unsigned long long *d_flag) {
    if (d_ncalls[0] > cap) *d_flag = 1ull;
}

}  // namespace

extern "C" int64_t mc_windows_workspace_bytes(int64_t rec_cap) {
    if (rec_cap < 1) rec_cap = 1;
    auto up = [](int64_t bytes) { return ((bytes + 255) / 256) * 256; };
    const int64_t nb = (rec_cap + WIN_RECS - 1) / WIN_RECS;
    // [unit_cnt: u32 rec_cap][first_ind: i32 rec_cap][blk_tot, blk_off: u32 nb each][tags: u8 rec_cap][spill cursor][scan sums]
    return up(rec_cap * 4) + up(rec_cap * 4) + up(2 * nb * 4) + up(rec_cap) + 256 + mc_exscan_ws_bytes(nb) + 512;
}

extern "C" int mc_build_windows(const mc_record *d_rec, const uint64_t *d_n_records, int64_t rec_cap, const uint32_t *d_seg_start,
                                const uint64_t *d_nseg, int64_t seg_cap, const double *d_seg_qual, const mc_refindex *ref,
                                int skip_thresh, double qual_thresh, int two_models, mc_call *d_calls, int64_t call_cap,
                                uint32_t *d_seg_count, uint64_t *d_ncalls, void *d_ws, double *d_spill, int64_t spill_cap,
                                void *stream) {
    MC_REQUIRE(d_rec && d_n_records && d_seg_start && d_nseg && d_seg_qual && ref && d_calls && d_seg_count && d_ncalls && d_ws,
               "null pointer");
    MC_REQUIRE(ref->k >= 1 && ref->k <= MC_MAXK, "k out of range");
    MC_REQUIRE(skip_thresh >= 0, "skip_thresh must be >= 0");
    MC_REQUIRE(spill_cap == 0 || d_spill, "spill arena missing");
    cudaStream_t st = (cudaStream_t)stream;
    MC_CUDA_CHECK(cudaMemsetAsync(d_ncalls, 0, 16, st));
    if (seg_cap <= 0 || rec_cap <= 0) return MC_OK;
    MC_REQUIRE(rec_cap < (1ll << 32), "record count must fit 32 bits");
    if (seg_cap > rec_cap) seg_cap = rec_cap;                       // a segment holds at least one record
    const unsigned long long *dn = reinterpret_cast<const unsigned long long *>(d_n_records);
    const unsigned long long *ds = reinterpret_cast<const unsigned long long *>(d_nseg);
    const int64_t nb = (rec_cap + WIN_RECS - 1) / WIN_RECS;
    auto up = [](int64_t bytes) { return ((bytes + 255) / 256) * 256; };
    uint8_t *w = reinterpret_cast<uint8_t *>(d_ws);
    uint32_t *unit_cnt = reinterpret_cast<uint32_t *>(w);
    int32_t *first_ind = reinterpret_cast<int32_t *>(w + up(rec_cap * 4));
    uint32_t *blk_tot = reinterpret_cast<uint32_t *>(w + 2 * up(rec_cap * 4));
    uint32_t *blk_off = blk_tot + nb;
    uint8_t *tags = w + 2 * up(rec_cap * 4) + up(2 * nb * 4);
    unsigned long long *spill_cursor = reinterpret_cast<unsigned long long *>(tags + up(rec_cap));
    void *scan_ws = reinterpret_cast<uint8_t *>(spill_cursor) + 256;
    MC_CUDA_CHECK(cudaMemsetAsync(spill_cursor, 0, 8, st));
    const Spill spill{d_spill, (unsigned long long)spill_cap, spill_cursor};
    uint32_t *first_idx = d_seg_count;                             // caller's seg_cap-sized scratch
    k_first_m<<<(unsigned)((seg_cap + 127) / 128), 128, 0, st>>>(d_rec, d_seg_start, seg_cap, ds, first_idx, first_ind);
    MC_LAUNCH_CHECK();
    constexpr size_t rec_bytes = sizeof(uint4) * WIN_RECS, diff_bytes = sizeof(double) * (WIN_RECS + MC_MAXK * WIN_THREADS);
    MC_CUDA_CHECK(cudaFuncSetAttribute(k_windows<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rec_bytes));
    MC_CUDA_CHECK(cudaFuncSetAttribute(k_windows<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(rec_bytes + diff_bytes)));
    k_windows<false><<<(unsigned)nb, WIN_THREADS, rec_bytes, st>>>(d_rec, rec_cap, dn, d_seg_start, seg_cap, ds, d_seg_qual, first_idx, first_ind,
                                                          *ref, skip_thresh, qual_thresh, two_models, d_calls,
                                                          (unsigned long long)call_cap, unit_cnt, blk_tot, nullptr, tags, spill);
    MC_LAUNCH_CHECK();
    int rc = mc_exscan_u32(blk_tot, blk_off, nb, nullptr, d_ncalls, scan_ws, st);
    if (rc) return rc;
    k_windows<true><<<(unsigned)nb, WIN_THREADS, rec_bytes + diff_bytes, st>>>(d_rec, rec_cap, dn, d_seg_start, seg_cap, ds, d_seg_qual, first_idx,
                                                                  first_ind, *ref, skip_thresh, qual_thresh, two_models, d_calls,
                                                                  (unsigned long long)call_cap, unit_cnt, nullptr, blk_off, tags, spill);
    MC_LAUNCH_CHECK();
    k_check_cap<<<1, 1, 0, st>>>(reinterpret_cast<unsigned long long *>(d_ncalls), (unsigned long long)call_cap,
                                 reinterpret_cast<unsigned long long *>(d_ncalls) + 1);
    MC_LAUNCH_CHECK();
    return MC_OK;
}
