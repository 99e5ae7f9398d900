// FASTQ read-quality ingest on the GPU (SURVEY.md section 8f rank 1; reference read_qual.py:6-19):
// for every 4-line record, key = id.split(':')[0].split('_')[0] (id = first whitespace-delimited token after '@') and
// value = mean(ord(c) - 33) over the quality line; the results go straight into the open-addressing table that stage 4
// (mc_segment_quality) probes, so a run never builds a Python dict of a million reads.
//   k_fq_count : newlines per 4 KB tile                      (one pass over the bytes)
//   (exclusive scan over the tile counts)
//   k_fq_lines : byte offset of every line start            (second pass, ordered within the tile by a block scan)
//   k_fq_insert: one warp per record -- lanes stride over the quality line, one lane hashes the id and claims the slot;
//                duplicates resolve like the reference's dict: the last record of the file wins.
#include "common.cuh"

namespace {

constexpr int FQ_TILE = 4096;
constexpr int FQ_THREADS = 256;

__global__ void __launch_bounds__(FQ_THREADS) k_fq_count(const uint8_t *__restrict__ text, int64_t nbytes, uint32_t *__restrict__ tile_cnt) {
    __shared__ int s_warp[FQ_THREADS / 32 + 1];
    const int64_t base = (int64_t)blockIdx.x * FQ_TILE + (int64_t)threadIdx.x * 16;
    int c = 0;
    if (base < nbytes) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(text + base));       // caller pads the buffer to a multiple of 16
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t t = ((w[j] ^ 0x0a0a0a0au) & 0x7f7f7f7fu) + 0x7f7f7f7fu;
            uint32_t m = ~(t | w[j]) & 0x80808080u;
            const int64_t room = nbytes - (base + 4 * j);
            if (room < 4) m &= room <= 0 ? 0u : ((1u << (8 * room)) - 1u);
            c += __popc(m);
        }
    }
    int total;
    mc_block_exscan<FQ_THREADS>(c, s_warp, total);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = (uint32_t)total;
}

__global__ void __launch_bounds__(FQ_THREADS) k_fq_lines(const uint8_t *__restrict__ text, int64_t nbytes, const uint32_t *__restrict__ tile_off,
                                                        unsigned long long *__restrict__ line_start, unsigned long long cap) {
    __shared__ int s_warp[FQ_THREADS / 32 + 1];
    const int64_t base = (int64_t)blockIdx.x * FQ_TILE + (int64_t)threadIdx.x * 16;
    uint32_t nlm = 0u;
    if (base < nbytes) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(text + base));
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if (((w[j] >> (8 * b)) & 0xFFu) == 0x0au && base + 4 * j + b < nbytes) nlm |= 1u << (4 * j + b);
        }
    }
    int total;
    int idx = mc_block_exscan<FQ_THREADS>(__popc(nlm), s_warp, total);
    // line k+1 starts after newline k; line 0 starts at byte 0 (written by the host wrapper's memset + first thread)
    unsigned long long out = (unsigned long long)tile_off[blockIdx.x] + (unsigned)idx + 1ull;
    if (blockIdx.x == 0 && threadIdx.x == 0 && cap > 0) line_start[0] = 0ull;
    while (nlm) {
        const int b = __ffs(nlm) - 1;
        nlm &= nlm - 1u;
        if (out < cap) line_start[out] = (unsigned long long)(base + b + 1);
        ++out;
    }
}

__global__ void __launch_bounds__(256) k_fq_insert(const uint8_t *__restrict__ text, int64_t nbytes, const unsigned long long *__restrict__ line_start,
                                                  unsigned long long n_lines, mc_qual_entry *__restrict__ table, unsigned long long mask,
                                                  uint32_t *__restrict__ owner, double *__restrict__ rec_mean, unsigned long long *__restrict__ d_stats) {
    const unsigned long long rec = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const unsigned long long n_rec = n_lines / 4ull;
    if (rec >= n_rec) return;
    const unsigned long long h0 = line_start[4 * rec], h1 = line_start[4 * rec + 1];
    const unsigned long long q0 = line_start[4 * rec + 3];
    const unsigned long long q1 = line_start[4 * rec + 4];       // sentinel after the last line: see mc_fastq_quality
    // quality line without its '\n' (and '\r')
    long long qlen = (long long)(q1 - 1ull) - (long long)q0;
    if (qlen > 0 && __ldg(text + q0 + qlen - 1) == '\r') --qlen;
    unsigned long long sum = 0ull;
    for (long long j = lane; j < qlen; j += 32) sum += (unsigned long long)__ldg(text + q0 + j);
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, d);
    if (lane != 0) return;
    if (__ldg(text + h0) != '@') { atomicAdd(&d_stats[1], 1ull); return; }             // not a FASTQ header
    // id = first whitespace-delimited token after '@'; key = id up to the first ':' or '_'
    const mc_read_key key = mc_read_key_of(text + h0 + 1, (int64_t)(h1 - h0) - 1);
    const unsigned long long h = key.hash;
    const double mean = qlen > 0 ? __ddiv_rn((double)(sum - 33ull * (unsigned long long)qlen), (double)qlen)
                                 : __longlong_as_double(0x7ff8000000000000ll);          // np.mean([]) is nan
    rec_mean[rec] = mean;
    unsigned long long slot = h & mask;
    for (unsigned long long probe = 0; probe <= mask; ++probe) {
        unsigned long long *hp = reinterpret_cast<unsigned long long *>(&table[slot].hash);
        unsigned long long cur = *hp;
        if (cur == 0ull) {
            cur = atomicCAS(hp, 0ull, h);
            if (cur == 0ull) {                       // claimed: publish the rest of the key
                table[slot].check = key.check;
                table[slot].len = key.len;
                cur = h;
            }
        }
        if (cur == h) {
            // same 64-bit hash: treat as the same key (the check word is verified at lookup); last record wins
            atomicMax(&owner[slot], (uint32_t)rec + 1u);
            atomicAdd(&d_stats[0], 1ull);
            return;
        }
        slot = (slot + 1) & mask;
    }
    atomicAdd(&d_stats[2], 1ull);                    // table full
}

// every slot takes the mean of its owner = the last record of the file with that key (dict semantics of read_qual.py)
__global__ void __launch_bounds__(256) k_fq_publish(mc_qual_entry *__restrict__ table, unsigned long long mask, const uint32_t *__restrict__ owner,
                                                   const double *__restrict__ rec_mean) {
    const unsigned long long slot = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot > mask) return;
    const uint32_t o = owner[slot];
    if (o != 0u) table[slot].qual = rec_mean[o - 1u];
}

}  // namespace

extern "C" int64_t mc_fastq_tiles(int64_t nbytes) { return nbytes <= 0 ? 0 : (nbytes + FQ_TILE - 1) / FQ_TILE; }

extern "C" int mc_fastq_index(const uint8_t *d_text, int64_t nbytes, uint32_t *d_tile_cnt, uint32_t *d_tile_off, uint64_t *d_line_start,
                              int64_t line_cap, uint64_t *d_n_newlines, void *d_ws, void *stream) {
    MC_REQUIRE(d_text && d_tile_cnt && d_tile_off && d_line_start && d_n_newlines && d_ws, "null pointer");
    MC_REQUIRE((reinterpret_cast<uintptr_t>(d_text) & 15) == 0, "d_text must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nt = mc_fastq_tiles(nbytes);
    if (nt == 0) { MC_CUDA_CHECK(cudaMemsetAsync(d_n_newlines, 0, 8, st)); return MC_OK; }
    k_fq_count<<<(unsigned)nt, FQ_THREADS, 0, st>>>(d_text, nbytes, d_tile_cnt);
    MC_LAUNCH_CHECK();
    int rc = mc_exscan_u32(d_tile_cnt, d_tile_off, nt, nullptr, d_n_newlines, d_ws, st);
    if (rc) return rc;
    k_fq_lines<<<(unsigned)nt, FQ_THREADS, 0, st>>>(d_text, nbytes, d_tile_off, reinterpret_cast<unsigned long long *>(d_line_start),
                                                    (unsigned long long)line_cap);
    MC_LAUNCH_CHECK();
    return MC_OK;
}

extern "C" int mc_fastq_quality(const uint8_t *d_text, int64_t nbytes, const uint64_t *d_line_start, int64_t n_lines, mc_qual_entry *d_table,
                                int64_t table_size, uint32_t *d_owner, double *d_rec_mean, uint64_t *d_stats, void *stream) {
    MC_REQUIRE(d_text && d_line_start && d_table && d_owner && d_rec_mean && d_stats, "null pointer");
    MC_REQUIRE(table_size > 0 && (table_size & (table_size - 1)) == 0, "table size must be a power of two");
    const int64_t n_rec = n_lines / 4;
    if (n_rec <= 0) return MC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t threads = n_rec * 32;
    k_fq_insert<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(d_text, nbytes, reinterpret_cast<const unsigned long long *>(d_line_start),
                                                                  (unsigned long long)n_lines, d_table, (unsigned long long)(table_size - 1),
                                                                  d_owner, d_rec_mean, reinterpret_cast<unsigned long long *>(d_stats));
    MC_LAUNCH_CHECK();
    k_fq_publish<<<(unsigned)((table_size + 255) / 256), 256, 0, st>>>(d_table, (unsigned long long)(table_size - 1), d_owner, d_rec_mean);
    MC_LAUNCH_CHECK();
    return MC_OK;
}
