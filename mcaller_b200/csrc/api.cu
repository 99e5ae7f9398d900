// Error reporting + tiny host utilities of the C ABI.
#include <stdarg.h>
#include "common.cuh"

static thread_local char g_err[512] = "";

void mc_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" int mc_version(void) { return MC_ABI_VERSION; }
extern "C" const char *mc_last_error(void) { return g_err; }

extern "C" int mc_read_u64(const uint64_t *d_src, int64_t n, uint64_t *h_dst, void *stream) {
    MC_REQUIRE(d_src && h_dst && n >= 0, "bad argument");
    MC_CUDA_CHECK(cudaMemcpyAsync(h_dst, d_src, sizeof(uint64_t) * (size_t)n, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    MC_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    return MC_OK;
}

// struct sizes, so bindings in other languages can verify their layout (0 record, 1 call, 2 refindex, 3 model,
// 4 qual entry, 5 synth spec, 6 locus entry, 7 diffs row, 8 carry, 9 training job,
// 10 row-log entry)
extern "C" int mc_sizeof(int what) {
    switch (what) {
        case 0: return (int)sizeof(mc_record);
        case 1: return (int)sizeof(mc_call);
        case 2: return (int)sizeof(mc_refindex);
        case 3: return (int)sizeof(mc_model);
        case 4: return (int)sizeof(mc_qual_entry);
        case 5: return (int)sizeof(mc_synth_spec);
        case 6: return (int)sizeof(mc_locus_entry);
        case 7: return (int)sizeof(mc_diffs_row);
        case 8: return (int)sizeof(mc_carry);
        case 9: return (int)sizeof(mc_train_job);
        case 10: return (int)sizeof(mc_row_entry);
        default: return -1;
    }
}
