// pg_ctc_fused_kernel<8, 512, *, *>: 8 CTC states per lane (see fused_impl.cuh)
#include "fused_impl.cuh"

namespace pgasr {
int launch_fused_spl8(int mode, FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word,
                      const ExploreArgs* explore) {
    return launch_fused_modes<8, 512>(mode, a, smem, st, word, explore);
}
}  // namespace pgasr

// timing build only (tools/phase_timing.py): the stamps live in this translation unit -- the headline variant
#ifdef PGASR_TIMING
extern "C" __attribute__((visibility("default"))) int pgasr_debug_cta_times(unsigned long long* host, int n) {
    cudaDeviceSynchronize();
    return cudaMemcpyFromSymbol(host, pgasr::g_cta_ns, sizeof(unsigned long long) * 3 * n) == cudaSuccess ? 0 : -5;
}
extern "C" __attribute__((visibility("default"))) int pgasr_debug_role_times(unsigned long long* host8, int reset) {
    cudaDeviceSynchronize();
    if (cudaMemcpyFromSymbol(host8, pgasr::g_role_ns, sizeof(unsigned long long) * 8) != cudaSuccess) return -5;
    if (reset) {
        unsigned long long z[8] = {0};
        cudaMemcpyToSymbol(pgasr::g_role_ns, z, sizeof(z));
    }
    return 0;
}
extern "C" __attribute__((visibility("default"))) int pgasr_debug_read(long long* host64, int reset) {
    cudaDeviceSynchronize();
    if (cudaMemcpyFromSymbol(host64, pgasr::g_dbg, sizeof(long long) * 64) != cudaSuccess) return -5;
    if (reset) {
        long long z[64] = {0};
        cudaMemcpyToSymbol(pgasr::g_dbg, z, sizeof(z));
    }
    return 0;
}
#endif
