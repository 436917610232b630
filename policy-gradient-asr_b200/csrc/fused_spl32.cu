// pg_ctc_fused_kernel<32, 256, *, *>: 32 CTC states per lane (see fused_impl.cuh)
#include "fused_impl.cuh"

namespace pgasr {
int launch_fused_spl32(int mode, FusedArgs& a, size_t smem, cudaStream_t st, const WordArgs* word,
                      const ExploreArgs* explore) {
    return launch_fused_modes<32, 256>(mode, a, smem, st, word, explore);
}
}  // namespace pgasr
