// The crossing queries' kernel (render.cuh crossings_kernel): compiled once per precision by the Makefile, with the flags of the
// render variants of that precision ([-DFTB_F64 --fmad=false] as the FP64 verification build).  Only the generic FEAT mask: the
// specialised variants earn their speed by culling against the best hit so far, which an enumeration of every crossing cannot do.
#include "render.cuh"

namespace ftb {
#ifdef FTB_F64
cudaError_t crossings_f64(const DevScene<double>& s, const DevCrossings& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    return launch_crossings_impl<double, (unsigned)FT_ALL>(s, q, stats, sm_count, stream, launches);
}
#else
cudaError_t crossings_f32(const DevScene<float>& s, const DevCrossings& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    return launch_crossings_impl<float, (unsigned)FT_ALL>(s, q, stats, sm_count, stream, launches);
}
#endif
}  // namespace ftb
