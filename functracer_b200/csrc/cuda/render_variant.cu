// One kernel variant: compiled once per (precision, FEAT mask) by the Makefile:
//   -DFTB_FEAT=0x.. [-DFTB_F64]     FP64 variants are built with --fmad=false so that a*b+c rounds
//                                   twice like the reference's JIT and the oracle.
#include "render.cuh"

#ifndef FTB_FEAT
#error "FTB_FEAT must be defined"
#endif
#define FTB_CAT2(a, b) a##b
#define FTB_CAT(a, b) FTB_CAT2(a, b)

namespace ftb {
#ifdef FTB_F64
typedef double VR;
#define FTB_VNAME FTB_CAT(launch_f64_, FTB_FEAT)
#define FTB_QNAME FTB_CAT(query_f64_, FTB_FEAT)
#define FTB_SNAME FTB_CAT(samples_f64_, FTB_FEAT)
#else
typedef float VR;
#define FTB_VNAME FTB_CAT(launch_f32_, FTB_FEAT)
#define FTB_QNAME FTB_CAT(query_f32_, FTB_FEAT)
#define FTB_SNAME FTB_CAT(samples_f32_, FTB_FEAT)
#endif

cudaError_t FTB_VNAME(const DevScene<VR>& s, const DevFrame<VR>& f, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    return launch_render_impl<VR, (unsigned)(FTB_FEAT), (FTB_FEAT) == FT_ALL>(s, f, stats, sm_count, stream, launches);
}

cudaError_t FTB_QNAME(const DevScene<VR>& s, const DevQuery& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    return launch_query_impl<VR, (unsigned)(FTB_FEAT), (FTB_FEAT) == FT_ALL>(s, q, stats, sm_count, stream, launches);
}

cudaError_t FTB_SNAME(const DevScene<VR>& s, const DevFrame<VR>& f, const unsigned long long* keys, bool stats, int sm_count, cudaStream_t stream,
                      int* launches)
{
    return launch_samples_impl<VR, (unsigned)(FTB_FEAT), (FTB_FEAT) == FT_ALL>(s, f, keys, stats, sm_count, stream, launches);
}
}  // namespace ftb
