// ftb_frame_rays' kernel: the primary ray and RNG key of every sample of a window, exactly as render_kernel generates them.
// Compiled once per precision by the Makefile, with the flags of that precision's render variants ([-DFTB_F64 --fmad=false] as the
// FP64 verification build, the fast-math flags in FP32), and it calls render_kernel's own primaryRay on a DevFrame that api.cu's
// fillCamera fills: the rays cannot drift from the frame's.  The generic FEAT mask: primaryRay reads only its FT_RNG bit (depth of
// field), which every variant that renders a depth-of-field frame has.
#include "render.cuh"

namespace ftb {
namespace {

// Entry e of the window [wx0, wx1) x [wy0, wy1) of the sample grid: sample e % spp of pixel e / spp, pixels row-major in the window
// (the debug planes' order).  rays: o.xyz d.xyz widened to double, before slightOffset; keys: (py * gw + px) * spp + s.
template <typename R>
__global__ void frame_rays_kernel(const __grid_constant__ DevFrame<R> F, double* rays, unsigned long long* keys)
{
    const int ww = F.wx1 - F.wx0;
    const long long n = (long long)ww * (F.wy1 - F.wy0) * F.spp;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const long long pix = e / F.spp;
        const int s = (int)(e - pix * F.spp);
        const int ly = (int)(pix / ww);
        const int px = F.wx0 + (int)(pix - (long long)ly * ww), py = F.wy0 + ly;
        const unsigned long long key = ((unsigned long long)py * (unsigned)F.gw + (unsigned)px) * (unsigned)F.spp + (unsigned)s;
        if (keys) keys[e] = key;
        if (rays) {
            const Ray<R> r = primaryRay<R, (unsigned)FT_ALL>(F, px, py, s, key);
            double* o = rays + 6 * e;
            o[0] = (double)r.o.x; o[1] = (double)r.o.y; o[2] = (double)r.o.z;
            o[3] = (double)r.d.x; o[4] = (double)r.d.y; o[5] = (double)r.d.z;
        }
    }
}

template <typename R>
cudaError_t launch_frame_rays_impl(const DevFrame<R>& f, long long n, double* rays, unsigned long long* keys, int sm_count, cudaStream_t stream)
{
    const long long blocks = (n + 255) / 256, cap = (long long)sm_count * 16;
    frame_rays_kernel<R><<<(int)(blocks < cap ? blocks : cap), 256, 0, stream>>>(f, rays, keys);
    return cudaGetLastError();
}

}  // namespace

#ifdef FTB_F64
cudaError_t frame_rays_f64(const DevFrame<double>& f, long long n, double* rays, unsigned long long* keys, int sm_count, cudaStream_t stream)
{
    return launch_frame_rays_impl<double>(f, n, rays, keys, sm_count, stream);
}
#else
cudaError_t frame_rays_f32(const DevFrame<float>& f, long long n, double* rays, unsigned long long* keys, int sm_count, cudaStream_t stream)
{
    return launch_frame_rays_impl<float>(f, n, rays, keys, sm_count, stream);
}
#endif
}  // namespace ftb
