// api.cu — the C ABI of include/functracer_b200.h: scene upload, frame set-up, kernel launch,
// tile assembly (blend / quantise), in-process multi-GPU with a P2P gather, statistics.
//
// There is NO CPU fallback in this file: without a CUDA device every entry point that computes
// returns FTB_ERR_NO_DEVICE.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../../include/functracer_b200.h"
#include "bvh_build.h"
#include "device_scene.h"
#include "lower.h"
#include "clear_boxes.h"
#include "lit_tiles.h"
#include "tiles.h"

namespace ftb {

// ---- assembly kernels (api.cu owns them; the render kernels live in render_f32/f64.cu) --------------
constexpr int kMaxShards = 64;
struct TilePtrs {
    const void* p[kMaxShards];
};

template <typename R>
__device__ __forceinline__ void loadTilePixel(const TilePtrs& bufs, int shard_count, int tiles_x, int x, int y, R& r, R& g, R& b)
{
    const int tile = (y / FTB_TILE_H) * tiles_x + (x / FTB_TILE_W);
    const int shard = shardOfTile(tile, shard_count), local = tile / shard_count;
    const R* src = static_cast<const R*>(bufs.p[shard]) + 3 * ((long long)local * FTB_TILE_PIXELS + (y % FTB_TILE_H) * FTB_TILE_W + (x % FTB_TILE_W));
    r = src[0]; g = src[1]; b = src[2];
}

// Image.write's toByte (Image.fs:36, Math.fs:12-16): clamp to [0,1], * 255.0, truncate.
template <typename R>
__device__ __forceinline__ unsigned char toByte(R c)
{
    R k = c > R(1) ? R(1) : (c < R(0) ? R(0) : c);  // NaN falls through both tests like Math.clamp
    return (unsigned char)(int)(k * R(255));
}

// Tile-major shard buffers -> row-major frame.  corner = 1: CornerSampling.blendPixels
// (Image.fs:134-144): pixel = average of the sample grid's [TL; TR; BL; BR] corners.
template <typename R>
__global__ void assemble_kernel(TilePtrs bufs, int shard_count, int tiles_x, int W, int y0, int y1, int corner, int out_format, void* out)
{
    const long long n = (long long)W * y1;
    for (long long i = (long long)W * y0 + blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int x = (int)(i % W), y = (int)(i / W);
        R r, g, b;
        if (!corner) {
            loadTilePixel<R>(bufs, shard_count, tiles_x, x, y, r, g, b);
        } else {
            R r1, g1, b1;
            loadTilePixel<R>(bufs, shard_count, tiles_x, x, y, r, g, b);  // Seq.average: Zero + TL + TR + BL + BR, then / 4
            r = R(0) + r; g = R(0) + g; b = R(0) + b;
            loadTilePixel<R>(bufs, shard_count, tiles_x, x + 1, y, r1, g1, b1); r += r1; g += g1; b += b1;
            loadTilePixel<R>(bufs, shard_count, tiles_x, x, y + 1, r1, g1, b1); r += r1; g += g1; b += b1;
            loadTilePixel<R>(bufs, shard_count, tiles_x, x + 1, y + 1, r1, g1, b1); r += r1; g += g1; b += b1;
            r = r / R(4); g = g / R(4); b = b / R(4);
        }
        if (out_format == FTB_OUT_RGB_F64) {
            double* o = static_cast<double*>(out) + 3 * i;
            o[0] = (double)r; o[1] = (double)g; o[2] = (double)b;
        } else if (out_format == FTB_OUT_RGB_F32) {
            float* o = static_cast<float*>(out) + 3 * i;
            o[0] = (float)r; o[1] = (float)g; o[2] = (float)b;
        } else {
            static_cast<uchar4*>(out)[i] = make_uchar4(toByte(r), toByte(g), toByte(b), 255);
        }
    }
}

// The blocks of the clear tiles (tiles.h: no primary sample of theirs hits anything, so every sample's colour is exactly zero),
// one warp per block, written without tracing: the render kernel's fold (render.cuh foldUnit) over all-zero samples - the
// running sum of the earlier passes, divided by spp on the last - and a miss in every requested debug plane.  With `counting`
// their samples are added to the primary rays, as the counting render kernel would.  A kernel of its own: the render kernel's
// code is exactly what it was without clear tiles (an extra path in it changes its register allocation and costs 2-3 %).
template <typename R>
__global__ void clear_kernel(const __grid_constant__ DevFrame<R> F, int counting)
{
    const int lane = threadIdx.x & 31;
    const int warps = gridDim.x * (blockDim.x >> 5);
    for (int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < F.n_clear_blocks; c += warps) {
        int slot0, x0, y0, w, npix;
        openBlock<R>(F, (unsigned)(F.n_blocks + c), slot0, x0, y0, w, npix);
        for (int i = lane; i < npix * 3; i += 32) {
            const int pix = i / 3, ch = i - 3 * pix;
            const int ly = pix / w;
            const long long o = 3 * ((long long)slot0 + ly * FTB_TILE_W + (pix - ly * w)) + ch;
            R acc = F.s_base > 0 ? F.out[o] : R(0);
            if (F.s_base + F.s_count >= F.spp) acc = acc / (R)F.spp;
            F.out[o] = acc;
        }
        if (F.dbg_prim) {
            for (int i = lane; i < npix * F.s_count; i += 32) {
                const int pix = i / F.s_count, s = F.s_base + (i - pix * F.s_count);
                const int ly = pix / w;
                const unsigned long long at = ((unsigned long long)(unsigned)(y0 + ly - F.wy0) * (unsigned)F.dbg_w + (unsigned)(x0 + pix - ly * w - F.wx0)) * (unsigned)F.spp + (unsigned)s;
                F.dbg_prim[at] = -1;
                if (F.dbg_sub) F.dbg_sub[at] = 0;
                if (F.dbg_t) F.dbg_t[at] = -1.0;
            }
        }
        if (counting && lane == 0 && npix > 0) atomicAdd(F.stats + ST_PRIMARY, (unsigned long long)npix * (unsigned long long)F.s_count);
    }
}

// ftb_shade_rays: [ray][3] in R -> doubles
template <typename R>
__global__ void widen_kernel(const R* in, double* out, long long n)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) out[i] = (double)in[i];
}

}  // namespace ftb

namespace ftb {
static_assert((unsigned)FT_TABLE == kFeatOriginTable, "lower.h and device_scene.h disagree on the table feature bit");
// kernel variants compiled by the Makefile (render_variant.cu), listed through -DFTB_FEAT_LIST_F32 / _F64
#define X(feat) cudaError_t launch_f32_##feat(const DevScene<float>&, const DevFrame<float>&, bool, int, cudaStream_t, int*); \
    cudaError_t query_f32_##feat(const DevScene<float>&, const DevQuery&, bool, int, cudaStream_t, int*); \
    cudaError_t samples_f32_##feat(const DevScene<float>&, const DevFrame<float>&, const unsigned long long*, bool, int, cudaStream_t, int*);
FTB_FEAT_LIST_F32
FTB_FEAT_LIST_F32_TMASK
#undef X
#define X(feat) cudaError_t launch_f64_##feat(const DevScene<double>&, const DevFrame<double>&, bool, int, cudaStream_t, int*); \
    cudaError_t query_f64_##feat(const DevScene<double>&, const DevQuery&, bool, int, cudaStream_t, int*); \
    cudaError_t samples_f64_##feat(const DevScene<double>&, const DevFrame<double>&, const unsigned long long*, bool, int, cudaStream_t, int*);
FTB_FEAT_LIST_F64
#undef X
// the crossing queries' kernel (crossings.cu): generic FEAT only, one object per precision
cudaError_t crossings_f32(const DevScene<float>&, const DevCrossings&, bool, int, cudaStream_t, int*);
cudaError_t crossings_f64(const DevScene<double>&, const DevCrossings&, bool, int, cudaStream_t, int*);
inline cudaError_t launchCrossings(const DevScene<float>& s, const DevCrossings& q, bool stats, int sm, cudaStream_t st, int* l) { return crossings_f32(s, q, stats, sm, st, l); }
inline cudaError_t launchCrossings(const DevScene<double>& s, const DevCrossings& q, bool stats, int sm, cudaStream_t st, int* l) { return crossings_f64(s, q, stats, sm, st, l); }
// the path queries' kernel (paths.cu): generic FEAT only, one object per precision
cudaError_t paths_f32(const DevScene<float>&, const DevPaths&, bool, int, cudaStream_t, int*);
cudaError_t paths_f64(const DevScene<double>&, const DevPaths&, bool, int, cudaStream_t, int*);
inline cudaError_t launchPaths(const DevScene<float>& s, const DevPaths& q, bool stats, int sm, cudaStream_t st, int* l) { return paths_f32(s, q, stats, sm, st, l); }
inline cudaError_t launchPaths(const DevScene<double>& s, const DevPaths& q, bool stats, int sm, cudaStream_t st, int* l) { return paths_f64(s, q, stats, sm, st, l); }
// ftb_frame_rays' kernel (frame_rays.cu): one object per precision
cudaError_t frame_rays_f32(const DevFrame<float>&, long long, double*, unsigned long long*, int, cudaStream_t);
cudaError_t frame_rays_f64(const DevFrame<double>&, long long, double*, unsigned long long*, int, cudaStream_t);
inline cudaError_t launchFrameRays(const DevFrame<float>& f, long long n, double* r, unsigned long long* k, int sm, cudaStream_t st) { return frame_rays_f32(f, n, r, k, sm, st); }
inline cudaError_t launchFrameRays(const DevFrame<double>& f, long long n, double* r, unsigned long long* k, int sm, cudaStream_t st) { return frame_rays_f64(f, n, r, k, sm, st); }
static const Variant<float> kVariantsF32[] = {
#define X(feat) {(unsigned)(feat), UnitCap<float, (unsigned)(feat)>::value, (feat) == FT_ALL, launch_f32_##feat, query_f32_##feat, samples_f32_##feat},
    FTB_FEAT_LIST_F32
#undef X
};
static const Variant<double> kVariantsF64[] = {
#define X(feat) {(unsigned)(feat), UnitCap<double, (unsigned)(feat)>::value, (feat) == FT_ALL, launch_f64_##feat, query_f64_##feat, samples_f64_##feat},
    FTB_FEAT_LIST_F64
#undef X
};
// the FT_TMASK instances (-DFTB_FEAT_LIST_F32_TMASK): picked by withTileMasks, never by pickCover
static const Variant<float> kTMaskVariantsF32[] = {
#define X(feat) {(unsigned)(feat), UnitCap<float, (unsigned)(feat)>::value, false, launch_f32_##feat, query_f32_##feat, samples_f32_##feat},
    FTB_FEAT_LIST_F32_TMASK
#undef X
};
template <typename R> struct VariantTable;
template <> struct VariantTable<float> { static const Variant<float>* begin() { return kVariantsF32; } static int size() { return (int)(sizeof(kVariantsF32) / sizeof(kVariantsF32[0])); } };
template <> struct VariantTable<double> { static const Variant<double>* begin() { return kVariantsF64; } static int size() { return (int)(sizeof(kVariantsF64) / sizeof(kVariantsF64[0])); } };

// the smallest compiled variant that covers `need` (and has the counting kernel if asked for)
template <typename R>
const Variant<R>* pickCover(unsigned need, bool stats)
{
    const Variant<R>* best = nullptr;
    for (int i = 0; i < VariantTable<R>::size(); ++i) {
        const Variant<R>* v = VariantTable<R>::begin() + i;
        if ((v->feat & need) != need || (stats && !v->has_stats)) continue;
        if (!best || __builtin_popcount(v->feat) < __builtin_popcount(best->feat)) best = v;
    }
    return best;
}
// FT_TABLE is an optimisation, not a requirement: a scene that would like the common-origin bound table but whose other
// needs are only covered together with it by the generic kernel runs on the specialised kernel without the table.
template <typename R>
const Variant<R>* pickVariant(unsigned need, bool stats)
{
    const Variant<R>* v = pickCover<R>(need, stats);
    if ((need & FT_TABLE) && (!v || v->feat == FT_ALL)) {
        const Variant<R>* w = pickCover<R>(need & ~(unsigned)FT_TABLE, stats);
        if (w && w->feat != FT_ALL) return w;
    }
    return v;
}
// The instance of variant v that reads the per-tile item masks (FT_TMASK), if one is compiled: FP32 only.
template <typename R>
const Variant<R>* withTileMasks(const Variant<R>* v)
{
    if constexpr (sizeof(R) == 4) {
        for (const Variant<float>& w : kTMaskVariantsF32)
            if (w.feat == (v->feat | (unsigned)FT_TMASK)) return &w;
    }
    return nullptr;
}
}  // namespace ftb

namespace {

using namespace ftb;

thread_local std::string g_err;

int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}
int cudaFail(cudaError_t e, const char* what)
{
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    (void)cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? FTB_ERR_OOM : FTB_ERR_CUDA;
}
#define CK(expr)                                              \
    do {                                                      \
        cudaError_t e__ = (expr);                             \
        if (e__ != cudaSuccess) return cudaFail(e__, #expr); \
    } while (0)

// A growable device buffer (scratch that survives between calls so steady-state frames do no cudaMalloc).
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct Control {  // device control block of one launch
    unsigned int tile_counter;
    unsigned int overflow;
    unsigned long long stats[ST_COUNT];
};

// The per-device control block and everything that resets, wires or reads it.  The queue counter is reset before every
// launch, the counters only when they are asked for; the overflow flag stays up until somebody reads it (finishStats /
// ftb_check_overflow), so that the banded and the device paths cannot lose it.
struct ControlBlock {
    DevBuf buf;
    bool zeroed = false;  // zeroed once by a frame launch (ftb_shade_rays zeroes the whole block itself)
    Control* ctl() const { return static_cast<Control*>(buf.p); }
    bool used() const { return buf.p != nullptr; }  // something has been launched on this device
    cudaError_t reserve() { return buf.reserve(sizeof(Control)); }
    // a frame launch: the block is zeroed the first time, the counters whenever they are counted
    cudaError_t prepare(bool counting, cudaStream_t s)
    {
        cudaError_t e = zeroed ? cudaSuccess : cudaMemsetAsync(buf.p, 0, sizeof(Control), s);
        zeroed = e == cudaSuccess;
        return e != cudaSuccess || !counting ? e : cudaMemsetAsync(ctl()->stats, 0, sizeof(Control::stats), s);
    }
    cudaError_t resetAll(cudaStream_t s) { cudaError_t e = reserve(); return e != cudaSuccess ? e : cudaMemsetAsync(buf.p, 0, sizeof(Control), s); }
    cudaError_t resetQueue(cudaStream_t s) { return cudaMemsetAsync(&ctl()->tile_counter, 0, sizeof(unsigned int), s); }
    template <typename R> void wire(DevFrame<R>& F) const { F.tile_counter = &ctl()->tile_counter; F.overflow = &ctl()->overflow; F.stats = ctl()->stats; }
    // D2H copy into h, synchronising `s`; a raised overflow flag is cleared on the device
    cudaError_t read(Control& h, cudaStream_t s)
    {
        cudaError_t e = cudaMemcpyAsync(&h, buf.p, sizeof(h), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        return e != cudaSuccess || !h.overflow ? e : cudaMemsetAsync(&ctl()->overflow, 0, sizeof(unsigned int), s);
    }
};

template <typename R>
struct SceneStorage {
    DevScene<R> view;
    std::vector<void*> allocs;
    bool ready = false;
    void release() { for (void* p : allocs) cudaFree(p); allocs.clear(); ready = false; }
};

struct PerDevice;
template <typename R> SceneStorage<R>& storageOf(PerDevice* pd);

// Device -> host copies of finished bands.  The destination is whatever the caller owns: usually ordinary pageable memory
// (a GC-pinned .NET array, a std::vector, numpy), sometimes CUDA page-locked memory.  A cudaMemcpyAsync into pageable
// memory does not return before the data is there (the driver stages it through its own page-locked buffers at link
// speed), so the order of work is what matters: every band's render + assembly is queued FIRST, then the bands are
// copied in the order they finish; while the host sits in the copy of band c the GPU is rendering band c + 1.
// Measured (B200, 16 host cores, RGBA8 frame of the 8K moon scene, 132 MB): driver-staged copy +1.3 ms per frame over the
// device-resident time, a library-owned page-locked ring + memcpy on the calling thread +5.7 ms, cudaHostRegister of
// the caller's buffer per call +21 ms; the 1080p hollow-sphere frame: 1.43 / 1.50 / 14.6 ms.  So the driver's path it is.
struct HostCopier {
    std::vector<cudaStream_t> used;  // streams that carry copies this frame (synchronised by finish)
    cudaError_t begin(const void* d_src, void* host_dst, size_t bytes, cudaStream_t stream)
    {
        if (bytes == 0) return cudaSuccess;
        cudaError_t e = cudaMemcpyAsync(host_dst, d_src, bytes, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess && std::find(used.begin(), used.end(), stream) == used.end()) used.push_back(stream);
        return e;
    }
    cudaError_t finish()
    {
        cudaError_t e = cudaSuccess;
        for (cudaStream_t st : used) {
            cudaError_t e2 = cudaStreamSynchronize(st);
            if (e == cudaSuccess) e = e2;
        }
        used.clear();
        return e;
    }
};

struct PerDevice {
    int device = -1;
    int sm_count = 0;
    SceneStorage<float> f32;
    SceneStorage<double> f64;
    cudaStream_t stream = nullptr;  // owned; used by the host-buffer entry points
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, done = nullptr;
    ControlBlock control;
    DevBuf jitter, tiles, out, dbg_prim, dbg_sub, dbg_t, rays, order, lit, items;
    DevBuf query;  // the host-buffer ray queries: max_t and the requested output planes
    std::vector<int> chunk_first;          // first position in the tile order of every chunk (+ end)
    std::vector<int> chunk_clear;          // position in the tile order where every chunk's clear tiles start
    cudaStream_t copy_stream = nullptr;    // assembly / D2H of finished bands while later bands render (highest priority)
    std::vector<cudaEvent_t> band_events;
    HostCopier copier;
    std::vector<unsigned char> order_key;  // what the cached tile order was computed for
    bool order_valid = false;
    int lit_leaf = -1;  // the cached lit-tile mask's ground leaf (in `lit`); -1: no tile is lit
    bool items_valid = false;  // `items` holds the cached per-tile item masks, and they pay (computeTileOrder)
    std::vector<DevBuf> peer_tiles;  // on the gather device: one per remote shard

    PerDevice() = default;
    PerDevice(const PerDevice&) = delete;
    PerDevice& operator=(const PerDevice&) = delete;
    // Releases everything the device holds, also when a create / upload failed half way (the owner switches devices).
    ~PerDevice()
    {
        if (device < 0) return;
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess) cur = -1;
        if (cudaSetDevice(device) == cudaSuccess) {
            if (stream) cudaStreamSynchronize(stream);
            if (copy_stream) cudaStreamSynchronize(copy_stream);
            f32.release(); f64.release();
            for (DevBuf* b : {&control.buf, &jitter, &tiles, &out, &dbg_prim, &dbg_sub, &dbg_t, &rays, &order, &lit, &items, &query}) b->release();
            for (DevBuf& b : peer_tiles) b.release();
            if (ev0) cudaEventDestroy(ev0);
            if (ev1) cudaEventDestroy(ev1);
            if (done) cudaEventDestroy(done);
            for (cudaEvent_t e : band_events) cudaEventDestroy(e);
            if (stream) cudaStreamDestroy(stream);
            if (copy_stream) cudaStreamDestroy(copy_stream);
        }
        (void)cudaGetLastError();
        if (cur >= 0) cudaSetDevice(cur);
    }
};

template <> SceneStorage<float>& storageOf<float>(PerDevice* pd) { return pd->f32; }
template <> SceneStorage<double>& storageOf<double>(PerDevice* pd) { return pd->f64; }

}  // namespace

struct ftb_scene {
    ftb::Lowered L;
    // host copies of the tables the upload needs
    std::vector<double> triangles;
    std::vector<ftb_light> lights;
    struct Img { int w, h; std::vector<uint8_t> rgb; };
    std::vector<Img> images;
    std::map<int, std::unique_ptr<PerDevice>> devices;
    ftb::DeviceBuildStats bvh_stats;  // mesh index built on the device at create time (bvh_build.h)
    bool bvh_on_device = false;
};

namespace {

template <typename R> struct Mk4;
template <> struct Mk4<float> { static float4 make(double a, double b, double c, double d) { return make_float4((float)a, (float)b, (float)c, (float)d); } };
template <> struct Mk4<double> { static double4 make(double a, double b, double c, double d) { return make_double4(a, b, c, d); } };

template <typename T>
int upload(std::vector<void*>& allocs, const std::vector<T>& host, const T*& dev)
{
    dev = nullptr;
    if (host.empty()) return FTB_OK;
    void* p = nullptr;
    CK(cudaMalloc(&p, host.size() * sizeof(T)));
    allocs.push_back(p);
    CK(cudaMemcpy(p, host.data(), host.size() * sizeof(T), cudaMemcpyHostToDevice));
    dev = static_cast<const T*>(p);
    return FTB_OK;
}

// Meshes of this many (clipped) triangles or more are walked by the whole warp (render.cuh packetMesh) and their samples are
// dealt one at a time; smaller ones by each lane for itself.  Measured on 960 / 9.6 k / 355 k triangles at 3840x2160x16: private
// walks 2.92 / 3.41 / 9.11 ms, packet walks 3.19 / 3.60 / 6.38 ms.
constexpr size_t kLargeMesh = 32768;
inline bool largeMesh(const Lowered& L) { return L.bvh_tri.size() >= kLargeMesh; }

template <typename R>
int uploadScene(const ftb_scene& sc, SceneStorage<R>& st)
{
    typedef typename V4<R>::type R4;
    const Lowered& L = sc.L;
    DevScene<R>& v = st.view;
    std::memset(&v, 0, sizeof(v));
    int rc;
#define UP(vec, field) if ((rc = upload(st.allocs, vec, field)) != FTB_OK) { st.release(); return rc; }
    {
        std::vector<R4> w2m, p0; std::vector<int4> meta;
        for (const Leaf& lf : L.leaves) {
            for (int r = 0; r < 3; ++r) w2m.push_back(Mk4<R>::make(lf.w2m[4 * r], lf.w2m[4 * r + 1], lf.w2m[4 * r + 2], lf.w2m[4 * r + 3]));
            {  // world point of the model origin: solve A p0 + b = 0 (Cramer; singular matrices keep p0 = 0)
                const double* m = lf.w2m;
                const double c00 = m[5] * m[10] - m[6] * m[9], c01 = m[6] * m[8] - m[4] * m[10], c02 = m[4] * m[9] - m[5] * m[8];
                const double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
                double q[3] = {0, 0, 0};
                if (std::fabs(det) > 0 && std::isfinite(det)) {
                    const double id = 1.0 / det, bx = -m[3], by = -m[7], bz = -m[11];
                    q[0] = (bx * c00 + by * (m[2] * m[9] - m[1] * m[10]) + bz * (m[1] * m[6] - m[2] * m[5])) * id;
                    q[1] = (bx * c01 + by * (m[0] * m[10] - m[2] * m[8]) + bz * (m[2] * m[4] - m[0] * m[6])) * id;
                    q[2] = (bx * c02 + by * (m[1] * m[8] - m[0] * m[9]) + bz * (m[0] * m[5] - m[1] * m[4])) * id;
                }
                p0.push_back(Mk4<R>::make(q[0], q[1], q[2], 0));
            }
            meta.push_back(make_int4(lf.kind | (lf.identity << 8) | (lf.top_level << 9), lf.surface, lf.prim, lf.payload));
        }
        UP(w2m, v.leaf_w2m) UP(meta, v.leaf_meta) UP(p0, v.leaf_p0)
        v.n_leaves = (int)L.leaves.size();
    }
    {
        std::vector<int4> items; std::vector<R4> bounds; std::vector<int2> ops, progs;
        for (const Item& it : L.items) {
            // kind | CSG op << 8 | kind word of leaf A << 12 | of leaf B << 21 (kind word = leaf kind | identity << 8, as in leaf_meta.x):
            // the walk branches on a top-level leaf's / a pair operand's kind without waiting for the leaf's own record
            auto kw = [&](int leaf) { const Leaf& lf = L.leaves[(size_t)(leaf & 0xffffff)]; return (lf.kind & 0xff) | (lf.identity ? 0x100 : 0); };
            int kx = it.kind & 0xfff;
            if ((it.kind & 0xff) == ITEM_LEAF) kx |= kw(it.a) << 12;
            else if ((it.kind & 0xff) == ITEM_CSG2) kx |= (kw(it.a) << 12) | (kw(it.b) << 21);
            items.push_back(make_int4(kx, it.a, it.b, it.casts_shadow));
            progs.push_back(make_int2(it.prog_first, it.prog_count));
            // conservative: radius inflated by 0.2 % + 1e-5 so that FP32 rounding of the test cannot cull a true hit
            // unbounded items (planes) carry r^2 = +inf: no line misses them and no origin is outside them
            const double ri = it.bound_r < 0 ? -1.0 : it.bound_r * 1.002 + 1e-5;
            bounds.push_back(Mk4<R>::make(it.bound_c[0], it.bound_c[1], it.bound_c[2], ri < 0 ? (double)INFINITY : ri * ri));
        }
        for (const CsgOp& op : L.ops) ops.push_back(make_int2(op.kind, op.arg));
        std::vector<unsigned> casts((L.items.size() + 31) / 32 + 1, 0u);
        for (size_t i = 0; i < L.items.size(); ++i)
            if (L.items[i].casts_shadow) casts[i >> 5] |= 1u << (i & 31);
        std::vector<unsigned> meshes(casts.size(), 0u);
        for (size_t i = 0; i < L.items.size(); ++i)
            if (L.items[i].kind == ITEM_LEAF && L.leaves[(size_t)L.items[i].a].kind == LEAF_MESH) meshes[i >> 5] |= 1u << (i & 31);
        std::vector<R4> bounds2;  // pairs of neighbouring items interleaved (render.cuh: the packed bound test of the FP32 kernels)
        for (size_t i = 0; i < bounds.size(); i += 2) {
            const R4 a = bounds[i], b = i + 1 < bounds.size() ? bounds[i + 1] : Mk4<R>::make(0, 0, 0, (double)INFINITY);
            bounds2.push_back(Mk4<R>::make(a.x, b.x, a.y, b.y));
            bounds2.push_back(Mk4<R>::make(a.z, b.z, a.w, b.w));
        }
        UP(bounds2, v.item_bound2)
        UP(items, v.items) UP(bounds, v.item_bound) UP(ops, v.ops) UP(casts, v.item_casts) UP(meshes, v.item_mesh) UP(progs, v.item_prog)
        v.mesh_packet = largeMesh(L) ? 1 : 0;
        v.n_items = (int)L.items.size();
    }
    {
        std::vector<R4> a, b; std::vector<int4> si;
        for (const Surface& s : L.surfaces) {
            a.push_back(Mk4<R>::make(s.colour[0], s.colour[1], s.colour[2], s.roughness));
            b.push_back(Mk4<R>::make(s.reflectance, s.shineyness, 0, 0));
            si.push_back(make_int4(s.texture, s.hue, s.apply_lighting, 0));
        }
        UP(a, v.surf_a) UP(b, v.surf_b) UP(si, v.surf_i)
    }
    {
        std::vector<int4> ti; std::vector<R4> c1, c2; std::vector<int> kinds; std::vector<R> ab;
        for (const TexDef& t : L.textures) {
            ti.push_back(make_int4(t.op_first, t.op_count, t.base_kind, t.image));
            c1.push_back(Mk4<R>::make(t.c1[0], t.c1[1], t.c1[2], 0));
            c2.push_back(Mk4<R>::make(t.c2[0], t.c2[1], t.c2[2], 0));
        }
        for (const TexOp& o : L.tex_ops) { kinds.push_back(o.kind); ab.push_back((R)o.a); ab.push_back((R)o.b); }
        UP(ti, v.tex_i) UP(c1, v.tex_c1) UP(c2, v.tex_c2) UP(kinds, v.texop_kind) UP(ab, v.texop_ab)
        std::vector<uchar4> texels; std::vector<int4> ii;
        for (const ftb_scene::Img& im : sc.images) {
            ii.push_back(make_int4((int)texels.size(), im.w, im.h, 0));
            const size_t n = (size_t)im.w * im.h;
            for (size_t k = 0; k < n; ++k) texels.push_back(make_uchar4(im.rgb[3 * k], im.rgb[3 * k + 1], im.rgb[3 * k + 2], 255));
        }
        UP(texels, v.texels) UP(ii, v.img_i)
    }
    {
        std::vector<int> roots(L.mesh_root.begin(), L.mesh_root.end()); std::vector<R4> box, btris, tris;
        for (const BvhNode& n : L.bvh_nodes) {
            for (int k = 0; k < 3; ++k) {  // one row per axis: (L.lo, R.lo, L.hi, R.hi)
                if (sizeof(R) == 4) box.push_back(Mk4<R>::make(n.lo[0][k], n.lo[1][k], n.hi[0][k], n.hi[1][k]));
                else box.push_back(Mk4<R>::make(n.dlo[0][k], n.dlo[1][k], n.dhi[0][k], n.dhi[1][k]));
            }
            R4 lk = Mk4<R>::make(n.child[0], n.child[1], 0, 0);  // the links in the record's fourth row: FP64 as values, FP32 as bits
            if (sizeof(R) == 4) { std::memcpy(&lk.x, &n.child[0], 4); std::memcpy(&lk.y, &n.child[1], 4); }
            box.push_back(lk);
        }
        const size_t nt = sc.triangles.size() / 9;
        auto pushTri = [&](std::vector<R4>& dst, size_t t, double w0, double w1) {  // v0, e1 = v1 - v0, e2 = v2 - v0 (Triangle.fs:45-46), differences taken in double
            const double* q = sc.triangles.data() + 9 * t;
            dst.push_back(Mk4<R>::make(q[0], q[1], q[2], w0));
            dst.push_back(Mk4<R>::make(q[3] - q[0], q[4] - q[1], q[5] - q[2], w1));
            dst.push_back(Mk4<R>::make(q[6] - q[0], q[7] - q[1], q[8] - q[2], 0));
        };
        for (size_t t = 0; t < nt; ++t) pushTri(tris, t, 0, 0);
        // slot ids ride in the w components as reals: exact up to 2^24 in float
        if (sizeof(R) == 4 && (L.bvh_tri.size() >= (1u << 24) || nt >= (1u << 24))) { st.release(); return fail(FTB_ERR_UNSUPPORTED, "more than 16M mesh triangles"); }
        for (size_t k = 0; k < L.bvh_tri.size(); ++k) pushTri(btris, (size_t)L.bvh_tri[k], (double)L.bvh_seq[k], (double)L.bvh_tri[k]);
        UP(roots, v.mesh_root) UP(box, v.bvh_node) UP(btris, v.bvh_tris) UP(tris, v.tris)
    }
    {
        std::vector<int2> li; std::vector<R4> la, lb, lc;
        for (const ftb_light& l : sc.lights) {
            li.push_back(make_int2(l.kind, l.samples));
            la.push_back(Mk4<R>::make(l.v[0], l.v[1], l.v[2], std::tan(l.scatter_rad / 2.0)));  // Jitter.fs:29
            lb.push_back(Mk4<R>::make(l.falloff[0], l.falloff[1], l.falloff[2], 0));
            lc.push_back(Mk4<R>::make(l.colour[0], l.colour[1], l.colour[2], 0));
        }
        UP(li, v.light_i) UP(la, v.light_a) UP(lb, v.light_b) UP(lc, v.light_c)
        v.n_lights = (int)sc.lights.size();
    }
    {  // the inverse of `rotate unitZ 180` (Cylinder.fs:27) exactly as Transform.matrix builds it (Transform.fs:60-69, CommonTypes.fs:98-99)
        const double ang = -(180.0 * 1.0 * (3.14159265358979323846 / 180.0));
        v.cyl_c = (R)std::cos(ang); v.cyl_s = (R)std::sin(ang);
    }
#undef UP
    st.ready = true;
    return FTB_OK;
}

int getDevice(ftb_scene* sc, int device, PerDevice** out)
{
    auto it = sc->devices.find(device);
    if (it == sc->devices.end()) {
        std::unique_ptr<PerDevice> pd(new PerDevice);  // ~PerDevice releases whatever exists if one of the calls below fails
        pd->device = device;
        CK(cudaSetDevice(device));
        CK(cudaDeviceGetAttribute(&pd->sm_count, cudaDevAttrMultiProcessorCount, device));
        int prLow = 0, prHigh = 0;
        CK(cudaDeviceGetStreamPriorityRange(&prLow, &prHigh));
        CK(cudaStreamCreateWithFlags(&pd->stream, cudaStreamNonBlocking));
        // the copy stream's kernels (assembly of a finished band) go ahead of the next band's render blocks
        CK(cudaStreamCreateWithPriority(&pd->copy_stream, cudaStreamNonBlocking, prHigh));
        CK(cudaEventCreate(&pd->ev0));
        CK(cudaEventCreate(&pd->ev1));
        CK(cudaEventCreateWithFlags(&pd->done, cudaEventDisableTiming));
        it = sc->devices.emplace(device, std::move(pd)).first;
    }
    *out = it->second.get();
    return FTB_OK;
}

// A pixel window [x0, x1) x [y0, y1) of the frame; the whole frame is {0, 0, width, height}.
struct Window { int x0, y0, x1, y1; };

// The geometry of one frame's work.  gw / gh are the whole frame's sample grid (ray directions, RNG keys); everything
// else - tile grid, local tiles, samples, bands - is the window's, whose tile grid starts at its origin.
struct FrameGeom {
    int gw, gh;                  // the whole frame's sample grid
    int wx0, wy0, ww, wh;        // the window in the sample grid: origin and size ((w+1) x (h+1) corners in corner mode)
    int width, height;           // the window in pixels: the frame that its tile buffer and assembly are those of
    int spp, tiles_x, tiles_y, n_tiles, shard_index, shard_count, n_local_tiles;
    int band_index, band_count;  // ftb_render_tiles_device: only the tiles of one band of tile rows (band_count <= 1: all)
    long long n_samples;
    bool corner;
};

int frameGeom(const ftb_render_params* p, FrameGeom& g, const Window* win = nullptr)
{
    if (!p) return fail(FTB_ERR_BAD_ARG, "null params");
    if (p->width < 1 || p->height < 1) return fail(FTB_ERR_BAD_ARG, "bad resolution");
    if ((long long)p->width * p->height > (1LL << 30)) return fail(FTB_ERR_BAD_ARG, "resolution too large");
    if (p->sampling != FTB_SAMPLING_JITTER && p->sampling != FTB_SAMPLING_CORNER) return fail(FTB_ERR_BAD_ARG, "bad sampling mode");
    if (p->precision != FTB_PRECISION_FP32 && p->precision != FTB_PRECISION_FP64_VERIFY) return fail(FTB_ERR_BAD_ARG, "bad precision");
    if (p->out_format < FTB_OUT_RGB_F64 || p->out_format > FTB_OUT_RGBA8) return fail(FTB_ERR_BAD_ARG, "bad output format");
    const Window w = win ? *win : Window{0, 0, p->width, p->height};
    if (w.x0 < 0 || w.y0 < 0 || w.x0 >= w.x1 || w.y0 >= w.y1 || w.x1 > p->width || w.y1 > p->height)
        return fail(FTB_ERR_BAD_ARG, "bad window: needs 0 <= x0 < x1 <= width and 0 <= y0 < y1 <= height");
    g.corner = p->sampling == FTB_SAMPLING_CORNER;
    if (!g.corner && (p->spp < 1 || !p->jitter_xy)) return fail(FTB_ERR_BAD_ARG, "jitter mode needs spp >= 1 and jitter_xy");
    g.gw = g.corner ? p->width + 1 : p->width;
    g.gh = g.corner ? p->height + 1 : p->height;
    g.width = w.x1 - w.x0; g.height = w.y1 - w.y0;
    g.wx0 = w.x0; g.wy0 = w.y0;
    g.ww = g.corner ? g.width + 1 : g.width;  // the corners [x0, x1] x [y0, y1]
    g.wh = g.corner ? g.height + 1 : g.height;
    g.spp = g.corner ? 1 : p->spp;
    g.tiles_x = (g.ww + FTB_TILE_W - 1) / FTB_TILE_W;
    g.tiles_y = (g.wh + FTB_TILE_H - 1) / FTB_TILE_H;
    g.n_tiles = g.tiles_x * g.tiles_y;
    g.shard_count = p->shard_count > 1 ? p->shard_count : 1;
    g.shard_index = p->shard_count > 1 ? p->shard_index : 0;
    if (g.shard_count > kMaxShards) return fail(FTB_ERR_BAD_ARG, "shard_count exceeds 64");
    if (g.shard_index < 0 || g.shard_index >= g.shard_count) return fail(FTB_ERR_BAD_ARG, "shard_index out of range");
    g.n_local_tiles = (g.n_tiles + g.shard_count - 1) / g.shard_count;  // one per group of shard_count tiles (device_scene.h tileOfLocal); the last group may lack this shard's
    g.n_samples = (long long)g.ww * g.wh * g.spp;
    g.band_count = p->band_count > 1 ? p->band_count : 1;
    g.band_index = p->band_count > 1 ? p->band_index : 0;
    if (g.band_count > 64) return fail(FTB_ERR_BAD_ARG, "band_count exceeds 64");
    if (g.band_index < 0 || g.band_index >= g.band_count) return fail(FTB_ERR_BAD_ARG, "band_index out of range");
    return FTB_OK;
}

inline size_t realSize(int precision) { return precision == FTB_PRECISION_FP64_VERIFY ? sizeof(double) : sizeof(float); }

// the FP32 kernels receive the narrowed results
template <typename R>
void fillCamera(DevFrame<R>& F, const ftb_camera& c, int resH, int resV)
{
    const CameraBasis b = cameraBasis(c, resH, resV);
    const V3 &o = b.o, &k = b.k, &i = b.i, &j = b.j;
    F.cam_o[0] = (R)o.x; F.cam_o[1] = (R)o.y; F.cam_o[2] = (R)o.z;
    F.primary_slack = (R)(2e-4 * std::sqrt(o.x * o.x + o.y * o.y + o.z * o.z));
    F.cam_k[0] = (R)k.x; F.cam_k[1] = (R)k.y; F.cam_k[2] = (R)k.z;
    F.cam_i[0] = (R)i.x; F.cam_i[1] = (R)i.y; F.cam_i[2] = (R)i.z;
    F.cam_j[0] = (R)j.x; F.cam_j[1] = (R)j.y; F.cam_j[2] = (R)j.z;
    F.pw = (R)b.pw; F.ph = (R)b.ph;
    F.tlx = (R)b.tlx; F.tly = (R)b.tly;
    F.has_focus = c.has_focus;
    F.focal = (R)c.focal_length;
    F.tan_half_aperture = (R)std::tan(c.aperture_rad / 2.0);
}

void fillStats(const Control& h, const ftb_scene& sc, ftb_stats* s)
{
    const unsigned long long* c = h.stats;
    s->primary_rays += c[ST_PRIMARY]; s->shadow_rays += c[ST_SHADOW]; s->reflection_rays += c[ST_REFLECTION]; s->shaded_hits += c[ST_SHADED];
    // device leaf kinds -> ftb_prim_kind slots.  A cube and a solidCylinder are one fused leaf each.
    static const int slot[kLeafKinds] = {FTB_PRIM_SPHERE, FTB_PRIM_PLANE, FTB_PRIM_SQUARE, FTB_PRIM_CIRCLE, FTB_PRIM_CYLINDER, FTB_PRIM_CONE, FTB_PRIM_CUBE, FTB_PRIM_TRIANGLE, FTB_PRIM_BSPMESH,
                                         FTB_PRIM_SOLIDCYLINDER};
    for (int k = 0; k < kLeafKinds; ++k) s->leaf_tests[slot[k]] += c[ST_LEAF0 + k];
    s->leaf_tests[FTB_PRIM_TRIANGLE] += c[ST_TRI_TESTS_IN_MESH];
    s->transformed_leaf_tests += c[ST_XFORM]; s->bsp_nodes_visited += c[ST_BSP_NODES]; s->bound_tests += c[ST_BOUND_TESTS] + c[ST_BOUND_FAST]; s->csg_ops += c[ST_CSG_OPS];
    // algorithmic flops, SURVEY.md 8(d) table (FMA = 2; compares / selects = 0)
    static const double F[kLeafKinds] = {28, 8, 8, 8, 26, 32, 20, 45, 0, 42};  // solidCylinder: side + 2 caps in one frame
    double f = 0;
    for (int k = 0; k < kLeafKinds; ++k) f += F[k] * (double)c[ST_LEAF0 + k];
    f += 45.0 * (double)c[ST_TRI_TESTS_IN_MESH] + 33.0 * (double)c[ST_XFORM] + 12.0 * (double)c[ST_BSP_NODES] + 17.0 * (double)c[ST_BOUND_TESTS]   // bound test: 3 sub + 2 dot (5 each) + 2 FMA
         + 5.0 * (double)c[ST_BOUND_FAST];  // common-origin form: one dot
    f += (double)c[ST_SHADED] * (60.0 + 110.0 * (double)sc.lights.size()) + 18.0 * (double)c[ST_REFLECTION];
    s->flops += f;
}

// Bands of tile rows for the host-buffer path: band k = tile rows [bandFirstRow(k), bandFirstRow(k + 1)).  The D2H copy
// of band k overlaps the rendering of band k + 1, so only the LAST band's copy is exposed: the bands shrink towards
// the end (30 / 30 / 25 / 15 % for four bands).
inline int bandFirstRow(int k, int n, int tiles_y)
{
    if (k <= 0) return 0;
    if (k >= n) return tiles_y;
    if (n == 4) { static const double cum[5] = {0.0, 0.30, 0.60, 0.85, 1.0}; return (int)(cum[k] * tiles_y + 0.5); }
    return (int)(((long long)k * tiles_y) / n);
}
inline int bandOfRow(int row, int n, int tiles_y)
{
    int k = 0;
    while (k + 1 < n && row >= bandFirstRow(k + 1, n, tiles_y)) ++k;
    return k;
}
// band k of n = pixel rows [bandPixelRow(k), bandPixelRow(k + 1))
inline int bandPixelRow(int k, int n, int tiles_y, int height) { return std::min(height, bandFirstRow(k, n, tiles_y) * FTB_TILE_H); }

// Longest-processing-time-first tile order.  The persistent kernel hands tiles out from an atomic queue; a lane
// keeps its pixel for all samples and all bounce generations, so the last tiles handed out set the tail.  A
// static estimate - the projected bounding spheres of the items, weighted by how much work a hit on them
// causes (CSG programs, reflective surfaces spawn up to recursion_limit more generations), tiles.h - puts the costly
// tiles first, so the tail consists of cheap ones.  Ordering cannot change any pixel: tiles are independent.
// Clear tiles (tiles.h: no primary sample hits anything, by the items' spheres and boxes, clear_boxes.h) go last in each chunk, from chunk_clear[k] on: the kernel writes
// their pixels without tracing.
// lit / lit_leaf: the window's lit ground tiles (lit_tiles.h), items: the window's per-tile item masks (tiles.h), both indexed by
// the window's tile, not the shard's.  items is left empty when there are none or when they do not pay: they must leave at most
// kTileMaskKept of the bits the spheres alone keep in the traced tiles, or the FT_TMASK instance's extra path costs more than they
// save (measured, profiles/r7a_tile_items_ab.txt: repeat keeps 0.41 of them and runs 6.0 % faster; house keeps 0.61 and night-house
// 0.81, and both run 1.5 % and 5.0 % slower with the masks).
constexpr double kTileMaskKept = 0.5;
// Returns false when every tile has the same estimate and none is clear (no order needed).
bool computeTileOrder(const ftb_scene& sc, const ftb_camera& c, const ftb_render_params& p, const FrameGeom& g, int n_chunks, std::vector<int>& order,
                      std::vector<int>& chunk_first, std::vector<int>& chunk_clear, std::vector<unsigned char>& lit, int& lit_leaf, std::vector<unsigned>& items)
{
    std::vector<float> cost;
    std::vector<unsigned char> clear;
    const TileGrid grid = {g.wx0, g.wy0, g.ww, g.wh, g.tiles_x, g.tiles_y};
    const std::vector<ImageRect> boxes = itemBoxRects(sc.L, c, p.width, p.height);
    double kept = 1.0;
    const bool any = estimateTiles(sc.L, (int)sc.lights.size(), c, p.width, p.height, p.recursion_limit, sampleOffsetExtent(p), grid, cost, clear, &boxes, &items, &kept);
    if (kept > kTileMaskKept) items.clear();
    lit_leaf = litTiles(sc.L, sc.lights.data(), (int)sc.lights.size(), c, p.width, p.height, sampleOffsetExtent(p), grid, lit);
    // chunks = bands of tile rows (only used unsharded), see bandFirstRow
    auto tileOf = [&](int l) { return tileOfLocal(l, g.shard_index, g.shard_count); };
    auto chunkOf = [&](int l) { return n_chunks <= 1 ? 0 : bandOfRow(std::min(tileOf(l), g.n_tiles - 1) / g.tiles_x, n_chunks, g.tiles_y); };
    auto clearOf = [&](int l) { const int t = tileOf(l); return t < g.n_tiles && clear[(size_t)t]; };
    chunk_first.assign((size_t)n_chunks + 1, 0);
    int n_clear = 0;
    for (int l = 0; l < g.n_local_tiles; ++l) { chunk_first[(size_t)chunkOf(l) + 1]++; n_clear += clearOf(l) ? 1 : 0; }
    for (int k = 0; k < n_chunks; ++k) chunk_first[(size_t)k + 1] += chunk_first[(size_t)k];
    chunk_clear.assign(chunk_first.begin() + 1, chunk_first.end());
    if (!any && n_clear == 0 && n_chunks <= 1) return false;
    order.resize((size_t)g.n_local_tiles);
    for (int l = 0; l < g.n_local_tiles; ++l) order[l] = l;
    auto costOf = [&](int l) { const int t = tileOf(l); return t < g.n_tiles ? cost[(size_t)t] : 0.0f; };
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        const int ca = chunkOf(a), cb = chunkOf(b);
        if (ca != cb) return ca < cb;
        const bool za = clearOf(a), zb = clearOf(b);
        return za != zb ? zb : costOf(a) > costOf(b);
    });
    for (int l = 0; l < g.n_local_tiles; ++l)
        if (clearOf(l)) chunk_clear[(size_t)chunkOf(l)]--;
    return true;
}

// The frame's sample offsets on the device (F.jitter).  CornerSampling.generateRays (Image.fs:128-132): every corner ray uses the
// offset (-0.5, +0.5).
template <typename R>
int uploadJitter(PerDevice* pd, const ftb_render_params* p, const FrameGeom& g, DevFrame<R>& F, cudaStream_t stream)
{
    std::vector<R> j = {R(-0.5), R(0.5)};
    if (!g.corner) j.assign(p->jitter_xy, p->jitter_xy + 2 * (size_t)g.spp);
    CK(pd->jitter.reserve(j.size() * sizeof(R)));
    CK(cudaMemcpyAsync(pd->jitter.p, j.data(), j.size() * sizeof(R), cudaMemcpyHostToDevice, stream));  // pageable source: staged before return
    F.jitter = static_cast<const R*>(pd->jitter.p);
    return FTB_OK;
}

// Runs fn(R()) with R the real type of `precision`.
template <typename Fn> int byPrecision(int precision, Fn&& fn) { return precision == FTB_PRECISION_FP64_VERIFY ? fn(double()) : fn(float()); }

// The kernel launches of one frame on the CURRENT device.  begin() does what both modes share; a mode-0 frame (one shard of a
// camera grid) is then set up by prepareFrame, launched one chunk (band of tile rows) at a time by launchChunk and closed by
// finishFrame.  Everything is queued on the given stream; nothing here synchronises unless the tile order changes.
template <typename R>
struct Launch {
    PerDevice* pd = nullptr;
    const DevScene<R>* scene = nullptr;  // this device's copy
    const Variant<R>* var = nullptr;
    DevFrame<R> F;
    bool counting = false;  // the counting kernel: stats asked for with collect_stats
    int launches = 0;
    // The scene on this device (uploaded on first use), the DevFrame fields of both modes and the variant that covers `need`.
    int begin(ftb_scene* sc, PerDevice* pd, const ftb_render_params* p, unsigned need, bool counting, void* out, const ftb_debug_out* dbg)
    {
        SceneStorage<R>& st = storageOf<R>(pd);
        if (!st.ready) { int rc = uploadScene<R>(*sc, st); if (rc != FTB_OK) return rc; }
        CK(pd->control.reserve());
        this->pd = pd; this->counting = counting; scene = &st.view;
        std::memset(&F, 0, sizeof(F));
        F.recursion_limit = p->recursion_limit; F.seed = p->seed; F.out = static_cast<R*>(out);
        if (dbg) { F.dbg_prim = dbg->prim_id; F.dbg_sub = dbg->sub_id; F.dbg_t = dbg->t; }
        pd->control.wire(F);
        var = pickVariant<R>(need, counting);
        return var ? FTB_OK : fail(FTB_ERR_UNSUPPORTED, "no kernel variant covers this scene's feature mask");
    }
    cudaError_t launchKernel(cudaStream_t s) { return var->launch(*scene, F, counting, pd->sm_count, s, &launches); }
    int prepareFrame(ftb_scene* sc, PerDevice* pd, const ftb_camera* cam, const ftb_render_params* p, const FrameGeom& g, void* d_tiles,
                     const ftb_debug_out* d_dbg, ftb_stats* stats, cudaStream_t stream, int n_chunks)
    {
        int rc = begin(sc, pd, p, sc->L.features | (cam->has_focus ? (unsigned)FT_RNG : 0u), stats && p->collect_stats, d_tiles, d_dbg);
        if (rc != FTB_OK) return rc;
        CK(pd->control.prepare(counting, stream));
        F.mode = 0; F.gw = g.gw; F.gh = g.gh; F.spp = g.spp; F.tiles_x = g.tiles_x;
        F.wx0 = g.wx0; F.wy0 = g.wy0; F.wx1 = g.wx0 + g.ww; F.wy1 = g.wy0 + g.wh; F.dbg_w = g.ww;
        // floor(2^32 / tiles_x) + 1 does not fit 32 bits for tiles_x == 1 (windows <= 16 sample columns wide): those divide
        F.tiles_x_magic = (g.tiles_x > 1 && (unsigned long long)g.n_tiles * (unsigned long long)g.tiles_x < (1ull << 32)) ? (unsigned)((1ull << 32) / (unsigned)g.tiles_x) + 1u : 0u;
        F.n_local_tiles = g.n_local_tiles; F.shard_index = g.shard_index; F.shard_count = g.shard_count;
        fillCamera<R>(F, *cam, p->width, p->height);
        if ((rc = uploadJitter<R>(pd, p, g, F, stream)) != FTB_OK) return rc;
        // tile order: cached per (camera, frame geometry, window, recursion limit, sample offsets); recomputed + uploaded only
        // when they change.  The order lists the window's local tiles: an order cached for another window would name tiles this
        // one lacks.  Which tiles are clear depends on how far the samples stray from their pixel centres.
        const double offset = sampleOffsetExtent(*p);
        std::vector<unsigned char> key(sizeof(ftb_camera) + 11 * sizeof(int) + sizeof(double));
        std::memcpy(key.data(), cam, sizeof(ftb_camera));
        const int kk[11] = {p->width, p->height, p->sampling, g.shard_index, g.shard_count, p->recursion_limit, n_chunks, g.wx0, g.wy0, g.ww, g.wh};
        std::memcpy(key.data() + sizeof(ftb_camera), kk, sizeof(kk));
        std::memcpy(key.data() + sizeof(ftb_camera) + sizeof(kk), &offset, sizeof(offset));
        if (key != pd->order_key) {
            std::vector<int> order;
            std::vector<unsigned char> lit;
            std::vector<unsigned> items;
            pd->order_valid = computeTileOrder(*sc, *cam, *p, g, n_chunks, order, pd->chunk_first, pd->chunk_clear, lit, pd->lit_leaf, items);
            if (pd->order_valid) {
                CK(pd->order.reserve(order.size() * sizeof(int)));
                CK(cudaMemcpyAsync(pd->order.p, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice, stream));
            }
            if (pd->lit_leaf >= 0) {
                CK(pd->lit.reserve(lit.size()));
                CK(cudaMemcpyAsync(pd->lit.p, lit.data(), lit.size(), cudaMemcpyHostToDevice, stream));
            }
            pd->items_valid = !items.empty();
            if (pd->items_valid) {
                CK(pd->items.reserve(items.size() * sizeof(unsigned)));
                CK(cudaMemcpyAsync(pd->items.p, items.data(), items.size() * sizeof(unsigned), cudaMemcpyHostToDevice, stream));
            }
            // `order`, `lit` and `items` are pageable locals
            if (pd->order_valid || pd->lit_leaf >= 0 || pd->items_valid) CK(cudaStreamSynchronize(stream));
            pd->order_key.swap(key);
        }
        F.lit_tiles = pd->lit_leaf >= 0 ? static_cast<const unsigned char*>(pd->lit.p) : nullptr;
        F.lit_leaf = pd->lit_leaf;
        // the masks are proven for the FP32 kernels' rounding (tiles.h, clear_boxes.h); the FP64 build and the counting kernel
        // trace every item
        if (pd->items_valid) {
            if (const Variant<R>* m = withTileMasks<R>(var)) { var = m; F.tile_items = static_cast<const unsigned*>(pd->items.p); }
        }
        if (stats) CK(cudaEventRecord(pd->ev0, stream));
        return FTB_OK;
    }
    // One launch covers at most UnitCap samples per pixel; more samples = more passes over the same tiles (pixels), each continuing
    // the left fold of the previous one (so the blend order is still Array.average's).  setPass sets up the pass that starts at
    // sample s_base: for frames (launchChunk) and for ftb_shade_samples alike, so both cut a pixel's samples into the same passes,
    // runs and fold segments.
    void setPass(int s_base)
    {
        F.s_base = s_base;
        F.s_count = std::min(var->unit_cap, F.spp - s_base);
        // run length: cheap samples amortise the dealing over up to 8 consecutive samples of a pixel, as long as
        // every pixel still splits into >= 8 runs (the chain a lane can be stuck with stays 1/8 of a pixel)
        // Large meshes deal single samples: a traversal's cost varies so much between neighbouring samples that a lane
        // stuck with a run of them holds its warp back (measured -11..-14 % on the 355 k mesh; +3 % on the 960-triangle
        // one and +7 % on moon the other way).
        const int runMax = scene->mesh_packet ? 1 : 8;
        int run = 1;
        while (run < runMax && F.s_count % (run * 2) == 0 && F.s_count / (run * 2) >= 8) run *= 2;
        F.run = run;
        const unsigned rpp = (unsigned)(F.s_count / run);
        F.rpp_magic = rpp <= 1 ? 0u : (unsigned)((1ull << 32) / rpp) + 1u;
    }
    // Work-queue granularity.  A lane takes runs of samples, a warp takes blocks of pixels from the atomic queue.  The block is
    // the indivisible quantum of the tail, so it shrinks (32 = 8x4 ... 1 pixel) until there are >= 24 blocks per resident
    // warp, but never below one warp-round of samples per block (and big frames keep big blocks, which also bounds the number
    // of atomics on the queue counter).
    int launchChunk(int chunk, cudaStream_t stream)
    {
        const int first = pd->chunk_first[(size_t)chunk], ntile = pd->chunk_first[(size_t)chunk + 1] - first;
        if (ntile <= 0) return FTB_OK;
        F.tile_order = pd->order_valid ? static_cast<const int*>(pd->order.p) + first : nullptr;
        const int traced = pd->order_valid ? pd->chunk_clear[(size_t)chunk] - first : ntile;  // the tiles before the clear ones
        const long long warps = (long long)pd->sm_count * 5 * (kBlockThreads / 32);
        const long long pixels = (long long)ntile * FTB_TILE_PIXELS;
        int ppb = 32;
        while (ppb > 1 && pixels / ppb < 24 * warps && (long long)(ppb / 2) * F.spp >= 32) ppb /= 2;
        int bw = ppb >= 8 ? 8 : ppb, bh = ppb / bw;
        F.bw_log = bw == 8 ? 3 : (bw == 4 ? 2 : (bw == 2 ? 1 : 0));
        F.bh_log = bh == 4 ? 2 : (bh == 2 ? 1 : 0);
        F.n_blocks = traced * (FTB_TILE_PIXELS / ppb);
        F.n_clear_blocks = (ntile - traced) * (FTB_TILE_PIXELS / ppb);
        for (int s_base = 0; s_base < F.spp; s_base += var->unit_cap) {
            setPass(s_base);
            CK(pd->control.resetQueue(stream));
            CK(launchKernel(stream));
            if (F.n_clear_blocks > 0) {
                const int grid = (int)std::min<long long>((F.n_clear_blocks + 3) / 4, (long long)pd->sm_count * 16);
                clear_kernel<R><<<grid, 128, 0, stream>>>(F, counting ? 1 : 0);
                CK(cudaGetLastError());
                ++launches;
            }
        }
        return FTB_OK;
    }
    int finishFrame(ftb_stats* stats, cudaStream_t stream)
    {
        if (stats) { CK(cudaEventRecord(pd->ev1, stream)); stats->kernel_launches += launches + 1; }  // + the control-block memset
        return FTB_OK;
    }
};

int overflowError() { return fail(FTB_ERR_HIT_OVERFLOW, "a CSG operand produced more than 32 crossings on one ray"); }

// Reads the control block back (synchronises the stream) and, with stats, folds its counters and the kernel time into them.
int finishStats(ftb_scene* sc, PerDevice* pd, ftb_stats* stats, cudaStream_t stream, bool* overflow)
{
    Control h;
    CK(pd->control.read(h, stream));
    if (h.overflow) *overflow = true;
    if (stats) {
        fillStats(h, *sc, stats);
        if (h.overflow) stats->hit_overflow = 1;
        float ms = 0; CK(cudaEventElapsedTime(&ms, pd->ev0, pd->ev1)); if ((double)ms > stats->kernel_ms) stats->kernel_ms = ms;
    }
    return FTB_OK;
}

int launchAssemble(const ftb_render_params* p, const FrameGeom& g, const void* const* bufs, void* d_out, cudaStream_t stream, int y0, int y1)
{
    TilePtrs tp;
    std::memset(&tp, 0, sizeof(tp));
    for (int i = 0; i < g.shard_count; ++i) tp.p[i] = bufs[i];
    const long long n = (long long)g.width * (y1 - y0);
    if (n <= 0) return FTB_OK;
    int grid = (int)std::min<long long>((n + 255) / 256, 148 * 16);
    return byPrecision(p->precision, [&](auto r) -> int {
        assemble_kernel<decltype(r)><<<grid, 256, 0, stream>>>(tp, g.shard_count, g.tiles_x, g.width, y0, y1, g.corner ? 1 : 0, p->out_format, d_out);
        CK(cudaGetLastError());
        return FTB_OK;
    });
}

// bytes of the window's pixels in out_format
inline size_t outBytes(int out_format, const FrameGeom& g)
{
    const size_t n = (size_t)g.width * g.height;
    return out_format == FTB_OUT_RGB_F64 ? n * 24 : (out_format == FTB_OUT_RGB_F32 ? n * 12 : n * 4);
}

// CUDA ordinals of the devices this library runs on (compute capability 10.x), in ordinal order: what ftb_device_count
// counts and what ftb_render(n_gpus = N) uses, so that the two agree on a box with other GPUs in it.
std::vector<int> b200Devices()
{
    std::vector<int> out;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return out; }
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) out.push_back(d);
    }
    return out;
}

struct DeviceRestore {
    int dev = -1;
    DeviceRestore() { if (cudaGetDevice(&dev) != cudaSuccess) dev = -1; }
    ~DeviceRestore() { if (dev >= 0) cudaSetDevice(dev); }
};

int currentDevice(ftb_scene* sc, PerDevice** out)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { (void)cudaGetLastError(); return fail(FTB_ERR_NO_DEVICE, "no CUDA device"); }
    return getDevice(sc, dev, out);
}

// BspMesh.fs:30-65 builds the reference's tree; the device's own index over the same triangles is built here: on the GPU for
// large meshes (bvh_build.cu), on the host for small ones and as the fallback
int buildMeshIndex(const ftb_scene_desc& desc, ftb_scene& sc)
{
    std::vector<std::vector<int32_t>> order;
    ftb::enumerateMeshes(desc, sc.L, order);
    size_t meshTriangles = 0;
    for (const auto& o : order) meshTriangles += o.size();
    bool done = false;
    if (meshTriangles >= kLargeMesh) {
        const int radii[3] = {16, 8, 4};
        for (int k = 0; k < 3 && !done; ++k) {
            std::string why;
            done = ftb::buildMeshIndexDevice(desc.triangles, desc.n_triangles, order, ftb::kBspStack, radii[k], sc.L, sc.bvh_stats, why);
            if (!done && std::getenv("FTB_VERBOSE")) std::fprintf(stderr, "functracer_b200: device BVH build not used (%s)\n", why.c_str());
        }
        sc.bvh_on_device = done;
    }
    if (!done) {
        const auto t0 = std::chrono::steady_clock::now();
        ftb::buildMeshIndexHost(desc, sc.L);
        sc.bvh_stats.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    if (sc.L.max_bvh_depth + 2 > ftb::kBspStack) return fail(FTB_ERR_UNSUPPORTED, "mesh index deeper than the 64-entry traversal stack");
    if (largeMesh(sc.L)) sc.L.features |= (unsigned)FT_MESHPK;  // the warp-packet walk (render.cuh)
    return FTB_OK;
}

// One device's part of an ftb_render frame; the primary device's assembly reads its tiles from `gather` (== target if direct).
struct Shard { PerDevice* pd; FrameGeom g; ftb_render_params ps; ftb_debug_out dbg; void* target; void* gather; bool direct; };

// Device k's shard of the window `win`: geometry, tile buffer, band events, debug planes (buffers sized by the window).  Shards of the other devices: the render kernel's fold
// stores finished pixels straight into a buffer on the primary device over NVLink (peer access), so there is no gather step;
// without peer access the shard is rendered locally and every finished band is copied with cudaMemcpyPeerAsync.
int setUpShard(ftb_scene* sc, const ftb_render_params& p, const Window& win, const FrameGeom& full, const ftb_debug_out* dbg, const std::vector<int>& devs, int kBands,
               std::vector<Shard>& sh, int k)
{
    const int dev = devs[(size_t)k], primary = devs[0], n_gpus = (int)devs.size();
    CK(cudaSetDevice(dev));
    Shard& S = sh[(size_t)k];
    int rc = getDevice(sc, dev, &S.pd);
    if (rc != FTB_OK) return rc;
    PerDevice* pd = S.pd;
    S.ps = p; S.ps.shard_index = n_gpus > 1 ? k : 0; S.ps.shard_count = n_gpus;
    if ((rc = frameGeom(&S.ps, S.g, &win)) != FTB_OK) return rc;
    const size_t tileBytes = (size_t)S.g.n_local_tiles * FTB_TILE_PIXELS * 3 * realSize(p.precision);
    CK(pd->tiles.reserve(tileBytes));
    while ((int)pd->band_events.size() < kBands) {
        cudaEvent_t e;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        pd->band_events.push_back(e);
    }
    S.dbg = {nullptr, nullptr, nullptr};
    if (dbg && dbg->prim_id) {
        CK(pd->dbg_prim.reserve((size_t)full.n_samples * 4));
        CK(cudaMemsetAsync(pd->dbg_prim.p, 0xff, (size_t)full.n_samples * 4, pd->stream));
        S.dbg.prim_id = static_cast<int32_t*>(pd->dbg_prim.p);
        if (dbg->sub_id) { CK(pd->dbg_sub.reserve((size_t)full.n_samples * 4)); CK(cudaMemsetAsync(pd->dbg_sub.p, 0, (size_t)full.n_samples * 4, pd->stream)); S.dbg.sub_id = static_cast<int32_t*>(pd->dbg_sub.p); }
        if (dbg->t) { CK(pd->dbg_t.reserve((size_t)full.n_samples * 8)); CK(cudaMemsetAsync(pd->dbg_t.p, 0, (size_t)full.n_samples * 8, pd->stream)); S.dbg.t = static_cast<double*>(pd->dbg_t.p); }
    }
    S.target = S.gather = pd->tiles.p; S.direct = false;
    if (k > 0) {
        PerDevice* p0 = sh[0].pd;
        if ((int)p0->peer_tiles.size() < n_gpus) p0->peer_tiles.resize((size_t)n_gpus);
        CK(cudaSetDevice(primary));
        CK(p0->peer_tiles[(size_t)k].reserve(tileBytes));
        CK(cudaSetDevice(dev));
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, dev, primary) == cudaSuccess && can) {
            cudaError_t pe = cudaDeviceEnablePeerAccess(primary, 0);
            if (pe == cudaSuccess || pe == cudaErrorPeerAccessAlreadyEnabled) S.direct = true;
            (void)cudaGetLastError();
        }
        S.gather = p0->peer_tiles[(size_t)k].p;
        if (S.direct) S.target = S.gather;
    }
    return FTB_OK;
}

// ---- ray queries ---------------------------------------------------------------------------------------------------
// The arguments every query entry point checks before it touches a device.  occlusion: max_t and blocked are required.
int checkQuery(const ftb_scene* sc, const double* rays, const double* max_t, int64_t n, const ftb_render_params* p, bool occlusion,
               const int32_t* blocked)
{
    if (!sc || !p || n < 0 || (n > 0 && (!rays || (occlusion && (!max_t || !blocked))))) return fail(FTB_ERR_BAD_ARG, "null argument or negative ray count");
    if (p->precision != FTB_PRECISION_FP32 && p->precision != FTB_PRECISION_FP64_VERIFY) return fail(FTB_ERR_BAD_ARG, "bad precision");
    if (n > 32LL * 0x7fffffffLL) return fail(FTB_ERR_BAD_ARG, "too many rays");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { (void)cudaGetLastError(); return fail(FTB_ERR_NO_DEVICE, "no CUDA device: functracer_b200 has no CPU path"); }
    return FTB_OK;
}

// The device entry points: one batch of queries (device pointers) queued on `s` on the current device, with the scene's own
// variant (the one its frames run) and the per-device control block (queue counter, overflow flag, counters).  Nothing here
// synchronises except the control block's read-back when stats are asked for.
// occlusion: queries into `blocked` up to max_t, else nearest-hit queries into the planes of `out` (may be null).
int queryDevice(ftb_scene* sc, bool occlusion, const double* rays, const double* max_t, int64_t n, const ftb_render_params* p,
                const ftb_hit_out* out, int32_t* blocked, ftb_stats* stats, cudaStream_t s)
{
    int rc = checkQuery(sc, rays, max_t, n, p, occlusion, blocked);
    if (rc != FTB_OK) return rc;
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (n == 0) return FTB_OK;
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    rc = byPrecision(p->precision, [&](auto r) -> int {
        Launch<decltype(r)> fr;
        int e = fr.begin(sc, pd, p, sc->L.features, stats && p->collect_stats, nullptr, nullptr);
        if (e != FTB_OK) return e;
        CK(pd->control.prepare(fr.counting, s));
        CK(pd->control.resetQueue(s));
        DevQuery q;
        std::memset(&q, 0, sizeof(q));
        q.rays = rays; q.n = n; q.n_groups = (int)((n + 31) / 32);
        if (occlusion) {
            q.max_t = max_t; q.blocked = blocked;
        } else if (out) {
            q.t = out->t; q.prim = out->prim_id; q.sub = out->sub_id;
            q.p = out->p; q.normal = out->normal; q.colour = out->colour; q.surface = out->surface;
        }
        q.record = (q.p || q.normal || q.colour || q.surface) ? 1 : 0;
        Control* c = pd->control.ctl();
        q.group_counter = &c->tile_counter; q.overflow = &c->overflow; q.stats = c->stats;
        if (stats) CK(cudaEventRecord(pd->ev0, s));
        CK(fr.var->query(*fr.scene, q, fr.counting, pd->sm_count, s, &fr.launches));
        if (stats) { CK(cudaEventRecord(pd->ev1, s)); stats->kernel_launches += fr.launches + 1; }  // + the control-block memset
        return FTB_OK;
    });
    if (rc != FTB_OK) return rc;
    bool overflow = false;
    if (stats && (rc = finishStats(sc, pd, stats, s, &overflow)) != FTB_OK) return rc;
    return overflow ? overflowError() : FTB_OK;
}

// The host entry points: a thin wrapper around queryDevice.  The rays (and max_t) are uploaded on the scene's stream, the
// device entry point queues the queries there, the control block is read back (queryDevice does that itself when it fills
// stats) and only then are the requested planes downloaded: on an overflow the caller's arrays are not written.  Synchronous.
int queryHost(ftb_scene* sc, bool occlusion, const double* rays, const double* max_t, int64_t n, const ftb_render_params* p,
              const ftb_hit_out* out, int32_t* blocked, ftb_stats* stats)
{
    const auto t0 = std::chrono::steady_clock::now();
    int rc = checkQuery(sc, rays, max_t, n, p, occlusion, blocked);  // before the uploads read the caller's arrays
    if (rc != FTB_OK || n == 0) return rc != FTB_OK ? rc : queryDevice(sc, occlusion, rays, max_t, n, p, out, blocked, stats, nullptr);
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    const cudaStream_t s = pd->stream;
    CK(pd->rays.reserve((size_t)n * 48));
    CK(cudaMemcpyAsync(pd->rays.p, rays, (size_t)n * 48, cudaMemcpyHostToDevice, s));
    // every host array of the call with its bytes per ray: max_t (in) and blocked, or the requested planes; one device buffer
    struct Plane { void* host; size_t per_ray; void* dev; };
    const ftb_hit_out none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    const ftb_hit_out& o = out ? *out : none;
    Plane planes[7] = {{o.t, 8, nullptr}, {o.prim_id, 4, nullptr}, {o.sub_id, 4, nullptr}, {o.p, 24, nullptr},
                       {o.normal, 24, nullptr}, {o.colour, 24, nullptr}, {o.surface, 32, nullptr}};
    const int np = occlusion ? 2 : 7;
    if (occlusion) { planes[0] = {const_cast<double*>(max_t), 8, nullptr}; planes[1] = {blocked, 4, nullptr}; }
    size_t bytes = 0;
    for (int k = 0; k < np; ++k) if (planes[k].host) bytes += ((planes[k].per_ray * (size_t)n + 255) & ~(size_t)255);
    CK(pd->query.reserve(std::max<size_t>(bytes, 1)));
    size_t at = 0;
    for (int k = 0; k < np; ++k)
        if (planes[k].host) { planes[k].dev = static_cast<char*>(pd->query.p) + at; at += ((planes[k].per_ray * (size_t)n + 255) & ~(size_t)255); }
    const double* d_rays = static_cast<const double*>(pd->rays.p);
    if (occlusion) {
        CK(cudaMemcpyAsync(planes[0].dev, max_t, (size_t)n * 8, cudaMemcpyHostToDevice, s));
        rc = queryDevice(sc, true, d_rays, static_cast<const double*>(planes[0].dev), n, p, nullptr, static_cast<int32_t*>(planes[1].dev), stats, s);
    } else {
        const ftb_hit_out d = {static_cast<double*>(planes[0].dev), static_cast<int32_t*>(planes[1].dev), static_cast<int32_t*>(planes[2].dev),
                               static_cast<double*>(planes[3].dev), static_cast<double*>(planes[4].dev), static_cast<double*>(planes[5].dev),
                               static_cast<double*>(planes[6].dev)};
        rc = queryDevice(sc, false, d_rays, nullptr, n, p, &d, nullptr, stats, s);
    }
    if (rc == FTB_OK && !stats) {  // with stats queryDevice has read the control block (and reported an overflow) already
        bool overflow = false;
        rc = finishStats(sc, pd, nullptr, s, &overflow);
        if (rc == FTB_OK && overflow) rc = overflowError();
    }
    if (rc != FTB_OK) return rc;
    for (int k = occlusion ? 1 : 0; k < np; ++k)
        if (planes[k].host) CK(cudaMemcpyAsync(planes[k].host, planes[k].dev, planes[k].per_ray * (size_t)n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (stats) stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return FTB_OK;
}

// ---- crossing queries -----------------------------------------------------------------------------------------------
// The arguments of a crossing query that the nearest / occlusion queries do not have, then checkQuery's (which ends with the
// device count): everything a caller can get wrong is reported before any device is looked for.
int checkCrossings(const ftb_scene* sc, const double* rays, int64_t n, int32_t max_hits, double t_min, double t_max, const ftb_render_params* p,
                   const int32_t* counts)
{
    if (max_hits < 1 || max_hits > FTB_MAX_CROSSINGS) return fail(FTB_ERR_BAD_ARG, "max_hits outside 1 .. FTB_MAX_CROSSINGS");
    if (t_min != t_min || t_max != t_max || !(t_min < t_max)) return fail(FTB_ERR_BAD_ARG, "t_min or t_max is NaN, or t_min >= t_max");
    if (n > 0 && !counts) return fail(FTB_ERR_BAD_ARG, "null argument: counts");
    return checkQuery(sc, rays, nullptr, n, p, false, nullptr);
}

// The device entry point: one batch of crossing queries (device pointers) queued on `s` on the current device, with the
// per-device control block, as queryDevice does for the other queries.  out may be null (counts only).
int crossingsDevice(ftb_scene* sc, const double* rays, int64_t n, int32_t max_hits, double t_min, double t_max, const ftb_render_params* p,
                    const ftb_hit_out* out, int32_t* counts, ftb_stats* stats, cudaStream_t s)
{
    int rc = checkCrossings(sc, rays, n, max_hits, t_min, t_max, p, counts);
    if (rc != FTB_OK) return rc;
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (n == 0) return FTB_OK;
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    rc = byPrecision(p->precision, [&](auto r) -> int {
        Launch<decltype(r)> fr;  // the scene on this device and the control block; the variant it picks is not used
        int e = fr.begin(sc, pd, p, sc->L.features, stats && p->collect_stats, nullptr, nullptr);
        if (e != FTB_OK) return e;
        CK(pd->control.prepare(fr.counting, s));
        CK(pd->control.resetQueue(s));
        DevCrossings q;
        std::memset(&q, 0, sizeof(q));
        q.rays = rays; q.n = n; q.n_groups = (int)((n + 31) / 32);
        q.max_hits = max_hits; q.t_min = t_min; q.t_max = t_max; q.counts = counts;
        if (out) {
            q.t = out->t; q.prim = out->prim_id; q.sub = out->sub_id;
            q.p = out->p; q.normal = out->normal; q.colour = out->colour; q.surface = out->surface;
        }
        q.record = (q.p || q.normal || q.colour || q.surface) ? 1 : 0;
        Control* c = pd->control.ctl();
        q.group_counter = &c->tile_counter; q.overflow = &c->overflow; q.stats = c->stats;
        if (stats) CK(cudaEventRecord(pd->ev0, s));
        CK(launchCrossings(*fr.scene, q, fr.counting, pd->sm_count, s, &fr.launches));
        if (stats) { CK(cudaEventRecord(pd->ev1, s)); stats->kernel_launches += fr.launches + 1; }  // + the control-block memset
        return FTB_OK;
    });
    if (rc != FTB_OK) return rc;
    bool overflow = false;
    if (stats && (rc = finishStats(sc, pd, stats, s, &overflow)) != FTB_OK) return rc;
    return overflow ? overflowError() : FTB_OK;
}

// The host entry point, the pattern of queryHost: upload the rays, queue the device entry, read the control block back, and
// only then download counts and the requested planes (max_hits entries per ray): on an overflow nothing of the caller's is written.
int crossingsHost(ftb_scene* sc, const double* rays, int64_t n, int32_t max_hits, double t_min, double t_max, const ftb_render_params* p,
                  const ftb_hit_out* out, int32_t* counts, ftb_stats* stats)
{
    const auto t0 = std::chrono::steady_clock::now();
    int rc = checkCrossings(sc, rays, n, max_hits, t_min, t_max, p, counts);
    if (rc != FTB_OK || n == 0) return rc != FTB_OK ? rc : crossingsDevice(sc, rays, n, max_hits, t_min, t_max, p, out, counts, stats, nullptr);
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    const cudaStream_t s = pd->stream;
    CK(pd->rays.reserve((size_t)n * 48));
    CK(cudaMemcpyAsync(pd->rays.p, rays, (size_t)n * 48, cudaMemcpyHostToDevice, s));
    // counts, then the requested planes with their bytes per ray; one device buffer
    struct Plane { void* host; size_t per_ray; void* dev; };
    const ftb_hit_out none = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    const ftb_hit_out& o = out ? *out : none;
    const size_t k = (size_t)max_hits;
    Plane planes[8] = {{counts, 4, nullptr}, {o.t, 8 * k, nullptr}, {o.prim_id, 4 * k, nullptr}, {o.sub_id, 4 * k, nullptr}, {o.p, 24 * k, nullptr},
                       {o.normal, 24 * k, nullptr}, {o.colour, 24 * k, nullptr}, {o.surface, 32 * k, nullptr}};
    size_t bytes = 0;
    for (const Plane& pl : planes) if (pl.host) bytes += ((pl.per_ray * (size_t)n + 255) & ~(size_t)255);
    CK(pd->query.reserve(bytes));
    size_t at = 0;
    for (Plane& pl : planes)
        if (pl.host) { pl.dev = static_cast<char*>(pd->query.p) + at; at += ((pl.per_ray * (size_t)n + 255) & ~(size_t)255); }
    const ftb_hit_out d = {static_cast<double*>(planes[1].dev), static_cast<int32_t*>(planes[2].dev), static_cast<int32_t*>(planes[3].dev),
                           static_cast<double*>(planes[4].dev), static_cast<double*>(planes[5].dev), static_cast<double*>(planes[6].dev),
                           static_cast<double*>(planes[7].dev)};
    rc = crossingsDevice(sc, static_cast<const double*>(pd->rays.p), n, max_hits, t_min, t_max, p, &d, static_cast<int32_t*>(planes[0].dev), stats, s);
    if (rc == FTB_OK && !stats) {  // with stats crossingsDevice has read the control block (and reported an overflow) already
        bool overflow = false;
        rc = finishStats(sc, pd, nullptr, s, &overflow);
        if (rc == FTB_OK && overflow) rc = overflowError();
    }
    if (rc != FTB_OK) return rc;
    for (const Plane& pl : planes)
        if (pl.host) CK(cudaMemcpyAsync(pl.host, pl.dev, pl.per_ray * (size_t)n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (stats) stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return FTB_OK;
}

// ---- path queries ---------------------------------------------------------------------------------------------------
// The argument a path query adds (the recursion limit, which sizes its planes), then checkQuery's (which ends with the device
// count): everything a caller can get wrong is reported before any device is looked for.
int checkPaths(const ftb_scene* sc, const double* rays, int64_t n, const ftb_render_params* p)
{
    if (p && (p->recursion_limit < 0 || p->recursion_limit > FTB_MAX_PATH_LEVELS - 1)) return fail(FTB_ERR_BAD_ARG, "recursion_limit outside 0 .. FTB_MAX_PATH_LEVELS - 1");
    return checkQuery(sc, rays, nullptr, n, p, false, nullptr);
}

// The device entry point: one batch of path queries (device pointers) queued on `s` on the current device, with the per-device
// control block, as queryDevice does for the other queries.  out may be null (stats only).
int pathsDevice(ftb_scene* sc, const double* rays, const uint64_t* keys, int64_t n, const ftb_render_params* p, const ftb_path_out* out,
                ftb_stats* stats, cudaStream_t s)
{
    int rc = checkPaths(sc, rays, n, p);
    if (rc != FTB_OK) return rc;
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (n == 0) return FTB_OK;
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    rc = byPrecision(p->precision, [&](auto r) -> int {
        Launch<decltype(r)> fr;  // the scene on this device and the control block; the variant it picks is not used
        int e = fr.begin(sc, pd, p, sc->L.features, stats && p->collect_stats, nullptr, nullptr);
        if (e != FTB_OK) return e;
        CK(pd->control.prepare(fr.counting, s));
        CK(pd->control.resetQueue(s));
        DevPaths q;
        std::memset(&q, 0, sizeof(q));
        q.rays = rays; q.sample_keys = reinterpret_cast<const unsigned long long*>(keys); q.n = n; q.n_groups = (int)((n + 31) / 32);
        q.recursion_limit = p->recursion_limit; q.seed = p->seed;
        if (out) {
            q.levels = out->levels; q.colour = out->colour; q.ray_od = out->ray_od; q.weight = out->weight;
            q.t = out->hit.t; q.prim = out->hit.prim_id; q.sub = out->hit.sub_id;
            q.p = out->hit.p; q.normal = out->hit.normal; q.hit_colour = out->hit.colour; q.surface = out->hit.surface;
            q.intensity = out->intensity; q.light_dir = out->light_dir; q.light_colour = out->light_colour;
        }
        q.record = (q.p || q.normal || q.hit_colour || q.surface) ? 1 : 0;
        Control* c = pd->control.ctl();
        q.group_counter = &c->tile_counter; q.overflow = &c->overflow; q.stats = c->stats;
        if (stats) CK(cudaEventRecord(pd->ev0, s));
        CK(launchPaths(*fr.scene, q, fr.counting, pd->sm_count, s, &fr.launches));
        if (stats) { CK(cudaEventRecord(pd->ev1, s)); stats->kernel_launches += fr.launches + 1; }  // + the control-block memset
        return FTB_OK;
    });
    if (rc != FTB_OK) return rc;
    bool overflow = false;
    if (stats && (rc = finishStats(sc, pd, stats, s, &overflow)) != FTB_OK) return rc;
    return overflow ? overflowError() : FTB_OK;
}

// The host entry point, the pattern of crossingsHost: upload the rays and keys, queue the device entry, read the control block
// back, and only then download the requested planes (D = recursion_limit + 1 level entries per ray, D * L light entries): on an
// overflow nothing of the caller's is written.
int pathsHost(ftb_scene* sc, const double* rays, const uint64_t* keys, int64_t n, const ftb_render_params* p, const ftb_path_out* out,
              ftb_stats* stats)
{
    const auto t0 = std::chrono::steady_clock::now();
    int rc = checkPaths(sc, rays, n, p);
    if (rc != FTB_OK || n == 0) return rc != FTB_OK ? rc : pathsDevice(sc, rays, keys, n, p, out, stats, nullptr);
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    const cudaStream_t s = pd->stream;
    CK(pd->rays.reserve((size_t)n * 48));
    CK(cudaMemcpyAsync(pd->rays.p, rays, (size_t)n * 48, cudaMemcpyHostToDevice, s));
    // the keys (in), then the requested planes with their bytes per ray; one device buffer
    struct Plane { void* host; size_t per_ray; void* dev; };
    ftb_path_out o;
    std::memset(&o, 0, sizeof(o));
    if (out) o = *out;
    const size_t D = (size_t)p->recursion_limit + 1, DL = D * sc->lights.size();
    Plane planes[15] = {{const_cast<uint64_t*>(keys), 8, nullptr}, {o.levels, 4, nullptr}, {o.colour, 24, nullptr}, {o.ray_od, 48 * D, nullptr},
                        {o.weight, 8 * D, nullptr}, {o.hit.t, 8 * D, nullptr}, {o.hit.prim_id, 4 * D, nullptr}, {o.hit.sub_id, 4 * D, nullptr},
                        {o.hit.p, 24 * D, nullptr}, {o.hit.normal, 24 * D, nullptr}, {o.hit.colour, 24 * D, nullptr}, {o.hit.surface, 32 * D, nullptr},
                        {o.intensity, 8 * DL, nullptr}, {o.light_dir, 24 * DL, nullptr}, {o.light_colour, 24 * DL, nullptr}};
    size_t bytes = 0;
    for (const Plane& pl : planes) if (pl.host) bytes += ((pl.per_ray * (size_t)n + 255) & ~(size_t)255);
    CK(pd->query.reserve(std::max<size_t>(bytes, 1)));
    size_t at = 0;
    for (Plane& pl : planes)
        if (pl.host) { pl.dev = static_cast<char*>(pd->query.p) + at; at += ((pl.per_ray * (size_t)n + 255) & ~(size_t)255); }
    if (keys) CK(cudaMemcpyAsync(planes[0].dev, keys, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    ftb_path_out d;
    d.levels = static_cast<int32_t*>(planes[1].dev); d.colour = static_cast<double*>(planes[2].dev);
    d.ray_od = static_cast<double*>(planes[3].dev); d.weight = static_cast<double*>(planes[4].dev);
    d.hit = {static_cast<double*>(planes[5].dev), static_cast<int32_t*>(planes[6].dev), static_cast<int32_t*>(planes[7].dev),
             static_cast<double*>(planes[8].dev), static_cast<double*>(planes[9].dev), static_cast<double*>(planes[10].dev),
             static_cast<double*>(planes[11].dev)};
    d.intensity = static_cast<double*>(planes[12].dev); d.light_dir = static_cast<double*>(planes[13].dev);
    d.light_colour = static_cast<double*>(planes[14].dev);
    rc = pathsDevice(sc, static_cast<const double*>(pd->rays.p), static_cast<const uint64_t*>(planes[0].dev), n, p, &d, stats, s);
    if (rc == FTB_OK && !stats) {  // with stats pathsDevice has read the control block (and reported an overflow) already
        bool overflow = false;
        rc = finishStats(sc, pd, nullptr, s, &overflow);
        if (rc == FTB_OK && overflow) rc = overflowError();
    }
    if (rc != FTB_OK) return rc;
    for (int k = 1; k < 15; ++k)
        if (planes[k].host && planes[k].per_ray) CK(cudaMemcpyAsync(planes[k].host, planes[k].dev, planes[k].per_ray * (size_t)n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (stats) stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return FTB_OK;
}

// ---- a frame's own samples: ftb_frame_rays and ftb_shade_samples ----------------------------------------------------------
// ftb_frame_rays reads width, height, spp, sampling, jitter_xy, precision and seed; the window and those fields are checked as
// ftb_render_window checks them (frameGeom), the fields it does not read are not.  Then the device count: everything a caller can
// get wrong is reported before any device is looked for.
int checkFrameRays(const ftb_scene* sc, const ftb_camera* cam, const ftb_render_params* p, const Window& win, FrameGeom& g)
{
    if (!sc || !cam || !p) return fail(FTB_ERR_BAD_ARG, "null argument");
    ftb_render_params q = *p;
    q.out_format = FTB_OUT_RGB_F64; q.shard_index = q.shard_count = 0; q.band_index = q.band_count = 0; q.n_gpus = 0;
    int rc = frameGeom(&q, g, &win);
    if (rc != FTB_OK) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { (void)cudaGetLastError(); return fail(FTB_ERR_NO_DEVICE, "no CUDA device: functracer_b200 has no CPU path"); }
    return FTB_OK;
}

// The device entry point: the window's rays and keys (device pointers, either may be null) queued on `s` on the current device.
int frameRaysDevice(ftb_scene* sc, const ftb_camera* cam, const ftb_render_params* p, const Window& win, double* rays, uint64_t* keys, cudaStream_t s)
{
    FrameGeom g;
    int rc = checkFrameRays(sc, cam, p, win, g);
    if (rc != FTB_OK) return rc;
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    return byPrecision(p->precision, [&](auto r) -> int {
        typedef decltype(r) R;
        DevFrame<R> F;  // the fields primaryRay reads, filled as prepareFrame fills them
        std::memset(&F, 0, sizeof(F));
        F.gw = g.gw; F.gh = g.gh; F.spp = g.spp; F.seed = p->seed;
        F.wx0 = g.wx0; F.wy0 = g.wy0; F.wx1 = g.wx0 + g.ww; F.wy1 = g.wy0 + g.wh;
        fillCamera<R>(F, *cam, p->width, p->height);
        int e = uploadJitter<R>(pd, p, g, F, s);
        if (e != FTB_OK) return e;
        CK(launchFrameRays(F, g.n_samples, rays, reinterpret_cast<unsigned long long*>(keys), pd->sm_count, s));
        return FTB_OK;
    });
}

// The host entry point: the device entry into scratch on the scene's stream, then the downloads.  Synchronous.
int frameRaysHost(ftb_scene* sc, const ftb_camera* cam, const ftb_render_params* p, const Window& win, double* rays, uint64_t* keys)
{
    FrameGeom g;
    int rc = checkFrameRays(sc, cam, p, win, g);
    if (rc != FTB_OK) return rc;
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    const cudaStream_t s = pd->stream;
    const size_t n = (size_t)g.n_samples;
    if (rays) CK(pd->rays.reserve(n * 48));
    if (keys) CK(pd->query.reserve(n * 8));
    rc = frameRaysDevice(sc, cam, p, win, rays ? static_cast<double*>(pd->rays.p) : nullptr, keys ? static_cast<uint64_t*>(pd->query.p) : nullptr, s);
    if (rc != FTB_OK) return rc;
    if (rays) CK(cudaMemcpyAsync(rays, pd->rays.p, n * 48, cudaMemcpyDeviceToHost, s));
    if (keys) CK(cudaMemcpyAsync(keys, pd->query.p, n * 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    return FTB_OK;
}

inline size_t pixelBytes(int out_format) { return out_format == FTB_OUT_RGB_F64 ? 24 : (out_format == FTB_OUT_RGB_F32 ? 12 : 4); }

// ftb_shade_samples' arguments, then the device count: everything a caller can get wrong is reported before any device is looked
// for.  The pixel count is also bounded: the kernel indexes pixels with 32-bit integers.
int checkSamples(const ftb_scene* sc, const double* rays, int64_t n_pixels, const ftb_render_params* p, const void* out)
{
    if (!sc || !p || n_pixels < 0 || (n_pixels > 0 && (!rays || !out))) return fail(FTB_ERR_BAD_ARG, "null argument or negative pixel count");
    if (p->spp < 1) return fail(FTB_ERR_BAD_ARG, "spp < 1");
    if (n_pixels > 0x7fffff00LL || n_pixels > (int64_t)FTB_TILE_PIXELS * 0x7fffff00LL / 2 / p->spp) return fail(FTB_ERR_BAD_ARG, "too many samples");
    if (p->precision != FTB_PRECISION_FP32 && p->precision != FTB_PRECISION_FP64_VERIFY) return fail(FTB_ERR_BAD_ARG, "bad precision");
    if (p->out_format < FTB_OUT_RGB_F64 || p->out_format > FTB_OUT_RGBA8) return fail(FTB_ERR_BAD_ARG, "bad output format");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { (void)cudaGetLastError(); return fail(FTB_ERR_NO_DEVICE, "no CUDA device: functracer_b200 has no CPU path"); }
    return FTB_OK;
}

// Queues one batch on `s` (n_pixels > 0, arguments checked): the passes of samples_kernel with the variant the scene's frames run
// (ftb_shade_rays' choice), then the conversion into pd->out.  The flat pixel buffer is the tile buffer of a 16-pixel-wide frame
// of ceil(n / 16) rows (pixel i is (i % 16, i / 16) there), so assemble_kernel writes the pixels in order in out_format; pd->out
// holds the first n_pixels of them when the queued work is done.
int samplesLaunch(ftb_scene* sc, PerDevice* pd, const double* rays, const uint64_t* keys, int64_t n_pixels, const ftb_render_params* p,
                  const ftb_debug_out* dbg, ftb_stats* stats, cudaStream_t s)
{
    const int rows = (int)((n_pixels + FTB_TILE_W - 1) / FTB_TILE_W);
    CK(pd->tiles.reserve((size_t)rows * FTB_TILE_W * 3 * realSize(p->precision)));
    CK(pd->out.reserve((size_t)rows * FTB_TILE_W * pixelBytes(p->out_format)));
    FrameGeom fg;
    std::memset(&fg, 0, sizeof(fg));
    fg.width = FTB_TILE_W; fg.height = rows; fg.tiles_x = 1; fg.shard_count = 1;
    return byPrecision(p->precision, [&](auto r) -> int {
        Launch<decltype(r)> fr;
        int e = fr.begin(sc, pd, p, sc->L.features, stats && p->collect_stats, pd->tiles.p, dbg);
        if (e != FTB_OK) return e;
        CK(pd->control.prepare(fr.counting, s));
        auto& F = fr.F;
        F.mode = 2; F.spp = p->spp; F.n_rays = n_pixels; F.n_blocks = (int)((n_pixels + 31) / 32); F.rays = rays; F.shard_count = 1;
        if (stats) CK(cudaEventRecord(pd->ev0, s));
        for (int s_base = 0; s_base < F.spp; s_base += fr.var->unit_cap) {
            fr.setPass(s_base);
            CK(pd->control.resetQueue(s));
            CK(fr.var->samples(*fr.scene, F, reinterpret_cast<const unsigned long long*>(keys), fr.counting, pd->sm_count, s, &fr.launches));
        }
        if (stats) { CK(cudaEventRecord(pd->ev1, s)); stats->kernel_launches += fr.launches + 2; }  // + the control-block memset and the assembly
        const void* bufs[1] = {pd->tiles.p};
        return launchAssemble(p, fg, bufs, pd->out.p, s, 0, rows);
    });
}

// The device entry point: device pointers, queued on `s`; synchronises only to fill stats.
int samplesDevice(ftb_scene* sc, const double* rays, const uint64_t* keys, int64_t n_pixels, const ftb_render_params* p, void* out,
                  const ftb_debug_out* dbg, ftb_stats* stats, cudaStream_t s)
{
    int rc = checkSamples(sc, rays, n_pixels, p, out);
    if (rc != FTB_OK) return rc;
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (n_pixels == 0) return FTB_OK;
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    if ((rc = samplesLaunch(sc, pd, rays, keys, n_pixels, p, dbg && dbg->prim_id ? dbg : nullptr, stats, s)) != FTB_OK) return rc;
    CK(cudaMemcpyAsync(out, pd->out.p, (size_t)n_pixels * pixelBytes(p->out_format), cudaMemcpyDeviceToDevice, s));
    bool overflow = false;
    if (stats && (rc = finishStats(sc, pd, stats, s, &overflow)) != FTB_OK) return rc;
    return overflow ? overflowError() : FTB_OK;
}

// The host entry point, the pattern of pathsHost: upload the rays and keys, queue the batch, read the control block back, and only
// then download the pixels and the requested debug planes: on an overflow nothing of the caller's is written.  Synchronous.
int samplesHost(ftb_scene* sc, const double* rays, const uint64_t* keys, int64_t n_pixels, const ftb_render_params* p, void* out,
                const ftb_debug_out* dbg, ftb_stats* stats)
{
    const auto t0 = std::chrono::steady_clock::now();
    int rc = checkSamples(sc, rays, n_pixels, p, out);
    if (rc != FTB_OK || n_pixels == 0) return rc != FTB_OK ? rc : samplesDevice(sc, rays, keys, n_pixels, p, out, nullptr, stats, nullptr);
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(sc, &pd)) != FTB_OK) return rc;
    if (stats) std::memset(stats, 0, sizeof(*stats));
    const cudaStream_t s = pd->stream;
    const size_t n = (size_t)n_pixels * (size_t)p->spp;  // rays
    CK(pd->rays.reserve(n * 48));
    CK(cudaMemcpyAsync(pd->rays.p, rays, n * 48, cudaMemcpyHostToDevice, s));
    if (keys) {
        CK(pd->query.reserve(n * 8));
        CK(cudaMemcpyAsync(pd->query.p, keys, n * 8, cudaMemcpyHostToDevice, s));
    }
    ftb_debug_out d = {nullptr, nullptr, nullptr};
    if (dbg && dbg->prim_id) {
        CK(pd->dbg_prim.reserve(n * 4)); d.prim_id = static_cast<int32_t*>(pd->dbg_prim.p);
        if (dbg->sub_id) { CK(pd->dbg_sub.reserve(n * 4)); d.sub_id = static_cast<int32_t*>(pd->dbg_sub.p); }
        if (dbg->t) { CK(pd->dbg_t.reserve(n * 8)); d.t = static_cast<double*>(pd->dbg_t.p); }
    }
    rc = samplesLaunch(sc, pd, static_cast<const double*>(pd->rays.p), keys ? static_cast<const uint64_t*>(pd->query.p) : nullptr, n_pixels, p,
                       d.prim_id ? &d : nullptr, stats, s);
    if (rc != FTB_OK) return rc;
    bool overflow = false;
    if ((rc = finishStats(sc, pd, stats, s, &overflow)) != FTB_OK) return rc;
    if (overflow) return overflowError();
    CK(cudaMemcpyAsync(out, pd->out.p, (size_t)n_pixels * pixelBytes(p->out_format), cudaMemcpyDeviceToHost, s));
    if (d.prim_id) {
        CK(cudaMemcpyAsync(dbg->prim_id, d.prim_id, n * 4, cudaMemcpyDeviceToHost, s));
        if (d.sub_id) CK(cudaMemcpyAsync(dbg->sub_id, d.sub_id, n * 4, cudaMemcpyDeviceToHost, s));
        if (d.t) CK(cudaMemcpyAsync(dbg->t, d.t, n * 8, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    if (stats) stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return FTB_OK;
}

}  // namespace

extern "C" {

int ftb_abi_version(void) { return FTB_ABI_VERSION; }

int ftb_device_count(void) { return (int)b200Devices().size(); }

const char* ftb_last_error(void) { return g_err.c_str(); }

int ftb_scene_create(const ftb_scene_desc* desc, ftb_scene** out)
{
    if (!desc || !out) return fail(FTB_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    std::unique_ptr<ftb_scene> sc(new ftb_scene);
    std::string err;
    const auto tc0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        static const bool verbose = std::getenv("FTB_VERBOSE") != nullptr;
        if (verbose) std::fprintf(stderr, "functracer_b200: scene_create %-14s at %8.2f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tc0).count());
    };
    int rc = ftb::lower_scene(*desc, sc->L, err, false);  // the mesh index is built below, on the device
    lap("lowered");
    if (rc != FTB_OK) return fail(rc, err);
    if (sc->L.max_csg_lists > ftb::kMaxLists) return fail(FTB_ERR_UNSUPPORTED, "CSG nesting needs more than 12 pending hit lists");
    if (sc->L.leaves.size() >= (1u << 22)) return fail(FTB_ERR_UNSUPPORTED, "more than 4M leaves");
    sc->triangles.assign(desc->triangles, desc->triangles + 9 * (size_t)desc->n_triangles);
    sc->lights.assign(desc->lights, desc->lights + desc->n_lights);
    for (int i = 0; i < desc->n_images; ++i) {
        ftb_scene::Img im;
        im.w = desc->images[i].width; im.h = desc->images[i].height;
        if (desc->images[i].rgb24 && im.w > 0 && im.h > 0) im.rgb.assign(desc->images[i].rgb24, desc->images[i].rgb24 + 3 * (size_t)im.w * im.h);
        else { im.w = im.h = 1; im.rgb.assign(3, 0); }
        sc->images.push_back(std::move(im));
    }
    lap("copied");
    // upload to the current device now, so that create fails loudly without a GPU
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n < 1) { (void)cudaGetLastError(); return fail(FTB_ERR_NO_DEVICE, "no CUDA device: functracer_b200 has no CPU path"); }
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (sc->L.has_mesh && (rc = buildMeshIndex(*desc, *sc)) != FTB_OK) return rc;
    lap("mesh index");
    PerDevice* pd = nullptr;
    rc = getDevice(sc.get(), dev, &pd);
    if (rc != FTB_OK) return rc;
    rc = uploadScene<float>(*sc, pd->f32);
    if (rc != FTB_OK) return rc;
    lap("uploaded");
    *out = sc.release();
    return FTB_OK;
}

void ftb_scene_destroy(ftb_scene* sc)
{
    if (!sc) return;
    DeviceRestore restore;
    delete sc;  // ~PerDevice synchronises and releases every device's buffers, streams and events
}

int ftb_scene_build_info(const ftb_scene* scene, int32_t* bvh_on_device, double* bvh_build_ms, double* bvh_total_ms)
{
    if (!scene) return fail(FTB_ERR_BAD_ARG, "null argument");
    if (bvh_on_device) *bvh_on_device = scene->bvh_on_device ? 1 : 0;
    if (bvh_build_ms) *bvh_build_ms = scene->bvh_stats.build_ms;
    if (bvh_total_ms) *bvh_total_ms = scene->bvh_stats.total_ms;
    return FTB_OK;
}

int64_t ftb_tile_buffer_bytes(const ftb_render_params* params)
{
    FrameGeom g;
    int rc = frameGeom(params, g);
    if (rc != FTB_OK) return rc;
    return (int64_t)g.n_local_tiles * FTB_TILE_PIXELS * 3 * (int64_t)realSize(params->precision);
}

int ftb_render_tiles_device(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params, void* d_tiles,
                            const ftb_debug_out* d_dbg, ftb_stats* stats, void* stream)
{
    if (!params) return fail(FTB_ERR_BAD_ARG, "null argument");
    return ftb_render_window_tiles_device(scene, camera, params, 0, 0, params->width, params->height, d_tiles, d_dbg, stats, stream);
}

int ftb_render_window_tiles_device(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params, int32_t x0, int32_t y0, int32_t x1,
                                   int32_t y1, void* d_tiles, const ftb_debug_out* d_dbg, ftb_stats* stats, void* stream)
{
    if (!scene || !camera || !params || !d_tiles) return fail(FTB_ERR_BAD_ARG, "null argument");
    FrameGeom g;
    const Window win = {x0, y0, x1, y1};
    int rc = frameGeom(params, g, &win);
    if (rc != FTB_OK) return rc;
    PerDevice* pd = nullptr;
    if ((rc = currentDevice(scene, &pd)) != FTB_OK) return rc;
    if (stats) std::memset(stats, 0, sizeof(*stats));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    rc = byPrecision(params->precision, [&](auto r) {  // band band_index of band_count (without bands: band 0 of 1, all tiles)
        Launch<decltype(r)> fr;
        int e = fr.prepareFrame(scene, pd, camera, params, g, d_tiles, d_dbg, stats, s, g.band_count);
        if (e == FTB_OK) e = fr.launchChunk(g.band_index, s);
        return e == FTB_OK ? fr.finishFrame(stats, s) : e;
    });
    if (rc != FTB_OK) return rc;
    bool overflow = false;
    if (stats && (rc = finishStats(scene, pd, stats, s, &overflow)) != FTB_OK) return rc;  // the only synchronising path of this entry point
    return overflow ? overflowError() : FTB_OK;
}

int ftb_assemble_device(const ftb_render_params* params, const void* const* d_tile_buffers, void* d_out, void* stream)
{
    return ftb_assemble_rows_device(params, d_tile_buffers, d_out, 0, params ? params->height : 0, stream);
}

int ftb_band_rows(const ftb_render_params* params, int band_index, int band_count, int* y0, int* y1)
{
    if (!params || !y0 || !y1) return fail(FTB_ERR_BAD_ARG, "null argument");
    FrameGeom g;
    int rc = frameGeom(params, g);
    if (rc != FTB_OK) return rc;
    if (band_count < 1 || band_count > 64 || band_index < 0 || band_index >= band_count) return fail(FTB_ERR_BAD_ARG, "bad band");
    if (g.corner && band_count > 1) return fail(FTB_ERR_UNSUPPORTED, "corner sampling blends across tile rows: render it as one band");
    *y0 = bandPixelRow(band_index, band_count, g.tiles_y, params->height);
    *y1 = bandPixelRow(band_index + 1, band_count, g.tiles_y, params->height);
    return FTB_OK;
}

int ftb_assemble_rows_device(const ftb_render_params* params, const void* const* d_tile_buffers, void* d_out, int y0, int y1, void* stream)
{
    if (!params || !d_tile_buffers || !d_out) return fail(FTB_ERR_BAD_ARG, "null argument");
    FrameGeom g;
    int rc = frameGeom(params, g);
    if (rc != FTB_OK) return rc;
    if (y0 < 0 || y1 > params->height || y0 > y1) return fail(FTB_ERR_BAD_ARG, "bad row range");
    for (int i = 0; i < g.shard_count; ++i)
        if (!d_tile_buffers[i]) return fail(FTB_ERR_BAD_ARG, "null tile buffer");
    return launchAssemble(params, g, d_tile_buffers, d_out, static_cast<cudaStream_t>(stream), y0, y1);
}

int ftb_host_copy_begin(ftb_scene* scene, const void* d_src, void* host_dst, int64_t bytes, void* stream)
{
    if (!scene || bytes < 0 || (bytes > 0 && (!d_src || !host_dst))) return fail(FTB_ERR_BAD_ARG, "null argument");
    PerDevice* pd = nullptr;
    int rc = currentDevice(scene, &pd);
    if (rc != FTB_OK) return rc;
    CK(pd->copier.begin(d_src, host_dst, (size_t)bytes, static_cast<cudaStream_t>(stream)));
    return FTB_OK;
}

int ftb_host_copy_finish(ftb_scene* scene)
{
    if (!scene) return fail(FTB_ERR_BAD_ARG, "null argument");
    PerDevice* pd = nullptr;
    int rc = currentDevice(scene, &pd);
    if (rc != FTB_OK) return rc;
    CK(pd->copier.finish());
    return FTB_OK;
}

int ftb_check_overflow(ftb_scene* scene, void* stream)
{
    if (!scene) return fail(FTB_ERR_BAD_ARG, "null argument");
    PerDevice* pd = nullptr;
    int rc = currentDevice(scene, &pd);
    if (rc != FTB_OK) return rc;
    if (!pd->control.used()) { CK(cudaStreamSynchronize(static_cast<cudaStream_t>(stream))); return FTB_OK; }  // nothing rendered yet
    bool overflow = false;
    if ((rc = finishStats(scene, pd, nullptr, static_cast<cudaStream_t>(stream), &overflow)) != FTB_OK) return rc;
    return overflow ? overflowError() : FTB_OK;
}

int ftb_render(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params, void* out, const ftb_debug_out* dbg, ftb_stats* stats)
{
    if (!params) return fail(FTB_ERR_BAD_ARG, "null argument");
    return ftb_render_window(scene, camera, params, 0, 0, params->width, params->height, out, dbg, stats);
}

int ftb_render_window(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params, int32_t x0, int32_t y0, int32_t x1, int32_t y1,
                      void* out, const ftb_debug_out* dbg, ftb_stats* stats)
{
    const auto t0 = std::chrono::steady_clock::now();
    if (!scene || !camera || !params || !out) return fail(FTB_ERR_BAD_ARG, "null argument");
    FrameGeom g;  // the window's geometry
    ftb_render_params p = *params;
    p.band_index = 0; p.band_count = 0;  // banding is this call's own business
    const Window win = {x0, y0, x1, y1};
    int rc = frameGeom(&p, g, &win);
    if (rc != FTB_OK) return rc;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { (void)cudaGetLastError(); return fail(FTB_ERR_NO_DEVICE, "no CUDA device: functracer_b200 has no CPU path"); }
    if (stats) std::memset(stats, 0, sizeof(*stats));
    DeviceRestore restore;
    const int n_gpus = p.n_gpus > 1 ? p.n_gpus : 1;
    std::vector<int> devs;
    if (n_gpus > 1) {
        devs = b200Devices();
        if (n_gpus > (int)devs.size()) return fail(FTB_ERR_NO_DEVICE, "n_gpus exceeds the visible sm_100 devices (ftb_device_count)");
        devs.resize((size_t)n_gpus);
    } else devs.push_back(restore.dev);
    if (n_gpus > 1 && p.shard_count > 1) return fail(FTB_ERR_BAD_ARG, "n_gpus > 1 cannot be combined with an external shard");
    if (n_gpus > 1 && dbg) return fail(FTB_ERR_UNSUPPORTED, "debug planes need n_gpus <= 1");
    if (g.shard_count > 1 && n_gpus == 1) {
        // a single external shard cannot be assembled into a frame: the caller wants the device entry point
        return fail(FTB_ERR_BAD_ARG, "ftb_render / ftb_render_window assemble all shards; use ftb_render_(window_)tiles_device for one shard");
    }
    const size_t rs = realSize(p.precision);
    const size_t frameBytes = outBytes(p.out_format, g);
    const size_t rowBytes = frameBytes / (size_t)g.height;
    // The frame is rendered in bands of tile rows, on every device; a finished band is assembled and sent to the host while
    // the next bands render, so only the last, smallest band's copy is exposed.  Four bands also for small downloads: a 1080p
    // RGBA8 frame (8 MB) measured 1.44 ms with four bands against 1.71 ms in one piece (hollow-sphere, 1.17 ms device-resident).
    const bool bandable = !dbg && !stats && !g.corner && (long long)g.width * g.height >= 262144 && g.tiles_y >= 8;
    const int kBands = bandable ? 4 : 1;
    const int primary = devs[0];

    std::vector<Shard> sh((size_t)n_gpus);
    // ---- render: one shard per device, every band of every device queued before anything is waited on ----------------
    for (int k = 0; k < n_gpus; ++k) {
        if ((rc = setUpShard(scene, p, win, g, dbg, devs, kBands, sh, k)) != FTB_OK) return rc;
        const Shard& S = sh[(size_t)k];
        rc = byPrecision(p.precision, [&](auto r) -> int {
            Launch<decltype(r)> fr;
            int e = fr.prepareFrame(scene, S.pd, camera, &S.ps, S.g, S.target, S.dbg.prim_id ? &S.dbg : nullptr, stats, S.pd->stream, kBands);
            if (e != FTB_OK) return e;
            for (int c = 0; c < kBands; ++c) {
                if ((e = fr.launchChunk(c, S.pd->stream)) != FTB_OK) return e;
                if (k > 0 && !S.direct) {  // the band's tiles are a contiguous run of local tiles (tile rows grow with the local index)
                    const size_t l0 = (size_t)S.pd->chunk_first[(size_t)c], l1 = (size_t)S.pd->chunk_first[(size_t)c + 1], off = l0 * FTB_TILE_PIXELS * 3 * rs, n = (l1 - l0) * FTB_TILE_PIXELS * 3 * rs;
                    if (n) CK(cudaMemcpyPeerAsync(static_cast<char*>(S.gather) + off, primary, static_cast<const char*>(S.pd->tiles.p) + off, S.pd->device, n, S.pd->stream));
                    if (stats) stats->kernel_launches += 1;
                }
                CK(cudaEventRecord(S.pd->band_events[(size_t)c], S.pd->stream));
            }
            return fr.finishFrame(stats, S.pd->stream);
        });
        if (rc != FTB_OK) return rc;
    }
    // ---- assemble + download on the primary device, band by band, behind the rendering ------------------------------------
    CK(cudaSetDevice(primary));
    PerDevice* p0 = sh[0].pd;
    CK(p0->out.reserve(frameBytes));
    std::vector<const void*> bufs;
    for (const Shard& S : sh) bufs.push_back(S.gather);
    for (int c = 0; c < kBands; ++c) {
        const int r0 = bandPixelRow(c, kBands, g.tiles_y, g.height), r1 = bandPixelRow(c + 1, kBands, g.tiles_y, g.height);
        for (int k = 0; k < n_gpus; ++k) CK(cudaStreamWaitEvent(p0->copy_stream, sh[(size_t)k].pd->band_events[(size_t)c], 0));
        if (r1 <= r0) continue;
        if ((rc = launchAssemble(&sh[0].ps, sh[0].g, bufs.data(), p0->out.p, p0->copy_stream, r0, r1)) != FTB_OK) return rc;
        if (stats) stats->kernel_launches += 1;
        CK(p0->copier.begin(static_cast<const char*>(p0->out.p) + (size_t)r0 * rowBytes, static_cast<char*>(out) + (size_t)r0 * rowBytes, (size_t)(r1 - r0) * rowBytes, p0->copy_stream));
    }
    CK(p0->copier.finish());
    CK(cudaStreamSynchronize(p0->copy_stream));
    bool overflow = false;
    for (const Shard& S : sh) {
        CK(cudaSetDevice(S.pd->device));
        if ((rc = finishStats(scene, S.pd, stats, S.pd->stream, &overflow)) != FTB_OK) return rc;
    }
    CK(cudaSetDevice(primary));
    if (dbg && dbg->prim_id) {
        CK(cudaMemcpyAsync(dbg->prim_id, p0->dbg_prim.p, (size_t)g.n_samples * 4, cudaMemcpyDeviceToHost, p0->stream));
        if (dbg->sub_id) CK(cudaMemcpyAsync(dbg->sub_id, p0->dbg_sub.p, (size_t)g.n_samples * 4, cudaMemcpyDeviceToHost, p0->stream));
        if (dbg->t) CK(cudaMemcpyAsync(dbg->t, p0->dbg_t.p, (size_t)g.n_samples * 8, cudaMemcpyDeviceToHost, p0->stream));
    }
    CK(cudaStreamSynchronize(p0->stream));
    if (stats) stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return overflow ? overflowError() : FTB_OK;
}

int ftb_shade_rays(ftb_scene* scene, const double* rays_od, int64_t n, const ftb_render_params* params, double* out_rgb,
                   const ftb_debug_out* dbg, ftb_stats* stats)
{
    const auto t0 = std::chrono::steady_clock::now();
    if (!scene || !params || (n > 0 && (!rays_od || !out_rgb)) || n < 0) return fail(FTB_ERR_BAD_ARG, "null argument");
    if (params->precision != FTB_PRECISION_FP32 && params->precision != FTB_PRECISION_FP64_VERIFY) return fail(FTB_ERR_BAD_ARG, "bad precision");
    if (n > (int64_t)FTB_TILE_PIXELS * 0x7fffff00LL / 2) return fail(FTB_ERR_BAD_ARG, "too many rays");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) { (void)cudaGetLastError(); return fail(FTB_ERR_NO_DEVICE, "no CUDA device: functracer_b200 has no CPU path"); }
    if (stats) std::memset(stats, 0, sizeof(*stats));
    if (n == 0) return FTB_OK;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    PerDevice* pd = nullptr;
    int rc = getDevice(scene, dev, &pd);
    if (rc != FTB_OK) return rc;
    cudaStream_t s = pd->stream;
    CK(pd->rays.reserve((size_t)n * 48));
    CK(cudaMemcpyAsync(pd->rays.p, rays_od, (size_t)n * 48, cudaMemcpyHostToDevice, s));
    CK(pd->tiles.reserve((size_t)n * 3 * realSize(params->precision)));
    CK(pd->out.reserve((size_t)n * 24));
    CK(pd->control.resetAll(s));
    ftb_debug_out ddbg = {nullptr, nullptr, nullptr};
    if (dbg && dbg->prim_id) {
        CK(pd->dbg_prim.reserve((size_t)n * 4)); ddbg.prim_id = static_cast<int32_t*>(pd->dbg_prim.p);
        if (dbg->sub_id) { CK(pd->dbg_sub.reserve((size_t)n * 4)); ddbg.sub_id = static_cast<int32_t*>(pd->dbg_sub.p); }
        if (dbg->t) { CK(pd->dbg_t.reserve((size_t)n * 8)); ddbg.t = static_cast<double*>(pd->dbg_t.p); }
    }
    rc = byPrecision(params->precision, [&](auto r) -> int {
        typedef decltype(r) R;
        Launch<R> fr;
        int e = fr.begin(scene, pd, params, scene->L.features, stats && params->collect_stats, pd->tiles.p, &ddbg);
        if (e != FTB_OK) return e;
        DevFrame<R>& F = fr.F;
        F.mode = 1; F.spp = 1; F.s_base = 0; F.s_count = 1; F.run = 1; F.rpp_magic = 0;
        F.n_blocks = (int)((n + 31) / 32); F.n_rays = n; F.rays = static_cast<const double*>(pd->rays.p);
        F.n_local_tiles = (int)((n + FTB_TILE_PIXELS - 1) / FTB_TILE_PIXELS); F.shard_count = 1;
        CK(cudaEventRecord(pd->ev0, s));
        CK(fr.launchKernel(s));
        CK(cudaEventRecord(pd->ev1, s));
        const long long m = 3 * (long long)n;
        widen_kernel<R><<<(int)std::min<long long>((m + 255) / 256, 148 * 16), 256, 0, s>>>(static_cast<const R*>(pd->tiles.p), static_cast<double*>(pd->out.p), m);
        CK(cudaGetLastError());
        if (stats) stats->kernel_launches = fr.launches + 2;
        return FTB_OK;
    });
    if (rc != FTB_OK) return rc;
    CK(cudaMemcpyAsync(out_rgb, pd->out.p, (size_t)n * 24, cudaMemcpyDeviceToHost, s));
    if (ddbg.prim_id) {
        CK(cudaMemcpyAsync(dbg->prim_id, ddbg.prim_id, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        if (ddbg.sub_id) CK(cudaMemcpyAsync(dbg->sub_id, ddbg.sub_id, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
        if (ddbg.t) CK(cudaMemcpyAsync(dbg->t, ddbg.t, (size_t)n * 8, cudaMemcpyDeviceToHost, s));
    }
    bool overflow = false;
    if ((rc = finishStats(scene, pd, stats, s, &overflow)) != FTB_OK) return rc;
    if (stats) stats->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return overflow ? overflowError() : FTB_OK;
}

int ftb_intersect_rays(ftb_scene* scene, const double* rays_od, int64_t n, const ftb_render_params* params, const ftb_hit_out* out, ftb_stats* stats)
{
    return queryHost(scene, false, rays_od, nullptr, n, params, out, nullptr, stats);
}

int ftb_occluded_rays(ftb_scene* scene, const double* rays_od, const double* max_t, int64_t n, const ftb_render_params* params, int32_t* blocked,
                      ftb_stats* stats)
{
    return queryHost(scene, true, rays_od, max_t, n, params, nullptr, blocked, stats);
}

int ftb_intersect_rays_device(ftb_scene* scene, const double* d_rays_od, int64_t n, const ftb_render_params* params, const ftb_hit_out* d_out,
                              ftb_stats* stats, void* stream)
{
    return queryDevice(scene, false, d_rays_od, nullptr, n, params, d_out, nullptr, stats, static_cast<cudaStream_t>(stream));
}

int ftb_occluded_rays_device(ftb_scene* scene, const double* d_rays_od, const double* d_max_t, int64_t n, const ftb_render_params* params,
                             int32_t* d_blocked, ftb_stats* stats, void* stream)
{
    return queryDevice(scene, true, d_rays_od, d_max_t, n, params, nullptr, d_blocked, stats, static_cast<cudaStream_t>(stream));
}

int ftb_intersect_all_rays(ftb_scene* scene, const double* rays_od, int64_t n, int32_t max_hits, double t_min, double t_max,
                           const ftb_render_params* params, const ftb_hit_out* out, int32_t* counts, ftb_stats* stats)
{
    return crossingsHost(scene, rays_od, n, max_hits, t_min, t_max, params, out, counts, stats);
}

int ftb_intersect_all_rays_device(ftb_scene* scene, const double* d_rays_od, int64_t n, int32_t max_hits, double t_min, double t_max,
                                  const ftb_render_params* params, const ftb_hit_out* d_out, int32_t* d_counts, ftb_stats* stats, void* stream)
{
    return crossingsDevice(scene, d_rays_od, n, max_hits, t_min, t_max, params, d_out, d_counts, stats, static_cast<cudaStream_t>(stream));
}

int ftb_trace_paths(ftb_scene* scene, const double* rays_od, const uint64_t* sample_keys, int64_t n, const ftb_render_params* params,
                    const ftb_path_out* out, ftb_stats* stats)
{
    return pathsHost(scene, rays_od, sample_keys, n, params, out, stats);
}

int ftb_trace_paths_device(ftb_scene* scene, const double* d_rays_od, const uint64_t* d_sample_keys, int64_t n, const ftb_render_params* params,
                           const ftb_path_out* d_out, ftb_stats* stats, void* stream)
{
    return pathsDevice(scene, d_rays_od, d_sample_keys, n, params, d_out, stats, static_cast<cudaStream_t>(stream));
}

int ftb_frame_rays(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params, int32_t x0, int32_t y0, int32_t x1, int32_t y1,
                   double* rays_od, uint64_t* sample_keys)
{
    return frameRaysHost(scene, camera, params, Window{x0, y0, x1, y1}, rays_od, sample_keys);
}

int ftb_frame_rays_device(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params, int32_t x0, int32_t y0, int32_t x1, int32_t y1,
                          double* d_rays_od, uint64_t* d_sample_keys, void* stream)
{
    return frameRaysDevice(scene, camera, params, Window{x0, y0, x1, y1}, d_rays_od, d_sample_keys, static_cast<cudaStream_t>(stream));
}

int ftb_shade_samples(ftb_scene* scene, const double* rays_od, const uint64_t* sample_keys, int64_t n_pixels, const ftb_render_params* params,
                      void* out, const ftb_debug_out* dbg, ftb_stats* stats)
{
    return samplesHost(scene, rays_od, sample_keys, n_pixels, params, out, dbg, stats);
}

int ftb_shade_samples_device(ftb_scene* scene, const double* d_rays_od, const uint64_t* d_sample_keys, int64_t n_pixels, const ftb_render_params* params,
                             void* d_out, const ftb_debug_out* d_dbg, ftb_stats* stats, void* stream)
{
    return samplesDevice(scene, d_rays_od, d_sample_keys, n_pixels, params, d_out, d_dbg, stats, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
