// The path queries' kernel: getColourForRay (Shading.fs:109-147) on caller-supplied rays, with every level (bounce) and every light
// of it written out the moment it is known.  Compiled once per precision by the Makefile, with the flags of that precision's render
// variants ([-DFTB_F64 --fmad=false] as the FP64 verification build).  Only the generic FEAT mask: this query explains results, it
// is not a throughput path, and in FP64 the generic kernel is also the one ftb_shade_rays runs.
#include "render.cuh"

namespace ftb {
namespace {

// The hit planes of level entry e: the fragment's record (query_kernel's layout), all zero for a miss.
template <typename R>
__device__ void writeRecord(const DevPaths& P, size_t e, const Fragment<R>& f, bool hit)
{
    double rec[13];  // p, normal, colour, roughness, reflectance, shineyness, apply_lighting
#pragma unroll
    for (int k = 0; k < 13; ++k) rec[k] = 0.0;
    if (hit) {
        rec[0] = f.p.x; rec[1] = f.p.y; rec[2] = f.p.z;
        rec[3] = f.n.x; rec[4] = f.n.y; rec[5] = f.n.z;
        rec[6] = f.colour.x; rec[7] = f.colour.y; rec[8] = f.colour.z;
        rec[9] = f.roughness; rec[10] = f.reflectance; rec[11] = f.shineyness; rec[12] = f.applyLighting ? 1.0 : 0.0;
    }
    if (P.p) { P.p[3 * e] = rec[0]; P.p[3 * e + 1] = rec[1]; P.p[3 * e + 2] = rec[2]; }
    if (P.normal) { P.normal[3 * e] = rec[3]; P.normal[3 * e + 1] = rec[4]; P.normal[3 * e + 2] = rec[5]; }
    if (P.hit_colour) { P.hit_colour[3 * e] = rec[6]; P.hit_colour[3 * e + 1] = rec[7]; P.hit_colour[3 * e + 2] = rec[8]; }
    if (P.surface) { P.surface[4 * e] = rec[9]; P.surface[4 * e + 1] = rec[10]; P.surface[4 * e + 2] = rec[11]; P.surface[4 * e + 3] = rec[12]; }
}

// Light l of level entry e.
__device__ void writeLight(const DevPaths& P, size_t e, int L, int l, double intensity, double dx, double dy, double dz, double cx, double cy, double cz)
{
    const size_t j = e * (size_t)L + (size_t)l;
    if (P.intensity) P.intensity[j] = intensity;
    if (P.light_dir) { P.light_dir[3 * j] = dx; P.light_dir[3 * j + 1] = dy; P.light_dir[3 * j + 2] = dz; }
    if (P.light_colour) { P.light_colour[3 * j] = cx; P.light_colour[3 * j + 1] = cy; P.light_colour[3 * j + 2] = cz; }
}

// Level entry e is a miss: t = -1, prim = -1, sub = 0, every other hit plane and every light plane 0.  The ray and the weight
// are the caller's to write.
template <typename R>
__device__ void writeMiss(const DevPaths& P, size_t e, int L, const Fragment<R>& f)
{
    if (P.t) P.t[e] = -1.0;
    if (P.prim) P.prim[e] = -1;
    if (P.sub) P.sub[e] = 0;
    if (P.record) writeRecord<R>(P, e, f, false);
    for (int l = 0; l < L; ++l) writeLight(P, e, L, l, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0);
}

// Ray ri's path ended after nlev levels: its level count and colour, and the unused levels as misses with weight 0.
template <typename R>
__device__ void finishPath(const DevPaths& P, long long ri, int nlev, Vec<R> scol, int L, const Fragment<R>& f)
{
    const int D = P.recursion_limit + 1;
    if (P.levels) P.levels[ri] = nlev;
    if (P.colour) { P.colour[3 * ri] = scol.x; P.colour[3 * ri + 1] = scol.y; P.colour[3 * ri + 2] = scol.z; }
    for (int k = nlev; k < D; ++k) {
        const size_t e = (size_t)ri * (size_t)D + (size_t)k;
        if (P.ray_od) for (int j = 0; j < 6; ++j) P.ray_od[6 * e + j] = 0.0;
        if (P.weight) P.weight[e] = 0.0;
        writeMiss<R>(P, e, L, f);
    }
}

}  // namespace

// render_kernel's lane state machine for one sample of mode 1 (explicit rays), without the blend ring and the tile logic: an idle
// lane takes the next ray of the warp's group of 32 (the warp takes groups from the per-device queue counter), and in every
// iteration each lane with work traces one ray, a nearest-hit ray or one shadow ray.  All lanes call traceScene together with the
// `tracing` ballot, so that the warp-packet walk of large meshes stays correct.  The colour is summed exactly as render_kernel sums
// it (local over the lights in order, then scol += W * local, W *= L * reflectance), with the same device functions, so in FP64 it
// is bit-identical to ftb_shade_rays'.  Not used here: the common-origin bound table (a frame's shared-memory shortcut whose use
// depends on which rays share a warp; it changes which bound tests run, never a result) and the lit-tile shortcut of primary
// fragments (frames only).
template <typename R, unsigned FEAT, bool STATS>
__global__ void __launch_bounds__(kBlockThreads, MinBlocks<FEAT>::value) path_kernel(const __grid_constant__ DevScene<R> S, const __grid_constant__ DevPaths P)
{
    typedef typename V4<R>::type R4;
    constexpr int WARPS = kBlockThreads / 32;
    __shared__ int mesh_stack[MeshWalks<FEAT>::kPacket ? WARPS : 1][MeshWalks<FEAT>::kPacket ? kBspStack : 1];  // packetMesh: one walk per warp
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int D = P.recursion_limit + 1, L = S.n_lights;
    Counters<STATS> cn;
    bool overflow = false;

    long long g_base = 0;  // warp-uniform: the group of rays being dealt
    int g_n = 0, g_pos = 0;
    bool exhausted = false;

    // per-lane path state
    long long ri = 0;           // the ray's index
    unsigned long long key = 0;  // its RNG sample key
    int phase = PH_IDLE, limit = 0;  // limit: bounces left; the level (and the RNG depth) is recursion_limit - limit
    R weight = R(1), tmax = R(0);
    Ray<R> ray;    // the ray to trace next: path ray (un-offset) in PH_NEAREST, shadow ray in PH_SHADOW
    Vec<R> pathD;  // direction of the current path ray
    ray.o = mk<R>(R(0), R(0), R(0)); ray.d = ray.o; pathD = ray.o;
    Fragment<R> f;
    f.p = ray.o; f.n = ray.o; f.colour = ray.o; f.roughness = f.reflectance = f.shineyness = R(0); f.applyLighting = false; f.planarLeaf = -1;
    Vec<R> local = ray.o, scol = ray.o;
    int li = 0, sk = 0, occluded = 0;

    for (;;) {
        // ---- deal the rays of the warp's group to idle lanes (ballot + popc = warp scan) ----------------------------------
        unsigned m = __ballot_sync(full, phase == PH_IDLE);
        while (m && !exhausted) {
            if (g_pos >= g_n) {
                unsigned c = 0;
                if (lane == 0) c = atomicAdd(P.group_counter, 1u);
                c = __shfl_sync(full, c, 0);
                if (c >= (unsigned)P.n_groups) { exhausted = true; break; }
                g_base = (long long)c * 32; g_n = (int)min(32LL, P.n - g_base); g_pos = 0;
            }
            const int rank = __popc(m & lt_mask), avail = g_n - g_pos;
            if (phase == PH_IDLE && rank < avail) { ri = g_base + g_pos + rank; phase = PH_START; }
            g_pos += min(__popc(m), avail);
            m = __ballot_sync(full, phase == PH_IDLE);
        }
        if (phase == PH_START) {
            const double* q = P.rays + 6 * (size_t)ri;
            ray.o = mk<R>((R)__ldg(q), (R)__ldg(q + 1), (R)__ldg(q + 2));
            ray.d = mk<R>((R)__ldg(q + 3), (R)__ldg(q + 4), (R)__ldg(q + 5));
            key = P.sample_keys ? __ldg(P.sample_keys + ri) : (unsigned long long)ri;
            phase = PH_NEAREST; limit = P.recursion_limit; weight = R(1);
            scol = mk<R>(R(0), R(0), R(0));
            cn.add(ST_PRIMARY);
        }
        if (!__any_sync(full, phase != PH_IDLE)) break;
        // phase alignment as in render_kernel: shadow-phase lanes go first, nearest-phase lanes hold for that iteration
        const bool hold = __any_sync(full, phase == PH_SHADOW) && phase == PH_NEAREST;
        unsigned tracing = full;
        if constexpr (MeshWalks<FEAT>::kPacket) tracing = __ballot_sync(full, !(phase == PH_IDLE || hold));
        if (phase == PH_IDLE || hold) continue;

        // ---- trace this lane's current ray --------------------------------------------------------------------------------
        Ray<R> tr = ray;
        if (phase == PH_NEAREST) {  // slightOffset (Shading.fs:129): d is NOT normalised
            tr.o = ray.o + R(0.0001) * ray.d;
            pathD = ray.d;
        } else cn.add(ST_SHADOW);
        int skipLeaf = -1;  // FP32: render_kernel's planar self-skip, for bounce and shadow rays alike
        if constexpr (sizeof(R) == 4 && (FEAT & FT_PLANAR) != 0) {
            if (f.planarLeaf >= 0 && (phase == PH_NEAREST ? limit < P.recursion_limit : dot(ray.d, f.n) >= R(0))) skipLeaf = f.planarLeaf;
        }
        const HitInfo<R> h = traceScene<R, FEAT, STATS>(S, tr, phase == PH_NEAREST ? inf_<R>() : tmax, phase == PH_SHADOW, skipLeaf, ~0u, (const R4*)nullptr, R(0),
                                                        overflow, cn, tracing, &mesh_stack[MeshWalks<FEAT>::kPacket ? wib : 0][0]);

        // ---- consume the result ---------------------------------------------------------------------------------------------
        const int level = P.recursion_limit - limit;
        const size_t e = (size_t)ri * (size_t)D + (size_t)level;
        bool got = false;  // an intensity for light `li` is ready
        R intensity = R(0);
        if (phase == PH_NEAREST) {
            if (P.ray_od) {
                P.ray_od[6 * e] = ray.o.x; P.ray_od[6 * e + 1] = ray.o.y; P.ray_od[6 * e + 2] = ray.o.z;
                P.ray_od[6 * e + 3] = ray.d.x; P.ray_od[6 * e + 4] = ray.d.y; P.ray_od[6 * e + 5] = ray.d.z;
            }
            if (P.weight) P.weight[e] = weight;
            if (h.leaf < 0) {  // miss: empty sum (Shading.fs:137-139)
                writeMiss<R>(P, e, L, f);
                finishPath<R>(P, ri, level + 1, scol, L, f);
                phase = PH_IDLE;
                continue;
            }
            {  // the debug planes' expression (render_kernel), written out again as query_kernel does
                const int4 meta = __ldg(S.leaf_meta + h.leaf);
                const int kind = meta.x & 0xff;
                if (P.prim) P.prim[e] = meta.z;
                if (P.sub) P.sub[e] = (kind == LEAF_CUBE || kind == LEAF_MESH || kind == LEAF_SOLIDCYL) ? h.sub : ((kind == LEAF_TRIANGLE) ? 0 : meta.w);
                if (P.t) P.t[e] = (double)h.t;
            }
            f = finalise<R, FEAT>(S, tr, h);
            if (P.record) writeRecord<R>(P, e, f, true);
            if (L <= 0) {  // nothing to shade, nothing to reflect: the colour is the empty sum
                finishPath<R>(P, ri, level + 1, scol, L, f);
                phase = PH_IDLE;
                continue;
            }
            cn.add(ST_SHADED);
            local = mk<R>(R(0), R(0), R(0));
            li = 0;
            ray.o = f.p + R(0.0001) * f.n;  // shadowRayOrigin (Shading.fs:111), the same for every light
        } else {
            const bool blocked = h.leaf >= 0;
            const int2 lk = __ldg(S.light_i + li);
            if (lk.x == FTB_LIGHT_SOFT_DIRECTIONAL) {  // softShadowLightIntensity (Shading.fs:24-31)
                if constexpr ((FEAT & FT_RNG) != 0) {
                    occluded += blocked ? 1 : 0;
                    ++sk;
                    if (sk < lk.y) {
                        const R4 la = ldg4<R>(S.light_a + li);
                        ray.d = jitterVector<R>(P.seed, key, (unsigned)level, (unsigned)li, (unsigned)sk, la.w, -mk<R>(la.x, la.y, la.z));
                        continue;  // next sample of the same light
                    }
                    intensity = (R)(lk.y - occluded) / (R)lk.y;
                }
            } else if (lk.x == FTB_LIGHT_POINT) {
                const R4 lb = ldg4<R>(S.light_b + li);
                intensity = blocked ? R(0) : R(1) / (lb.x + tmax * (lb.y + tmax * lb.z));  // Light.attenuate (Light.fs:16-17)
            } else {
                intensity = blocked ? R(0) : R(1);
            }
            got = true;
        }
        // advance through the lights until one needs a shadow ray or the level is complete
        for (;;) {
            if (got) {
                const Vec<R> c = shadeLight<R, FEAT>(S, f, pathD, li, intensity);
                const int2 lk = __ldg(S.light_i + li);
                const R4 la = ldg4<R>(S.light_a + li);
                const Vec<R> lv = mk<R>(la.x, la.y, la.z);
                const Vec<R> ldir = (lk.x == FTB_LIGHT_POINT) ? normalise(f.p - lv) : lv;  // lightDirection (Shading.fs:44-48)
                writeLight(P, e, L, li, intensity, ldir.x, ldir.y, ldir.z, c.x, c.y, c.z);
                local = local + c;
                ++li;
                got = false;
            }
            if (li >= L) break;
            // fragments whose colour ignores the light's intensity need no shadow ray: unlit surfaces
            // (shadeIfRequired) and Oren-Nayar surfaces without a specular term (Shading.fs:50-63, 85-86)
            bool needShadow = f.applyLighting;
            if constexpr ((FEAT & FT_ROUGH) != 0) needShadow = needShadow && !(f.roughness != R(0) && !(f.shineyness > R(0)));
            if (!needShadow) { intensity = R(1); got = true; continue; }
            const int2 lk = __ldg(S.light_i + li);
            const R4 la = ldg4<R>(S.light_a + li);
            const Vec<R> lv = mk<R>(la.x, la.y, la.z);
            if (lk.x == FTB_LIGHT_POINT) {  // shadowLightIntensity (Shading.fs:33-42)
                const Vec<R> dvec = lv - ray.o;
                tmax = length(dvec);
                ray.d = normalise(dvec);
            } else if (lk.x == FTB_LIGHT_SOFT_DIRECTIONAL) {
                if (lk.y <= 0) { intensity = (R)(lk.y - 0) / (R)lk.y; got = true; continue; }  // 0/0: NaN like the reference
                if constexpr ((FEAT & FT_RNG) != 0) {
                    sk = 0; occluded = 0;
                    tmax = realmax_<R>();
                    ray.d = jitterVector<R>(P.seed, key, (unsigned)level, (unsigned)li, 0u, la.w, -lv);
                }
            } else {
                tmax = realmax_<R>();
                ray.d = -lv;
            }
            phase = PH_SHADOW;
            break;
        }
        if (li < L) continue;  // a shadow ray is pending
        // ---- level complete (getColourForRay's Seq.sumBy, Shading.fs:139) -------------------------------------------------
        scol = scol + weight * local;
        // reflectionShader (Shading.fs:89-98) sits inside the per-light sum: L identical re-traces => weight L * reflectance
        if (f.applyLighting && f.reflectance > R(0) && limit > 0) {
            weight = weight * ((R)L * f.reflectance);
            ray.o = f.p; ray.d = reflect(f.n, pathD);
            --limit;
            phase = PH_NEAREST;
            cn.add(ST_REFLECTION);
        } else {
            finishPath<R>(P, ri, level + 1, scol, L, f);
            phase = PH_IDLE;
        }
    }
    if (overflow) atomicExch(P.overflow, 1u);
    if constexpr (STATS) {
        for (int k = 0; k < ST_COUNT; ++k) {
            unsigned long long v = cn.get(k);
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(full, v, o);
            if (lane == 0 && v) atomicAdd(P.stats + k, v);
        }
    }
}

template <typename R>
cudaError_t launch_paths_impl(const DevScene<R>& s, const DevPaths& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    int per_sm = 0;
    cudaError_t e = stats ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, path_kernel<R, (unsigned)FT_ALL, true>, kBlockThreads, 0)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, path_kernel<R, (unsigned)FT_ALL, false>, kBlockThreads, 0);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) per_sm = 1;
    // persistent grid: a multiple of the SM count, never more warps than there are groups of rays
    const long long want = (long long)sm_count * per_sm, cap = ((long long)q.n_groups + (kBlockThreads / 32) - 1) / (kBlockThreads / 32);
    int grid = (int)(want < cap ? want : cap);
    if (grid < 1) grid = 1;
    if (stats) path_kernel<R, (unsigned)FT_ALL, true><<<grid, kBlockThreads, 0, stream>>>(s, q);
    else path_kernel<R, (unsigned)FT_ALL, false><<<grid, kBlockThreads, 0, stream>>>(s, q);
    if (launches) ++*launches;
    return cudaGetLastError();
}

#ifdef FTB_F64
cudaError_t paths_f64(const DevScene<double>& s, const DevPaths& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    return launch_paths_impl<double>(s, q, stats, sm_count, stream, launches);
}
#else
cudaError_t paths_f32(const DevScene<float>& s, const DevPaths& q, bool stats, int sm_count, cudaStream_t stream, int* launches)
{
    return launch_paths_impl<float>(s, q, stats, sm_count, stream, launches);
}
#endif
}  // namespace ftb
