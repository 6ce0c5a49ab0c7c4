// MPI over-composite renderer for B200 (sm_100a): kernels + C ABI (include/gmpi_mpi_render.h).
//
// Replaces gmpi/core/mpi.py MPI.forward (:308-436) + homography (:26-153) and their autograd.
// DESIGN.md describes the data layout, each kernel and its roofline.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <mutex>

#include "../../include/gmpi_mpi_render.h"
#include "mpi_common.cuh"
#include "mpi_fwd_staged.cuh"
#include "mpi_bwd_box.cuh"
#include "mpi_light.cuh"

namespace gmpi {

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define GMPI_CUDA_OK(expr)                                                                        \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess)                                                                    \
            return fail(GMPI_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                        __FILE__, __LINE__);                                                      \
    } while (0)

// ------------------------------------------------------------------------------------------
// Forward, direct-gather variant: one thread = one output pixel, a warp = 32 consecutive x.
// Taps are read straight from global memory through L1 (per channel a warp touches one or two
// 128-byte lines per tap row).  Works for every shape; the TMA-staged variant is the fast path.
// ------------------------------------------------------------------------------------------
constexpr int kFwdTileW = 32;
constexpr int kFwdTileH = 8;

// kCut: early ray termination, each pixel stops at the first plane in front of which T < p.stop_transmittance (inference only);
// p.skipped (nullable) accumulates the planes not composited, one atomic per warp.
template <bool kAlignCorners, bool kCut>
__device__ __forceinline__ void fwd_direct_body(const RenderParams p) {     // (by value: by reference, ptxas schedules the
                                                                            // kCut = false instance differently from the kernel it was)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PlaneConst* s_pc = reinterpret_cast<PlaneConst*>(smem_raw);

    const int v = blockIdx.z;
    const int m = __ldg(p.view2mpi + v);
    const int tid = threadIdx.y * kFwdTileW + threadIdx.x;
    float ev[3], zd[3];
    load_eye_z(p, v, ev, zd);
    const float eye0_z = __ldg(p.eye0 + 2);  // mpi.py:70 compares every distance with view 0's eye
    uint32_t flag = 0;
    for (int i = tid; i < p.N; i += kFwdTileW * kFwdTileH) {
        const float* dp = p.dhw + ((size_t)m * p.N + i) * 3;
        s_pc[i] = make_plane_const(dp, ev[2]);
        if (!(__ldg(dp) >= eye0_z)) flag |= GMPI_FLAG_PLANE_BEHIND_EYE;
    }
    __syncthreads();

    const int px = blockIdx.x * kFwdTileW + threadIdx.x;
    const int py = blockIdx.y * kFwdTileH + threadIdx.y;
    unsigned skip = 0;      // kCut: planes this pixel did not composite
    if (px < p.W && py < p.H) {
        const size_t img = (size_t)p.H * p.W;
        const size_t pix = (size_t)py * p.W + px;
        float qx, qy, qz;
        load_ray(p, v, px, py, img, qx, qy, qz);
        const RayConst rc = make_ray_const(qx, qy, qz, ev, zd);

        const int Ht = p.Ht, Wt = p.Wt;
        const float fWt = (float)Wt, fHt = (float)Ht;
        const float hsx = 0.5f * (float)(Wt - 1), hsy = 0.5f * (float)(Ht - 1);
        const size_t tex = (size_t)Ht * Wt;
        const bool check_last = (p.options & GMPI_CHECK_LAST_PLANE) != 0;

        float T = 1.0f, cr = 0.0f, cg = 0.0f, cb = 0.0f, cws = 0.0f;
        const float tau = kCut ? p.stop_transmittance : 0.0f;
#pragma unroll 2
        for (int i = 0; i < p.N; ++i) {
            if (kCut && T < tau) {           // planes i.. add less than tau * max value
                if (check_last) {            // the last-plane check still sees every pixel
                    const TexCoord tl = plane_coord<kAlignCorners>(s_pc[p.N - 1], rc, hsx, hsy, fWt, fHt);
                    if (!(tl.u >= -1.0f && tl.u <= 1.0f && tl.v >= -1.0f && tl.v <= 1.0f)) flag |= GMPI_FLAG_LAST_PLANE_OOB;
                }
                skip = (unsigned)(p.N - i);
                break;
            }
            const PlaneConst pc = s_pc[i];
            const PlaneChans plane = plane_chans(p, m, i, tex);
            if (p.transmittance) p.transmittance[((size_t)v * p.N + i) * img + pix] = T;   // training: T_i for the backward sweep
            const TexCoord tc = plane_coord<kAlignCorners>(pc, rc, hsx, hsy, fWt, fHt);
            if (check_last && i == p.N - 1) {
                if (!(tc.u >= -1.0f && tc.u <= 1.0f && tc.v >= -1.0f && tc.v <= 1.0f)) flag |= GMPI_FLAG_LAST_PLANE_OOB;
            }
            if (coord_hits(tc.ix, tc.iy, fWt, fHt)) {
                const Taps t = make_taps(tc.ix, tc.iy, Ht, Wt);
                const float r = tap4(plane.c[0], t);
                const float g = tap4(plane.c[1], t);
                const float b = tap4(plane.c[2], t);
                const float a = tap4(plane.c[3], t);
                const float w = a * T;                                   // mpi.py:423
                cr = fmaf(w, r, cr);                                     // mpi.py:430
                cg = fmaf(w, g, cg);
                cb = fmaf(w, b, cb);
                cws = fmaf(w, tc.scale, cws);                            // depth_i = scale * (ray.z_dir), :150
                T *= (1.0f - a) + 1e-10f;                                // mpi.py:421
            }
        }
        const float dep = cws * rc.dz;
        if (p.options & GMPI_COLOR_MINUS1_1) {                           // mpi_renderer.py:467
            cr = fmaf(2.0f, cr, -1.0f);
            cg = fmaf(2.0f, cg, -1.0f);
            cb = fmaf(2.0f, cb, -1.0f);
        }
        store_pixel(p, v, img, pix, cr, cg, cb, dep);
    }
    if (kCut && p.skipped) {      // one atomic per warp (a warp is one row of 32 x: all lanes reach this point)
        const unsigned n = __reduce_add_sync(0xffffffffu, skip);
        if (threadIdx.x == 0 && n) atomicAdd(p.skipped, (unsigned long long)n);
    }
    if (flag) atomicOr(p.flags, flag);
}

template <bool kAlignCorners>
__global__ void __launch_bounds__(kFwdTileW* kFwdTileH)
mpi_fwd_direct_kernel(const RenderParams p) {
    fwd_direct_body<kAlignCorners, false>(p);
}
template <bool kAlignCorners>
__global__ void __launch_bounds__(kFwdTileW* kFwdTileH)
mpi_fwd_direct_cut_kernel(const RenderParams p) {
    fwd_direct_body<kAlignCorners, true>(p);
}

// ------------------------------------------------------------------------------------------
// Backward, direct variant.
//   pass A (front to back, alpha only): T_i = prod_{j<i}(1 - a_j + 1e-10), stashed per thread in
//           shared memory ([plane][thread], conflict free).
//   pass B (back to front, all channels): R_{i-1} = a_i q_i + s_i R_i with R_{N-1} = 0,
//           q_i = G.rgb_i + Gd*depth_i, s_i = 1 - a_i + 1e-10, and
//             dL/d rgb_i = G * a_i T_i
//             dL/d a_i   = T_i (q_i - R_i)
//           which equals autograd's  T_i q_i - (sum_{k>i} a_k q_k P_k)/s_i  (cumprod_backward)
//           without the division by s_i (1e-10 when a_i == 1) and without cancellation.
//           The four bilinear weights scatter each value with red.global.add.f32.
// ------------------------------------------------------------------------------------------
template <bool kAlignCorners>
__global__ void __launch_bounds__(128)
mpi_bwd_direct_kernel(const RenderParams p, const int tile_w, const int tile_h) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PlaneConst* s_pc = reinterpret_cast<PlaneConst*>(smem_raw);
    const int nthreads = tile_w * tile_h;
    float* s_T = reinterpret_cast<float*>(smem_raw + sizeof(PlaneConst) * p.N);   // [N][nthreads]

    const int v = blockIdx.z;
    const int m = __ldg(p.view2mpi + v);
    const int tid = threadIdx.y * tile_w + threadIdx.x;
    const float* e = p.eye + 3 * v;
    for (int i = tid; i < p.N; i += nthreads) {
        s_pc[i] = make_plane_const(p.dhw + ((size_t)m * p.N + i) * 3, __ldg(e + 2));
    }
    __syncthreads();

    const int px = blockIdx.x * tile_w + threadIdx.x;
    const int py = blockIdx.y * tile_h + threadIdx.y;
    if (px >= p.W || py >= p.H) return;

    const size_t img = (size_t)p.H * p.W;
    const size_t pix = (size_t)py * p.W + px;
    const float* rd = p.ray_dir + (size_t)v * 3 * img + pix;
    const float ev[3] = {__ldg(e), __ldg(e + 1), __ldg(e + 2)};
    const float zd[3] = {__ldg(p.z_dir + 3 * v), __ldg(p.z_dir + 3 * v + 1), __ldg(p.z_dir + 3 * v + 2)};
    const RayConst rc = make_ray_const(__ldg(rd), __ldg(rd + img), __ldg(rd + 2 * img), ev, zd);

    const int Ht = p.Ht, Wt = p.Wt, N = p.N;
    const float fWt = (float)Wt, fHt = (float)Ht;
    const float hsx = 0.5f * (float)(Wt - 1), hsy = 0.5f * (float)(Ht - 1);
    const size_t tex = (size_t)Ht * Wt;

    float gscale = (p.options & GMPI_COLOR_MINUS1_1) ? 2.0f : 1.0f;
    const float* gc = p.g_color + (size_t)v * 3 * img + pix;
    const float G0 = gscale * __ldg(gc), G1 = gscale * __ldg(gc + img), G2 = gscale * __ldg(gc + 2 * img);
    const float Gd = p.g_depth ? __ldg(p.g_depth + (size_t)v * img + pix) : 0.0f;
    const float Gdz = Gd * rc.dz;   // depth_i = scale_i * dz

    // pass A
    float T = 1.0f;
    for (int i = 0; i < N; ++i) {
        s_T[(size_t)i * nthreads + tid] = T;
        const TexCoord tc = plane_coord<kAlignCorners>(s_pc[i], rc, hsx, hsy, fWt, fHt);
        if (coord_hits(tc.ix, tc.iy, fWt, fHt)) {
            const Taps t = make_taps(tc.ix, tc.iy, Ht, Wt);
            const float a = tap4(plane_chans(p, m, i, tex).c[3], t);
            T *= (1.0f - a) + 1e-10f;
        }
    }
    // pass B
    float R = 0.0f;
    for (int i = N - 1; i >= 0; --i) {
        const TexCoord tc = plane_coord<kAlignCorners>(s_pc[i], rc, hsx, hsy, fWt, fHt);
        if (!coord_hits(tc.ix, tc.iy, fWt, fHt)) continue;
        const Taps t = make_taps(tc.ix, tc.iy, Ht, Wt);
        const PlaneChans plane = plane_chans(p, m, i, tex);
        const float r = tap4(plane.c[0], t);
        const float g = tap4(plane.c[1], t);
        const float b = tap4(plane.c[2], t);
        const float a = tap4(plane.c[3], t);
        const float Ti = s_T[(size_t)i * nthreads + tid];
        const float q = fmaf(G0, r, fmaf(G1, g, fmaf(G2, b, Gdz * tc.scale)));
        const float w = a * Ti;
        const float gv[4] = {G0 * w, G1 * w, G2 * w, Ti * (q - R)};
        R = fmaf(a, q, ((1.0f - a) + 1e-10f) * R);
        const GradChans gp = grad_chans(p, m, i, tex);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float* gch = gp.c[c];
            if (t.w00 != 0.0f) atomicAdd(gch + t.o00, gv[c] * t.w00);
            if (t.w01 != 0.0f) atomicAdd(gch + t.o01, gv[c] * t.w01);
            if (t.w10 != 0.0f) atomicAdd(gch + t.o10, gv[c] * t.w10);
            if (t.w11 != 0.0f) atomicAdd(gch + t.o11, gv[c] * t.w11);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Range check: one streaming pass over rgba.  A float is inside [0,1] iff its bit pattern,
// read as unsigned, is <= 0x3f800000 (or it is -0.0); NaN and negatives have larger patterns.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ bool out_of_unit(float x) {
    const uint32_t b = __float_as_uint(x);
    return b > 0x3f800000u && b != 0x80000000u;
}

__global__ void __launch_bounds__(256)
mpi_check_range_kernel(const float4* __restrict__ rgba4, size_t n_slabs, size_t slab4, uint32_t* flags) {
    // one slab = one (mpi, plane, channel) image of slab4 float4's; channel = slab % 4
    uint32_t flag = 0;
    const size_t total = n_slabs * slab4;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const float4 x = __ldcs(rgba4 + i);
        if (out_of_unit(x.x) || out_of_unit(x.y) || out_of_unit(x.z) || out_of_unit(x.w)) {
            const size_t slab = i / slab4;
            flag |= ((slab & 3) == 3) ? (GMPI_FLAG_ALPHA_RANGE | GMPI_FLAG_RGBA_RANGE) : GMPI_FLAG_RGBA_RANGE;
        }
    }
    flag = __reduce_or_sync(0xffffffffu, flag);
    if (flag && (threadIdx.x & 31) == 0) atomicOr(flags, flag);
}

__global__ void mpi_check_range_scalar_kernel(const float* __restrict__ rgba, size_t n_slabs, size_t slab,
                                              uint32_t* flags) {
    uint32_t flag = 0;
    const size_t total = n_slabs * slab;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        if (out_of_unit(__ldcs(rgba + i))) {
            flag |= (((i / slab) & 3) == 3) ? (GMPI_FLAG_ALPHA_RANGE | GMPI_FLAG_RGBA_RANGE) : GMPI_FLAG_RGBA_RANGE;
        }
    }
    if (flag) atomicOr(flags, flag);
}

// ------------------------------------------------------------------------------------------
// Occupancy map of empty-space skipping (gmpi_mpi_occupancy): one bit per 8x8-texel block of every alpha plane, set iff some
// alpha of the block has !(|alpha| <= threshold) (NaN is occupied); texels outside the texture do not exist.  One warp per
// 64-bit word = 8 texel rows x 512 texels: every load of the warp covers 32 * kVec consecutive texels of one row (kVec = 4:
// float4, rows and strides 16-byte aligned), its ballot has 8 / kVec bits per block; the ballots of the 8 rows are OR-ed, then
// folded into one bit per block.  A streaming read of the alpha planes alone, 4 bytes per texel-plane.
// ------------------------------------------------------------------------------------------
template <int kVec>
__global__ void __launch_bounds__(256)
mpi_occupancy_kernel(const float* __restrict__ alpha, long long mpi_stride, long long plane_stride, int N, int Ht, int Wt, int n_wy,
                     int n_wx, long long n_words, float threshold, uint64_t* __restrict__ occ) {
    constexpr int kLoads = 512 / (32 * kVec), kLanesPerBlock = 8 / kVec, kBlocksPerLoad = 32 / kLanesPerBlock;
    const long long word = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (word >= n_words) return;     // warp-uniform
    const int wx = (int)(word % n_wx);
    const long long t = word / n_wx;
    const int wy = (int)(t % n_wy);
    const long long plane = t / n_wy, m = plane / N, i = plane - m * N;
    const float* base = alpha + m * mpi_stride + i * plane_stride;
    uint32_t bal[kLoads];
#pragma unroll
    for (int k = 0; k < kLoads; ++k) bal[k] = 0u;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int y = 8 * wy + r;
        const float* row = base + (long long)y * Wt;
#pragma unroll
        for (int k = 0; k < kLoads; ++k) {
            const int x = 512 * wx + kVec * (32 * k + lane);
            bool o = false;
            if (y < Ht && x < Wt) {          // (kVec = 4: Wt % 4 == 0, so the whole float4 is inside the row)
                if constexpr (kVec == 4) {
                    const float4 a = __ldcs(reinterpret_cast<const float4*>(row + x));
                    o = !(fabsf(a.x) <= threshold) || !(fabsf(a.y) <= threshold) || !(fabsf(a.z) <= threshold) || !(fabsf(a.w) <= threshold);
                } else {
                    o = !(fabsf(__ldcs(row + x)) <= threshold);
                }
            }
            bal[k] |= __ballot_sync(0xffffffffu, o);
        }
    }
    if (lane != 0) return;
    uint64_t w = 0;
#pragma unroll
    for (int k = 0; k < kLoads; ++k)
#pragma unroll
        for (int q = 0; q < kBlocksPerLoad; ++q)
            if ((bal[k] >> (q * kLanesPerBlock)) & ((1u << kLanesPerBlock) - 1u)) w |= 1ull << (k * kBlocksPerLoad + q);
    occ[word] = w;
}

// ------------------------------------------------------------------------------------------
// Test hook: texel coordinates.
// ------------------------------------------------------------------------------------------
template <bool kAlignCorners>
__global__ void mpi_debug_coords_kernel(const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                                        const float* eye, float* out, int V, int N, int Ht, int Wt, int H, int W) {
    const size_t img = (size_t)H * W;
    const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int v = blockIdx.y;
    if (pix >= img) return;
    const int m = view2mpi[v];
    const float* e = eye + 3 * v;
    const float ev[3] = {e[0], e[1], e[2]};
    const float zd[3] = {0.f, 0.f, 1.f};
    const float* rd = ray_dir + (size_t)v * 3 * img + pix;
    const RayConst rc = make_ray_const(rd[0], rd[img], rd[2 * img], ev, zd);
    const float hsx = 0.5f * (float)(Wt - 1), hsy = 0.5f * (float)(Ht - 1);
    for (int i = 0; i < N; ++i) {
        const PlaneConst pc = make_plane_const(dhw + ((size_t)m * N + i) * 3, ev[2]);
        const TexCoord tc = plane_coord<kAlignCorners>(pc, rc, hsx, hsy, (float)Wt, (float)Ht);
        out[(((size_t)v * N + i) * 2 + 0) * img + pix] = tc.ix;
        out[(((size_t)v * N + i) * 2 + 1) * img + pix] = tc.iy;
    }
}

// Test hook for the packed (f32x2) coordinate path of the staged kernel: pixels 2k, 2k+1 of a row form a pair.
template <bool kAlignCorners>
__global__ void mpi_debug_coords_packed_kernel(const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                                               const float* eye, float* out, int V, int N, int Ht, int Wt, int H, int W) {
    const size_t img = (size_t)H * W;
    const size_t pair = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int v = blockIdx.y;
    if (pair * 2 + 1 >= img) return;
    const int m = view2mpi[v];
    const float* e = eye + 3 * v;
    const float ev[3] = {e[0], e[1], e[2]};
    const float zd[3] = {0.f, 0.f, 1.f};
    RayConst rc[2];
    for (int k = 0; k < 2; ++k) {
        const float* rd = ray_dir + (size_t)v * 3 * img + pair * 2 + k;
        rc[k] = make_ray_const(rd[0], rd[img], rd[2 * img], ev, zd);
    }
    RayPairs rp;
    for (int P = 0; P < 2; ++P) {
        rp.rx2[P] = make_float2(rc[0].rx2, rc[1].rx2); rp.ry2[P] = make_float2(rc[0].ry2, rc[1].ry2);
        rp.nrz[P] = make_float2(-rc[0].rz, -rc[1].rz); rp.yrz[P] = make_float2(rc[0].yrz, rc[1].yrz);
    }
    const float hsx = 0.5f * (float)(Wt - 1), hsy = 0.5f * (float)(Ht - 1);
    for (int i = 0; i < N; ++i) {
        const PlaneConst pc = make_plane_const(dhw + ((size_t)m * N + i) * 3, ev[2]);
        CoordPairs c;
        coords_pairs<kAlignCorners>(pc, rp, splat(rc[0].ex2), splat(rc[0].ey2), splat(hsx), splat(hsy), (float)Wt, (float)Ht, c);
        float* o = out + (((size_t)v * N + i) * 2) * img + pair * 2;
        o[0] = c.ix[0].x; o[1] = c.ix[0].y; o[img] = c.iy[0].x; o[img + 1] = c.iy[0].y;
    }
}

__global__ void mpi_debug_division_kernel(const float* a, const float* b, float* out_fast, float* out_ieee, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const float x = a[i], y = b[i];
        out_fast[i] = in_safe_range(y) && (x == 0.0f || in_safe_range(x)) ? div_by_rcp(x, y, __frcp_rn(y)) : __fdiv_rn(x, y);
        out_ieee[i] = __fdiv_rn(x, y);
    }
}

__global__ void mpi_debug_cam_rays_kernel(const float* __restrict__ cam, float* __restrict__ ray_dir, int V, int H, int W) {
    const size_t img = (size_t)H * W;
    const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int v = blockIdx.y;
    if (pix >= img) return;
    float rx, ry, rz;
    cam_ray(cam + 16 * (size_t)v, (int)(pix % W), (int)(pix / W), H, W, rx, ry, rz);
    float* o = ray_dir + (size_t)v * 3 * img + pix;
    o[0] = rx; o[img] = ry; o[2 * img] = rz;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
}  // namespace gmpi

using namespace gmpi;

static std::atomic<int> g_fwd_variant{0};   // 0 auto, 1 direct, 2 staged (test hook; relaxed atomic: any thread may set it)

// Argument checks shared by every entry point.  `bwd`: gradients instead of outputs.
static int check_params(const RenderParams& p, bool bwd) {
    const bool factored = p.alpha != nullptr || p.rgb != nullptr;
    if (factored ? (!p.alpha || !p.rgb || p.rgba) : !p.rgba)
        return fail(GMPI_ERR_INVALID_ARGUMENT, "null input pointer (MPI: pass rgba, or rgb + alpha)");
    if (!p.view2mpi || !p.dhw) return fail(GMPI_ERR_INVALID_ARGUMENT, "null input pointer");
    if (!p.cam && (!p.ray_dir || !p.eye || !p.z_dir))
        return fail(GMPI_ERR_INVALID_ARGUMENT, "null input pointer (camera: pass ray_dir + eye + z_dir, or cam)");
    if (p.M < 1 || p.V < 0 || p.N < 1 || p.Ht < 1 || p.Wt < 1 || p.H < 1 || p.W < 1)
        return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes M=%d V=%d N=%d Ht=%d Wt=%d H=%d W=%d", p.M, p.V, p.N, p.Ht, p.Wt, p.H, p.W);
    if ((size_t)p.Ht * p.Wt > (size_t)0x7fffffff)
        return fail(GMPI_ERR_UNSUPPORTED, "texture of %dx%d texels exceeds 2^31 elements per channel", p.Ht, p.Wt);
    if (p.view_group < 0 || (p.view_group > 1 && p.V % p.view_group != 0))
        return fail(GMPI_ERR_INVALID_ARGUMENT, "view_group=%d does not divide V=%d", p.view_group, p.V);
    if (!(p.stop_transmittance >= 0.0f && p.stop_transmittance < 1.0f))      // (NaN fails both comparisons)
        return fail(GMPI_ERR_INVALID_ARGUMENT, "stop_transmittance=%g must be in [0, 1)", (double)p.stop_transmittance);
    if (p.stop_transmittance > 0.0f) {
        if (bwd)
            return fail(GMPI_ERR_INVALID_ARGUMENT, "stop_transmittance > 0 in the backward: gradients are exact, the backward "
                        "composites every plane");
        if (p.transmittance)
            return fail(GMPI_ERR_INVALID_ARGUMENT, "stop_transmittance > 0 with a transmittance buffer: the training forward saves "
                        "every T, termination is for inference only");
    }
    if (bwd) {
        if (p.cam) return fail(GMPI_ERR_UNSUPPORTED, "the backward needs the reference's ray tensors (cam is forward-only)");
        if (!p.g_color) return fail(GMPI_ERR_INVALID_ARGUMENT, "null gradient pointer");
        if (factored ? (!p.g_rgb || !p.g_alpha || (p.bg_rgb && !p.g_bg_rgb) || p.g_rgba) : !p.g_rgba)
            return fail(GMPI_ERR_INVALID_ARGUMENT, "null gradient pointer (pass g_rgba, or g_rgb + g_alpha [+ g_bg_rgb])");
    }
    return GMPI_OK;
}

// staged needs 16-byte row strides for the tensor map and enough tiles to fill the persistent grid; `why` receives the
// GMPI_WHY_* bits of every reason the TMA-staged kernel is NOT used (0 = staged)
static bool staged_eligible(int V, int N, int Ht, int Wt, int H, int W, uint32_t* why = nullptr) {
    (void)Ht;
    uint32_t w = 0;
    if (N > kMaxPlanesStaged) w |= GMPI_WHY_MANY_PLANES;
    if (Wt % 4 != 0) w |= GMPI_WHY_TEX_WIDTH;
    const int forced = g_fwd_variant.load(std::memory_order_relaxed);
    if (forced == 1) w |= GMPI_WHY_FORCED;
    const long tiles = (long)((W + kTileW - 1) / kTileW) * ((H + kTileH - 1) / kTileH) * V;
    if (forced != 2 && tiles < 120) w |= GMPI_WHY_FEW_TILES;
    if (why) *why = w;
    return w == 0;
}

static bool aligned16(const void* a) { return ((uintptr_t)a & 15) == 0; }
static bool mpi_aligned(const RenderParams& p) {
    return p.alpha ? aligned16(p.rgb) && aligned16(p.alpha) && (!p.bg_rgb || aligned16(p.bg_rgb)) : aligned16(p.rgba);
}

// Tensor maps of the MPI (expanded or factored) for the five box-width classes.  Returns 0 on success.
// box_h, colour_rows: the ring's box height and kColourCopyRows (factored: colour copies of colour_rows rows, one alpha copy of box_h).
// wide: the factored forward's ring (FwdRingWide) -- slot 4 holds the kWideBW-wide boxes, slot 1 the 64-wide ones, the rest unused.
static int encode_mpi_maps(TmaMaps& maps, const RenderParams& p, int box_h, int colour_rows, bool wide = false) {
    for (int k = 0; k < kNumMaps; ++k) {
        const int bw = (wide && k == kNumMaps - 1) ? kWideBW : kMinBW + k * kBWStep;
        if (p.alpha) {
            if (encode_color_map(&maps.rgb[k], p.rgb, (uint64_t)p.M, p.Ht, p.Wt, bw, colour_rows) != 0) return -1;
            if (p.bg_rgb && encode_color_map(&maps.bg[k], p.bg_rgb, (uint64_t)p.M, p.Ht, p.Wt, bw, colour_rows) != 0) return -1;
            if (encode_slab_map(&maps.a[k], p.alpha, (uint64_t)p.M * p.N, p.Ht, p.Wt, bw, box_h, 1) != 0) return -1;
        } else {
            CUtensorMap* const by_rows[4] = {&maps.m[k], &maps.m8[k], &maps.m16[k], &maps.m32[k]};
            for (int b = 0; b < 4; ++b)
                if (encode_plane_map(by_rows[b], p.rgba, (uint64_t)p.M * p.N, p.Ht, p.Wt, bw, kRowsPerOp << b) != 0) return -1;
        }
    }
    return 0;
}

static int device_sms(int* sms) {
    int dev = 0;
    GMPI_CUDA_OK(cudaGetDevice(&dev));
    GMPI_CUDA_OK(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return GMPI_OK;
}

template <bool AC, bool EMIT, bool FAC>
static cudaError_t launch_fwd_staged(const RenderParams& p, const TmaMaps& maps, int grid, int tiles_x, int tiles_y, cudaStream_t st) {
    auto kernel = mpi_fwd_staged_kernel<AC, EMIT, FAC>;
    constexpr size_t smem = FwdRingFor<FAC>::kWideFact ? kStagedSmemWide : kStagedSmem;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, kStagedThreads, smem, st>>>(p, maps, tiles_x, tiles_y);
    return cudaSuccess;
}
template <bool AC, bool FAC>
static cudaError_t launch_fwd_cut(const RenderParams& p, const TmaMaps& maps, int grid, int tiles_x, int tiles_y, cudaStream_t st) {
    auto kernel = mpi_fwd_cut_kernel<AC, FAC>;
    constexpr size_t smem = FwdRingFor<FAC>::kWideFact ? kStagedSmemWide : kStagedSmem;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, kStagedThreads, smem, st>>>(p, maps, tiles_x, tiles_y, p.stop_transmittance, p.skipped);
    return cudaSuccess;
}
template <bool AC, bool FAC, bool CUT>
static cudaError_t launch_fwd_skip(const RenderParams& p, const TmaMaps& maps, int grid, int tiles_x, int tiles_y, const uint64_t* occ,
                                   unsigned long long* empty, cudaStream_t st) {
    auto kernel = mpi_fwd_skip_kernel<AC, FAC, CUT>;
    constexpr size_t smem = FwdRingFor<FAC>::kWideFact ? kStagedSmemWide : kStagedSmem;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, kStagedThreads, smem, st>>>(p, maps, tiles_x, tiles_y, p.stop_transmittance, p.skipped, occ, empty);
    return cudaSuccess;
}
typedef cudaError_t (*SkipLaunch)(const RenderParams&, const TmaMaps&, int, int, int, const uint64_t*, unsigned long long*, cudaStream_t);
static const SkipLaunch kSkipLaunch[2][2][2] = {     // [align_corners][factored][stop_transmittance > 0]
    {{launch_fwd_skip<false, false, false>, launch_fwd_skip<false, false, true>},
     {launch_fwd_skip<false, true, false>, launch_fwd_skip<false, true, true>}},
    {{launch_fwd_skip<true, false, false>, launch_fwd_skip<true, false, true>},
     {launch_fwd_skip<true, true, false>, launch_fwd_skip<true, true, true>}}};

// Forward launch for a filled RenderParams.  occ (nullable): the occupancy map of empty-space skipping, honoured by the staged
// kernels (the direct kernel renders every plane); `empty` (nullable) accumulates the pixel-planes skipped as empty.
static int launch_fwd(RenderParams p, cudaStream_t st, const uint64_t* occ = nullptr, unsigned long long* empty = nullptr) {
    int rc = check_params(p, false);
    if (rc) return rc;
    if (!p.flags) return fail(GMPI_ERR_INVALID_ARGUMENT, "null flags pointer");
    if (p.video_rgb) {
        if (p.n_peers > 0) return fail(GMPI_ERR_INVALID_ARGUMENT, "video outputs and peer frames are exclusive");
        if (p.video_depth && !(p.depth_range != 0.0f)) return fail(GMPI_ERR_INVALID_ARGUMENT, "depth_range must be non-zero");
    } else if (p.n_peers > 0) {
        if (!p.peer_frames || p.frame_offset < 0) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad peer frame buffers");
    } else if (!p.color || !p.depth) {
        return fail(GMPI_ERR_INVALID_ARGUMENT, "null output pointer");
    }
    if (p.V == 0) return GMPI_OK;
    if (!p.eye0) p.eye0 = p.cam ? p.cam + 13 : p.eye;
    if (p.view_group < 1) p.view_group = 1;
    // float4 epilogue stores: whole quads of x stay inside a row and every destination is 16-byte aligned.  Peer buffers are
    // symmetric-memory allocations (256-byte aligned bases; frame slabs are multiples of 16 bytes when W % 4 == 0).
    if (p.W % 4 == 0 && !p.video_rgb && (p.n_peers > 0 || (aligned16(p.color) && aligned16(p.depth)))) p.options |= kOptVec4Stores;
    const bool ac = (p.options & GMPI_ALIGN_CORNERS) != 0, emit = p.transmittance != nullptr, fac = p.alpha != nullptr;
    if (staged_eligible(p.V, p.N, p.Ht, p.Wt, p.H, p.W) && mpi_aligned(p) && (size_t)p.M * p.N < ((size_t)1 << 31)) {
        TmaMaps maps;
        if (encode_mpi_maps(maps, p, kMaxBH, FwdRingFor<true>::kColourCopyRows, fac && FwdRingFor<true>::kWideFact) != 0) {
            if (g_fwd_variant.load(std::memory_order_relaxed) == 2) return fail(GMPI_ERR_CUDA, "cuTensorMapEncodeTiled failed");
        } else {
            int sms = 0;
            if ((rc = device_sms(&sms)) != 0) return rc;
            const int tiles_x = (p.W + kTileW - 1) / kTileW, tiles_y = (p.H + kTileH - 1) / kTileH;
            const long n_tiles = (long)tiles_x * tiles_y * p.V;
            const int grid = (int)(n_tiles < (long)sms * kCtasPerSm ? n_tiles : (long)sms * kCtasPerSm);
            cudaError_t e;
            if (occ) {                              // (gmpi_mpi_render_fwd_skip_ex: never together with the transmittance output)
                e = kSkipLaunch[ac][fac][p.stop_transmittance > 0.0f](p, maps, grid, tiles_x, tiles_y, occ, empty, st);
            } else if (p.stop_transmittance > 0.0f) {      // (check_params: never together with the transmittance output)
                if (fac) e = ac ? launch_fwd_cut<true, true>(p, maps, grid, tiles_x, tiles_y, st) : launch_fwd_cut<false, true>(p, maps, grid, tiles_x, tiles_y, st);
                else e = ac ? launch_fwd_cut<true, false>(p, maps, grid, tiles_x, tiles_y, st) : launch_fwd_cut<false, false>(p, maps, grid, tiles_x, tiles_y, st);
            } else if (fac) {
                if (ac && emit) e = launch_fwd_staged<true, true, true>(p, maps, grid, tiles_x, tiles_y, st);
                else if (ac) e = launch_fwd_staged<true, false, true>(p, maps, grid, tiles_x, tiles_y, st);
                else if (emit) e = launch_fwd_staged<false, true, true>(p, maps, grid, tiles_x, tiles_y, st);
                else e = launch_fwd_staged<false, false, true>(p, maps, grid, tiles_x, tiles_y, st);
            } else {
                if (ac && emit) e = launch_fwd_staged<true, true, false>(p, maps, grid, tiles_x, tiles_y, st);
                else if (ac) e = launch_fwd_staged<true, false, false>(p, maps, grid, tiles_x, tiles_y, st);
                else if (emit) e = launch_fwd_staged<false, true, false>(p, maps, grid, tiles_x, tiles_y, st);
                else e = launch_fwd_staged<false, false, false>(p, maps, grid, tiles_x, tiles_y, st);
            }
            GMPI_CUDA_OK(e);
            GMPI_CUDA_OK(cudaGetLastError());
            return GMPI_OK;
        }
    }
    p.options &= ~kOptVec4Stores;      // the direct kernel stores pixel by pixel
    const size_t smem = sizeof(PlaneConst) * (size_t)p.N;
    if (smem > 200 * 1024) return fail(GMPI_ERR_UNSUPPORTED, "N=%d planes exceed the shared-memory plane table", p.N);
    dim3 block(kFwdTileW, kFwdTileH);
    dim3 grid((p.W + kFwdTileW - 1) / kFwdTileW, (p.H + kFwdTileH - 1) / kFwdTileH, p.V);
    if (grid.y > 65535) return fail(GMPI_ERR_UNSUPPORTED, "image height %d too large", p.H);
    if (p.V > 65535) return fail(GMPI_ERR_UNSUPPORTED, "V=%d views exceed one launch of the direct kernel (65535); split the batch", p.V);
    const bool cut = p.stop_transmittance > 0.0f;
    void (*kernel)(const RenderParams) = ac ? (cut ? mpi_fwd_direct_cut_kernel<true> : mpi_fwd_direct_kernel<true>)
                                            : (cut ? mpi_fwd_direct_cut_kernel<false> : mpi_fwd_direct_kernel<false>);
    if (smem > 48 * 1024) GMPI_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, block, smem, st>>>(p);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

static std::atomic<int> g_bwd_zero_in_kernel{0};      // 1: GMPI_ZERO_GRAD inside the staged backward kernel (gmpi_debug_set_bwd_zero; measured slower)

static int zero_grads(const RenderParams& p, cudaStream_t st) {
    const size_t tex = (size_t)p.Ht * p.Wt;
    if (p.g_alpha) {
        GMPI_CUDA_OK(cudaMemsetAsync(p.g_rgb, 0, sizeof(float) * (size_t)p.M * 3 * tex, st));
        GMPI_CUDA_OK(cudaMemsetAsync(p.g_alpha, 0, sizeof(float) * (size_t)p.M * p.N * tex, st));
        if (p.g_bg_rgb) GMPI_CUDA_OK(cudaMemsetAsync(p.g_bg_rgb, 0, sizeof(float) * (size_t)p.M * 3 * tex, st));
    } else {
        GMPI_CUDA_OK(cudaMemsetAsync(p.g_rgba, 0, sizeof(float) * (size_t)p.M * p.N * 4 * tex, st));
    }
    return GMPI_OK;
}

// Two-pass direct backward (any shape, no saved state).
static int launch_bwd_direct(RenderParams p, cudaStream_t st, bool zero) {
    if (zero && (p.options & GMPI_ZERO_GRAD)) {
        int rc = zero_grads(p, st);
        if (rc) return rc;
    }
    if (p.V == 0) return GMPI_OK;
    p.eye0 = p.eye;
    if (p.view_group < 1) p.view_group = 1;
    // tile: as many threads (<=128) as the per-thread transmittance stash allows
    int tile_w = 32, tile_h = 4;
    size_t smem = 0;
    for (;; tile_h >>= 1) {
        if (tile_h == 0) return fail(GMPI_ERR_UNSUPPORTED, "N=%d planes exceed the backward stash (227 KB / 32 threads)", p.N);
        smem = sizeof(PlaneConst) * (size_t)p.N + sizeof(float) * (size_t)p.N * tile_w * tile_h;
        if (smem <= 227 * 1024) break;
    }
    dim3 block(tile_w, tile_h);
    dim3 grid((p.W + tile_w - 1) / tile_w, (p.H + tile_h - 1) / tile_h, p.V);
    if (grid.y > 65535) return fail(GMPI_ERR_UNSUPPORTED, "image height %d too large", p.H);
    if (p.V > 65535) return fail(GMPI_ERR_UNSUPPORTED, "V=%d views exceed one launch of the direct kernel (65535); split the batch", p.V);
    if (p.options & GMPI_ALIGN_CORNERS) {
        GMPI_CUDA_OK(cudaFuncSetAttribute(mpi_bwd_direct_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mpi_bwd_direct_kernel<true><<<grid, block, smem, st>>>(p, tile_w, tile_h);
    } else {
        GMPI_CUDA_OK(cudaFuncSetAttribute(mpi_bwd_direct_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mpi_bwd_direct_kernel<false><<<grid, block, smem, st>>>(p, tile_w, tile_h);
    }
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

template <bool AC, bool FAC>
static cudaError_t launch_bwd_box(const RenderParams& p, const TmaMaps& maps, int grid, int tiles_x, int tiles_y, cudaStream_t st) {
    auto kernel = mpi_bwd_box_kernel<AC, FAC>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, kBwdThreads, kBwdSmem, st>>>(p, maps, tiles_x, tiles_y);
    return cudaSuccess;
}

// Backward: the staged box kernel when the forward saved the transmittance and the shapes allow, else the direct kernel.
static int launch_bwd(RenderParams p, cudaStream_t st) {
    int rc = check_params(p, true);
    if (rc) return rc;
    const bool fac = p.alpha != nullptr;
    const bool grads_aligned = fac ? aligned16(p.g_rgb) && aligned16(p.g_alpha) && (!p.g_bg_rgb || aligned16(p.g_bg_rgb)) : aligned16(p.g_rgba);
    if (!(p.transmittance && staged_eligible(p.V, p.N, p.Ht, p.Wt, p.H, p.W) && mpi_aligned(p) && grads_aligned &&
          (size_t)p.M * p.N < ((size_t)1 << 31) && p.W % 4 == 0 && aligned16(p.transmittance) && (size_t)p.V * p.N < ((size_t)1 << 31)))
        return launch_bwd_direct(p, st, true);
    if (p.V == 0) return (p.options & GMPI_ZERO_GRAD) ? zero_grads(p, st) : GMPI_OK;
    p.eye0 = p.eye;
    if (p.view_group < 1) p.view_group = 1;
    TmaMaps maps;
    if (encode_mpi_maps(maps, p, kBwdMaxBH, BwdRing::kColourCopyRows) != 0) return fail(GMPI_ERR_CUDA, "cuTensorMapEncodeTiled failed");
    if (encode_slab_map(&maps.t, p.transmittance, (uint64_t)p.V * p.N, p.H, p.W, kTileW, kBwdTileH, 1) != 0)
        return fail(GMPI_ERR_CUDA, "cuTensorMapEncodeTiled (transmittance) failed");
    int sms = 0;
    if ((rc = device_sms(&sms)) != 0) return rc;
    const int tiles_x = (p.W + kTileW - 1) / kTileW, tiles_y = (p.H + kBwdTileH - 1) / kBwdTileH;
    const long n_tiles = (long)tiles_x * tiles_y * p.V;
    const int grid = (int)(n_tiles < sms ? n_tiles : sms);
    const bool ac = (p.options & GMPI_ALIGN_CORNERS) != 0;
    // GMPI_ZERO_GRAD: stream memsets before the kernel (default), or -- gmpi_debug_set_bwd_zero(1) -- the kernel zeroes the large
    // buffer (g_rgba / g_alpha) itself, one MPI slab ahead of the tiles that add to it (GradZeroPacer, measured 4.5 % slower); the
    // small factored colour gradients and the counters then take stream-ordered memsets.
    unsigned* zero_flags = nullptr;
    if (p.options & GMPI_ZERO_GRAD) {
        const size_t tex = (size_t)p.Ht * p.Wt;
        if (g_bwd_zero_in_kernel.load(std::memory_order_relaxed) &&
            cudaMallocAsync(reinterpret_cast<void**>(&zero_flags), sizeof(unsigned) * (size_t)p.M, st) == cudaSuccess) {
            cudaError_t ez = cudaMemsetAsync(zero_flags, 0, sizeof(unsigned) * (size_t)p.M, st);
            if (ez == cudaSuccess && fac) {
                ez = cudaMemsetAsync(p.g_rgb, 0, sizeof(float) * (size_t)p.M * 3 * tex, st);
                if (ez == cudaSuccess && p.g_bg_rgb) ez = cudaMemsetAsync(p.g_bg_rgb, 0, sizeof(float) * (size_t)p.M * 3 * tex, st);
            }
            if (ez != cudaSuccess) {
                (void)cudaFreeAsync(zero_flags, st);
                GMPI_CUDA_OK(ez);
            }
            p.zero_base = reinterpret_cast<float4*>(fac ? p.g_alpha : p.g_rgba);
            p.zero_slab16 = (unsigned long long)p.N * (fac ? 1 : 4) * tex / 4;            // Wt % 4 == 0: whole float4s
            p.zero_flags = zero_flags;
            // pace: a CTA's share of one slab within half of the stages it spends on one MPI's tiles
            const double stages_per_mpi = (double)n_tiles / p.M / grid * p.N;
            const double stores = (double)p.zero_slab16 / grid / 32.0;
            double rate = stores / (0.5 * stages_per_mpi > 1.0 ? 0.5 * stages_per_mpi : 1.0);
            p.zero_rate = rate < 4.0 ? 4 : rate > 4096.0 ? 4096 : (int)rate + 1;
        } else {
            (void)cudaGetLastError();
            zero_flags = nullptr;
            if ((rc = zero_grads(p, st)) != 0) return rc;
        }
    }
    cudaError_t e;
    if (fac) e = ac ? launch_bwd_box<true, true>(p, maps, grid, tiles_x, tiles_y, st) : launch_bwd_box<false, true>(p, maps, grid, tiles_x, tiles_y, st);
    else e = ac ? launch_bwd_box<true, false>(p, maps, grid, tiles_x, tiles_y, st) : launch_bwd_box<false, false>(p, maps, grid, tiles_x, tiles_y, st);
    if (zero_flags) (void)cudaFreeAsync(zero_flags, st);
    GMPI_CUDA_OK(e);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

static RenderParams params_from_desc(const gmpi_render_desc* d) {
    RenderParams p{};
    p.rgba = d->rgba; p.rgb = d->rgb; p.alpha = d->alpha; p.bg_rgb = d->bg_rgb;
    p.view2mpi = d->view2mpi; p.dhw = d->dhw; p.ray_dir = d->ray_dir; p.eye = d->eye; p.z_dir = d->z_dir; p.cam = d->cam;
    p.color = d->color; p.depth = d->depth; p.transmittance = d->transmittance; p.flags = d->flags;
    p.peer_frames = d->peer_frames; p.n_peers = d->n_peers; p.frame_offset = d->frame_offset;
    p.video_rgb = d->video_rgb; p.video_depth = d->video_depth; p.depth_near = d->depth_near; p.depth_range = d->depth_range;
    p.g_color = d->g_color; p.g_depth = d->g_depth; p.g_rgba = d->g_rgba; p.g_rgb = d->g_rgb; p.g_bg_rgb = d->g_bg_rgb; p.g_alpha = d->g_alpha;
    p.M = d->M; p.V = d->V; p.N = d->N; p.Ht = d->Ht; p.Wt = d->Wt; p.H = d->H; p.W = d->W;
    p.view_group = d->view_group;
    p.options = d->options & 0xffffu;      // the upper bits are internal
    if (d->struct_bytes >= sizeof(gmpi_render_desc)) {      // the early-termination fields (an older descriptor ends before them)
        p.stop_transmittance = d->stop_transmittance;
        p.skipped = reinterpret_cast<unsigned long long*>(d->skipped_pixel_planes);
    }
    return p;
}

static constexpr size_t kDescBytesWithoutStop = offsetof(gmpi_render_desc, stop_transmittance);
static_assert(sizeof(uint64_t) == sizeof(unsigned long long), "skip counter");

static int check_desc(const gmpi_render_desc* d) {
    if (!d) return fail(GMPI_ERR_INVALID_ARGUMENT, "null descriptor");
    // the descriptor before the early-termination fields (everything up to stop_transmittance) is accepted: they read as absent
    if (d->struct_bytes != sizeof(gmpi_render_desc) && d->struct_bytes != kDescBytesWithoutStop)
        return fail(GMPI_ERR_INVALID_ARGUMENT, "gmpi_render_desc.struct_bytes = %u, this library expects %zu (ABI %d) or %zu (without stop_transmittance)",
                    d->struct_bytes, sizeof(gmpi_render_desc), GMPI_ABI_VERSION, kDescBytesWithoutStop);
    return GMPI_OK;
}

static RenderParams params_classic(const float* rgba, const int32_t* view2mpi, const float* dhw, const float* ray_dir, const float* eye,
                                   const float* z_dir, int M, int V, int N, int Ht, int Wt, int H, int W, uint32_t options) {
    RenderParams p{};
    p.rgba = rgba; p.view2mpi = view2mpi; p.dhw = dhw; p.ray_dir = ray_dir; p.eye = eye; p.z_dir = z_dir;
    p.M = M; p.V = V; p.N = N; p.Ht = Ht; p.Wt = Wt; p.H = H; p.W = W;
    p.options = options & 0xffffu;
    p.view_group = 1;
    return p;
}

extern "C" {

int gmpi_abi_version(void) { return GMPI_ABI_VERSION; }

const char* gmpi_last_error(void) { return g_err; }

int gmpi_debug_set_bwd_zero(int in_kernel) {
    g_bwd_zero_in_kernel.store(in_kernel != 0, std::memory_order_relaxed);
    return GMPI_OK;
}

int gmpi_debug_set_fwd_variant(int variant) {
    if (variant < 0 || variant > 2) return fail(GMPI_ERR_INVALID_ARGUMENT, "variant must be 0 (auto), 1 (direct) or 2 (staged)");
    g_fwd_variant.store(variant, std::memory_order_relaxed);
    return GMPI_OK;
}

// Host evaluation of the staged kernels' tile order (same TileWalk code): tiles of CTA `cta` in a grid of `grid` CTAs, as
// (view, px0, py0) triples.  Returns the count, or a negative error.
int gmpi_debug_tile_walk_ex(int H, int W, int V, int tile_h, int view_group, int grid, int cta, int* out_v_px0_py0, int max_tiles) {
    if (H < 1 || W < 1 || V < 1 || tile_h < 1 || grid < 1 || cta < 0 || cta >= grid || max_tiles < 0 || (max_tiles > 0 && !out_v_px0_py0))
        return -fail(GMPI_ERR_INVALID_ARGUMENT, "gmpi_debug_tile_walk: bad argument");
    TileWalk w;
    w.init((W + kTileW - 1) / kTileW, H, V, cta, grid, tile_h, view_group);
    TileXY t;
    int n = 0;
    for (; w.at(n, t); ++n)
        if (n < max_tiles) { out_v_px0_py0[3 * n] = t.v; out_v_px0_py0[3 * n + 1] = t.px0; out_v_px0_py0[3 * n + 2] = t.py0; }
    return n;
}

// Host evaluation of the expanded forward's copies of one stage (same code as the producer): for a footprint of n_rows staged rows
// (a multiple of 4, at most the ring's box height) writes (first row, rows) of every copy; returns their number.
int gmpi_debug_copy_plan(int n_rows, int* out_row_rows, int max_copies) {
    if (n_rows < 0 || n_rows % kRowsPerOp != 0 || n_rows > kMaxBH || max_copies < 0 || (max_copies > 0 && !out_row_rows))
        return -fail(GMPI_ERR_INVALID_ARGUMENT, "gmpi_debug_copy_plan: n_rows must be a multiple of %d in [0, %d]", kRowsPerOp, kMaxBH);
    int n = 0;
    for (int lane = 0; lane < 4; ++lane) {
        int before;
        const int h = binary_copy_of_lane(n_rows / kRowsPerOp, lane, before);
        if (!h) continue;
        if (n < max_copies) { out_row_rows[2 * n] = before * kRowsPerOp; out_row_rows[2 * n + 1] = h * kRowsPerOp; }
        ++n;
    }
    return n;
}

int gmpi_debug_tile_walk(int H, int W, int V, int grid, int cta, int* out_v_px0_py0, int max_tiles) {
    return gmpi_debug_tile_walk_ex(H, W, V, kTileH, 1, grid, cta, out_v_px0_py0, max_tiles);
}

int gmpi_mpi_render_fwd_plan(int V, int N, int Ht, int Wt, int H, int W, const void* rgba, uint32_t* why) {
    uint32_t w = 0;
    staged_eligible(V, N, Ht, Wt, H, W, &w);
    if (rgba && ((uintptr_t)rgba & 15) != 0) w |= GMPI_WHY_ALIGNMENT;
    if (why) *why = w;
    return w == 0 ? GMPI_PLAN_STAGED : GMPI_PLAN_DIRECT;
}

const char* gmpi_mpi_render_fwd_variant(int N, int Ht, int Wt, int H, int W) {
    return staged_eligible(1 << 20, N, Ht, Wt, H, W) ? "fwd_staged_tma_64x30" : "fwd_direct_32x8";
}

int gmpi_mpi_render_fwd(const float* rgba, const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                        const float* eye, const float* z_dir, float* color, float* depth, uint32_t* flags, int M,
                        int V, int N, int Ht, int Wt, int H, int W, uint32_t options, void* stream) {
    RenderParams p = params_classic(rgba, view2mpi, dhw, ray_dir, eye, z_dir, M, V, N, Ht, Wt, H, W, options);
    p.color = color; p.depth = depth; p.flags = flags;
    return launch_fwd(p, (cudaStream_t)stream);
}

int gmpi_mpi_render_fwd_train(const float* rgba, const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                              const float* eye, const float* z_dir, float* color, float* depth, float* transmittance,
                              uint32_t* flags, int M, int V, int N, int Ht, int Wt, int H, int W, uint32_t options,
                              void* stream) {
    if (!transmittance) return fail(GMPI_ERR_INVALID_ARGUMENT, "null transmittance buffer");
    RenderParams p = params_classic(rgba, view2mpi, dhw, ray_dir, eye, z_dir, M, V, N, Ht, Wt, H, W, options);
    p.color = color; p.depth = depth; p.flags = flags; p.transmittance = transmittance;
    return launch_fwd(p, (cudaStream_t)stream);
}

int gmpi_mpi_render_fwd_gather(const float* rgba, const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                               const float* eye, const float* z_dir, float* const* peer_frames, int n_peers,
                               int frame_offset, uint32_t* flags, int M, int V, int N, int Ht, int Wt, int H, int W,
                               uint32_t options, void* stream) {
    if (n_peers < 1) return fail(GMPI_ERR_INVALID_ARGUMENT, "n_peers must be >= 1");
    RenderParams p = params_classic(rgba, view2mpi, dhw, ray_dir, eye, z_dir, M, V, N, Ht, Wt, H, W, options);
    p.flags = flags; p.peer_frames = peer_frames; p.n_peers = n_peers; p.frame_offset = frame_offset;
    return launch_fwd(p, (cudaStream_t)stream);
}

int gmpi_mpi_render_bwd(const float* rgba, const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                        const float* eye, const float* z_dir, const float* g_color, const float* g_depth,
                        float* g_rgba, int M, int V, int N, int Ht, int Wt, int H, int W, uint32_t options,
                        void* stream) {
    RenderParams p = params_classic(rgba, view2mpi, dhw, ray_dir, eye, z_dir, M, V, N, Ht, Wt, H, W, options);
    p.g_color = g_color; p.g_depth = g_depth; p.g_rgba = g_rgba;
    return launch_bwd(p, (cudaStream_t)stream);
}

int gmpi_mpi_render_bwd_saved(const float* rgba, const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                              const float* eye, const float* z_dir, const float* transmittance, const float* g_color,
                              const float* g_depth, float* g_rgba, int M, int V, int N, int Ht, int Wt, int H, int W,
                              uint32_t options, void* stream) {
    if (!transmittance) return fail(GMPI_ERR_INVALID_ARGUMENT, "null gradient / transmittance pointer");
    RenderParams p = params_classic(rgba, view2mpi, dhw, ray_dir, eye, z_dir, M, V, N, Ht, Wt, H, W, options);
    p.g_color = g_color; p.g_depth = g_depth; p.g_rgba = g_rgba; p.transmittance = const_cast<float*>(transmittance);
    return launch_bwd(p, (cudaStream_t)stream);
}

int gmpi_mpi_zero_async(void* ptr, size_t bytes, void* stream) {
    if (!ptr && bytes) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    GMPI_CUDA_OK(cudaMemsetAsync(ptr, 0, bytes, (cudaStream_t)stream));
    return GMPI_OK;
}

int gmpi_mpi_render_fwd_ex(const gmpi_render_desc* d) {
    int rc = check_desc(d);
    if (rc) return rc;
    return launch_fwd(params_from_desc(d), (cudaStream_t)d->stream);
}

int gmpi_mpi_render_fwd_skip_ex(const gmpi_render_desc* d, const uint64_t* occupancy, uint64_t* empty_pixel_planes) {
    int rc = check_desc(d);
    if (rc) return rc;
    if (!occupancy) return fail(GMPI_ERR_INVALID_ARGUMENT, "null occupancy map (gmpi_mpi_occupancy builds it)");
    if (d->transmittance)
        return fail(GMPI_ERR_INVALID_ARGUMENT, "empty-space skipping with a transmittance buffer: the training forward saves every T "
                    "and stays exact, skipping is for inference only");
    return launch_fwd(params_from_desc(d), (cudaStream_t)d->stream, occupancy, reinterpret_cast<unsigned long long*>(empty_pixel_planes));
}

size_t gmpi_mpi_occupancy_plane_words(int Ht, int Wt) {
    if (Ht < 1 || Wt < 1) return 0;
    return (size_t)((Ht + 7) / 8) * (size_t)((Wt + 511) / 512);
}

int gmpi_mpi_occupancy(const float* alpha, long long mpi_stride, long long plane_stride, int M, int N, int Ht, int Wt, float threshold,
                       uint64_t* occupancy, void* stream) {
    if (!alpha || !occupancy) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (!(threshold >= 0.0f && threshold < 1.0f))      // (NaN fails both comparisons)
        return fail(GMPI_ERR_INVALID_ARGUMENT, "occupancy threshold=%g must be in [0, 1)", (double)threshold);
    if (M < 1 || N < 1 || Ht < 1 || Wt < 1 || mpi_stride < 0 || plane_stride < 0)
        return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes M=%d N=%d Ht=%d Wt=%d", M, N, Ht, Wt);
    const int n_wy = (Ht + 7) / 8, n_wx = (Wt + 511) / 512;
    const long long n_words = (long long)M * N * n_wy * n_wx;
    const long long blocks = (n_words + 7) / 8;      // 8 warps of 256 threads, one word each
    if (blocks > 0x7fffffffLL) return fail(GMPI_ERR_UNSUPPORTED, "%lld occupancy words exceed one launch", n_words);
    cudaStream_t st = (cudaStream_t)stream;
    if (Wt % 4 == 0 && plane_stride % 4 == 0 && mpi_stride % 4 == 0 && ((uintptr_t)alpha & 15) == 0)
        mpi_occupancy_kernel<4><<<(unsigned)blocks, 256, 0, st>>>(alpha, mpi_stride, plane_stride, N, Ht, Wt, n_wy, n_wx, n_words, threshold,
                                                                  occupancy);
    else
        mpi_occupancy_kernel<1><<<(unsigned)blocks, 256, 0, st>>>(alpha, mpi_stride, plane_stride, N, Ht, Wt, n_wy, n_wx, n_words, threshold,
                                                                  occupancy);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_mpi_render_bwd_ex(const gmpi_render_desc* d) {
    int rc = check_desc(d);
    if (rc) return rc;
    return launch_bwd(params_from_desc(d), (cudaStream_t)d->stream);
}

int gmpi_mpi_check_range(const float* rgba, int M, int N, int Ht, int Wt, uint32_t* flags, void* stream) {
    if (!rgba || !flags) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (M < 1 || N < 1 || Ht < 1 || Wt < 1) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t slab = (size_t)Ht * Wt, n_slabs = (size_t)M * N * 4;
    int sms = 148;
    int rc = device_sms(&sms);
    if (rc) return rc;
    const int grid = sms * 8;
    if (slab % 4 == 0 && ((uintptr_t)rgba & 15) == 0) {
        mpi_check_range_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float4*>(rgba), n_slabs, slab / 4, flags);
    } else {
        mpi_check_range_scalar_kernel<<<grid, 256, 0, st>>>(rgba, n_slabs, slab, flags);
    }
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_debug_plane_coords(const int32_t* view2mpi, const float* dhw, const float* ray_dir, const float* eye,
                            float* out, int V, int N, int Ht, int Wt, int H, int W, uint32_t options, void* stream) {
    if (!view2mpi || !dhw || !ray_dir || !eye || !out) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (V < 1 || N < 1 || Ht < 1 || Wt < 1 || H < 1 || W < 1) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t img = (size_t)H * W;
    dim3 grid((unsigned)((img + 255) / 256), V);
    if (options & GMPI_ALIGN_CORNERS)
        mpi_debug_coords_kernel<true><<<grid, 256, 0, st>>>(view2mpi, dhw, ray_dir, eye, out, V, N, Ht, Wt, H, W);
    else
        mpi_debug_coords_kernel<false><<<grid, 256, 0, st>>>(view2mpi, dhw, ray_dir, eye, out, V, N, Ht, Wt, H, W);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_debug_plane_coords_packed(const int32_t* view2mpi, const float* dhw, const float* ray_dir, const float* eye,
                                   float* out, int V, int N, int Ht, int Wt, int H, int W, uint32_t options, void* stream) {
    if (!view2mpi || !dhw || !ray_dir || !eye || !out) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (V < 1 || N < 1 || Ht < 1 || Wt < 1 || H < 1 || W < 1 || ((size_t)H * W) % 2) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t pairs = (size_t)H * W / 2;
    dim3 grid((unsigned)((pairs + 255) / 256), V);
    if (options & GMPI_ALIGN_CORNERS)
        mpi_debug_coords_packed_kernel<true><<<grid, 256, 0, st>>>(view2mpi, dhw, ray_dir, eye, out, V, N, Ht, Wt, H, W);
    else
        mpi_debug_coords_packed_kernel<false><<<grid, 256, 0, st>>>(view2mpi, dhw, ray_dir, eye, out, V, N, Ht, Wt, H, W);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_debug_division(const float* a, const float* b, float* out_fast, float* out_ieee, size_t n, void* stream) {
    if (!a || !b || !out_fast || !out_ieee) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    mpi_debug_division_kernel<<<1184, 256, 0, (cudaStream_t)stream>>>(a, b, out_fast, out_ieee, n);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_debug_cam_rays(const float* cam, float* ray_dir, int V, int H, int W, void* stream) {
    if (!cam || !ray_dir || V < 1 || H < 1 || W < 1) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad argument");
    dim3 grid((unsigned)(((size_t)H * W + 255) / 256), V);
    mpi_debug_cam_rays_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(cam, ray_dir, V, H, W);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

// ------------------------------------------------------------------------------------------
// LightRenderer kernels (gmpi/core/light_renderer.py), SURVEY.md 8(f) N3
// ------------------------------------------------------------------------------------------
static int check_alpha_view(const float* alpha, long long mpi_stride, long long plane_stride, int M, int N, int Ht, int Wt) {
    if (!alpha) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (M < 1 || N < 1 || Ht < 1 || Wt < 1 || M > 65535) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes");
    if (((size_t)Ht * Wt) % 4 != 0 || plane_stride % 4 != 0 || mpi_stride % 4 != 0 || ((uintptr_t)alpha & 15) != 0)
        return fail(GMPI_ERR_UNSUPPORTED, "alpha planes must be 16-byte aligned with Ht*Wt %% 4 == 0 (float4 streaming)");
    return GMPI_OK;
}

int gmpi_mpi_alpha_depth_fwd(const float* alpha, long long mpi_stride, long long plane_stride, const float* plane_d, float* depth,
                             float* transmittance, int M, int N, int Ht, int Wt, void* stream) {
    int rc = check_alpha_view(alpha, mpi_stride, plane_stride, M, N, Ht, Wt);
    if (rc) return rc;
    if (!plane_d || !depth) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    const long long tex4 = (long long)Ht * Wt / 4;
    AlphaView a{alpha, mpi_stride, plane_stride};
    dim3 grid((unsigned)((tex4 + 255) / 256), M);
    if (transmittance) mpi_alpha_depth_fwd_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(a, plane_d, depth, transmittance, N, tex4);
    else mpi_alpha_depth_fwd_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(a, plane_d, depth, nullptr, N, tex4);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_mpi_alpha_depth_bwd(const float* alpha, long long mpi_stride, long long plane_stride, const float* plane_d,
                             const float* transmittance, const float* g_depth, float* g_alpha, long long g_mpi_stride,
                             long long g_plane_stride, int M, int N, int Ht, int Wt, void* stream) {
    int rc = check_alpha_view(alpha, mpi_stride, plane_stride, M, N, Ht, Wt);
    if (rc) return rc;
    if (!plane_d || !transmittance || !g_depth || !g_alpha) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (g_plane_stride % 4 != 0 || g_mpi_stride % 4 != 0 || ((uintptr_t)g_alpha & 15) != 0)
        return fail(GMPI_ERR_UNSUPPORTED, "g_alpha planes must be 16-byte aligned");
    const long long tex4 = (long long)Ht * Wt / 4;
    AlphaView a{alpha, mpi_stride, plane_stride};
    dim3 grid((unsigned)((tex4 + 255) / 256), M);
    mpi_alpha_depth_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a, plane_d, transmittance, g_depth, g_alpha, g_mpi_stride,
                                                                        g_plane_stride, N, tex4);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_mpi_apply_shading_fwd(const float* rgba, const float* shade, float* out, int M, int N, int Ht, int Wt, void* stream) {
    if (!rgba || !shade || !out) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (M < 1 || N < 1 || Ht < 1 || Wt < 1 || M > 65535 || N > 65535) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes");
    if (((size_t)Ht * Wt) % 4 != 0 || (((uintptr_t)rgba | (uintptr_t)shade | (uintptr_t)out) & 15) != 0)
        return fail(GMPI_ERR_UNSUPPORTED, "tensors must be 16-byte aligned with Ht*Wt %% 4 == 0 (float4 streaming)");
    const long long tex4 = (long long)Ht * Wt / 4;
    dim3 grid((unsigned)((tex4 + 255) / 256), N, M);
    mpi_apply_shading_fwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rgba, shade, out, N, tex4);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

int gmpi_mpi_apply_shading_bwd(const float* rgba, const float* shade, const float* g_out, float* g_rgba, float* g_shade, int M, int N,
                               int Ht, int Wt, void* stream) {
    if (!rgba || !shade || !g_out || !g_rgba || !g_shade) return fail(GMPI_ERR_INVALID_ARGUMENT, "null pointer");
    if (M < 1 || N < 1 || Ht < 1 || Wt < 1 || M > 65535) return fail(GMPI_ERR_INVALID_ARGUMENT, "bad sizes");
    if (((size_t)Ht * Wt) % 4 != 0 ||
        (((uintptr_t)rgba | (uintptr_t)shade | (uintptr_t)g_out | (uintptr_t)g_rgba | (uintptr_t)g_shade) & 15) != 0)
        return fail(GMPI_ERR_UNSUPPORTED, "tensors must be 16-byte aligned with Ht*Wt %% 4 == 0 (float4 streaming)");
    const long long tex4 = (long long)Ht * Wt / 4;
    dim3 grid((unsigned)((tex4 + 255) / 256), M);
    mpi_apply_shading_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rgba, shade, g_out, g_rgba, g_shade, N, tex4);
    GMPI_CUDA_OK(cudaGetLastError());
    return GMPI_OK;
}

// ------------------------------------------------------------------------------------------
// host-buffer entry points
// ------------------------------------------------------------------------------------------
// Per-device staging cache (grow-only; released by gmpi_mpi_release_host_cache or at exit): two MPI slots (the copy of MPI m+1
// overlaps the render of MPI m), per-view inputs/outputs, two streams, four events.
struct HostCache {
    float* mpi[2] = {nullptr, nullptr};
    size_t mpi_bytes = 0;
    void* misc = nullptr;           // dhw | ray/cam | eye | z | color | depth | video | v2m | flags, carved from one allocation
    size_t misc_bytes = 0;
    cudaStream_t s_copy = nullptr, s_run = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
};
static HostCache g_host_cache[64];
static std::mutex g_host_mutex[64];     // one call at a time per device: the staging buffers are shared state

static void host_cache_release(HostCache& c) {
    for (int k = 0; k < 2; ++k) {
        if (c.mpi[k]) cudaFree(c.mpi[k]);
        if (c.ev_in[k]) cudaEventDestroy(c.ev_in[k]);
        if (c.ev_free[k]) cudaEventDestroy(c.ev_free[k]);
    }
    if (c.misc) cudaFree(c.misc);
    if (c.s_copy) cudaStreamDestroy(c.s_copy);
    if (c.s_run) cudaStreamDestroy(c.s_run);
    c = HostCache();
}

int gmpi_mpi_release_host_cache(void) {
    int cur = 0;
    cudaGetDevice(&cur);
    for (int d = 0; d < 64; ++d) {
        std::lock_guard<std::mutex> lock(g_host_mutex[d]);
        HostCache& c = g_host_cache[d];
        if (!c.misc && !c.mpi[0] && !c.s_run) continue;
        cudaSetDevice(d);
        host_cache_release(c);
    }
    cudaSetDevice(cur);
    return GMPI_OK;
}

// `h` holds HOST pointers.  Streams every MPI through a double-buffered device slot and renders its views.
static int host_render_locked(HostCache& c, const RenderParams& h, uint32_t* flags_out) {
    int rc = GMPI_OK;
    const int M = h.M, V = h.V, N = h.N, H = h.H, W = h.W;
    const size_t tex = (size_t)h.Ht * h.Wt, img = (size_t)H * W;
    const bool fac = h.alpha != nullptr, video = h.video_rgb != nullptr;
    // one slot = one MPI: expanded [N,4,tex], or factored rgb [3,tex] | bg [3,tex] | alpha [N,tex]
    const size_t o_bg = 3 * tex, o_alpha = h.bg_rgb ? 6 * tex : 3 * tex;
    const size_t mpi_bytes = sizeof(float) * (fac ? o_alpha + (size_t)N * tex : (size_t)N * 4 * tex);
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t o_dhw = 0, o_ray = o_dhw + up(sizeof(float) * (size_t)M * N * 3),
                 o_eye = o_ray + up(h.cam ? sizeof(float) * (size_t)V * 16 : sizeof(float) * (size_t)V * 3 * img),
                 o_z = o_eye + up(sizeof(float) * (size_t)V * 3), o_color = o_z + up(sizeof(float) * (size_t)V * 3),
                 o_depth = o_color + up(video ? (size_t)V * 3 * img : sizeof(float) * (size_t)V * 3 * img),
                 o_v2m = o_depth + up(video ? (size_t)V * img : sizeof(float) * (size_t)V * img),
                 o_flags = o_v2m + up(sizeof(int32_t) * (size_t)(V > 0 ? V : 1)), misc_bytes = o_flags + 256;
    if (!c.s_run) {
        GMPI_CUDA_OK(cudaStreamCreateWithFlags(&c.s_copy, cudaStreamNonBlocking));
        GMPI_CUDA_OK(cudaStreamCreateWithFlags(&c.s_run, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            GMPI_CUDA_OK(cudaEventCreateWithFlags(&c.ev_in[k], cudaEventDisableTiming));
            GMPI_CUDA_OK(cudaEventCreateWithFlags(&c.ev_free[k], cudaEventDisableTiming));
        }
    }
    if (c.mpi_bytes < mpi_bytes) {
        for (int k = 0; k < 2; ++k) {
            if (c.mpi[k]) GMPI_CUDA_OK(cudaFree(c.mpi[k]));
            c.mpi[k] = nullptr;
        }
        c.mpi_bytes = 0;
        for (int k = 0; k < 2; ++k) GMPI_CUDA_OK(cudaMalloc(&c.mpi[k], mpi_bytes));
        c.mpi_bytes = mpi_bytes;
    }
    if (c.misc_bytes < misc_bytes) {
        if (c.misc) GMPI_CUDA_OK(cudaFree(c.misc));
        c.misc = nullptr; c.misc_bytes = 0;
        GMPI_CUDA_OK(cudaMalloc(&c.misc, misc_bytes));
        c.misc_bytes = misc_bytes;
    }
    char* base = static_cast<char*>(c.misc);
    float *d_dhw = (float*)(base + o_dhw), *d_ray = (float*)(base + o_ray), *d_eye = (float*)(base + o_eye), *d_z = (float*)(base + o_z);
    int32_t* d_v2m = (int32_t*)(base + o_v2m);
    uint32_t* d_flags = (uint32_t*)(base + o_flags);
    unsigned long long* d_skipped = (unsigned long long*)(base + o_flags + 8);     // (within the 256 bytes of the flags slot)
    cudaStream_t s_copy = c.s_copy, s_run = c.s_run;
    GMPI_CUDA_OK(cudaMemsetAsync(d_flags, 0, 16, s_run));
    GMPI_CUDA_OK(cudaMemsetAsync(d_v2m, 0, sizeof(int32_t) * (size_t)(V > 0 ? V : 1), s_run));   // a staged MPI is slot-local index 0
    GMPI_CUDA_OK(cudaMemcpyAsync(d_dhw, h.dhw, sizeof(float) * (size_t)M * N * 3, cudaMemcpyHostToDevice, s_run));
    if (h.cam) {
        GMPI_CUDA_OK(cudaMemcpyAsync(d_ray, h.cam, sizeof(float) * (size_t)V * 16, cudaMemcpyHostToDevice, s_run));
    } else {
        GMPI_CUDA_OK(cudaMemcpyAsync(d_ray, h.ray_dir, sizeof(float) * (size_t)V * 3 * img, cudaMemcpyHostToDevice, s_run));
        GMPI_CUDA_OK(cudaMemcpyAsync(d_eye, h.eye, sizeof(float) * (size_t)V * 3, cudaMemcpyHostToDevice, s_run));
        GMPI_CUDA_OK(cudaMemcpyAsync(d_z, h.z_dir, sizeof(float) * (size_t)V * 3, cudaMemcpyHostToDevice, s_run));
    }
    int v0 = 0, slot = 0, used[2] = {0, 0};
    for (int m = 0; m < M; ++m) {
        int v1 = v0;
        while (v1 < V && h.view2mpi[v1] == m) ++v1;
        if (v1 == v0) continue;
        if (used[slot]) GMPI_CUDA_OK(cudaStreamWaitEvent(s_copy, c.ev_free[slot], 0));
        float* d_mpi = c.mpi[slot];
        if (fac) {
            GMPI_CUDA_OK(cudaMemcpyAsync(d_mpi, h.rgb + (size_t)m * 3 * tex, sizeof(float) * 3 * tex, cudaMemcpyHostToDevice, s_copy));
            if (h.bg_rgb)
                GMPI_CUDA_OK(cudaMemcpyAsync(d_mpi + o_bg, h.bg_rgb + (size_t)m * 3 * tex, sizeof(float) * 3 * tex, cudaMemcpyHostToDevice, s_copy));
            GMPI_CUDA_OK(cudaMemcpyAsync(d_mpi + o_alpha, h.alpha + (size_t)m * N * tex, sizeof(float) * (size_t)N * tex, cudaMemcpyHostToDevice, s_copy));
        } else {
            GMPI_CUDA_OK(cudaMemcpyAsync(d_mpi, h.rgba + (size_t)m * N * 4 * tex, mpi_bytes, cudaMemcpyHostToDevice, s_copy));
        }
        GMPI_CUDA_OK(cudaEventRecord(c.ev_in[slot], s_copy));
        GMPI_CUDA_OK(cudaStreamWaitEvent(s_run, c.ev_in[slot], 0));
        RenderParams p = h;
        p.M = 1; p.V = v1 - v0;
        if (fac) { p.rgb = d_mpi; p.bg_rgb = h.bg_rgb ? d_mpi + o_bg : nullptr; p.alpha = d_mpi + o_alpha; p.rgba = nullptr; }
        else p.rgba = d_mpi;
        p.view2mpi = d_v2m; p.dhw = d_dhw + (size_t)m * N * 3;
        // mpi.py:70 compares every plane distance with the eye of the CALL's view 0, not of this launch's first view
        if (h.cam) { p.cam = d_ray + (size_t)v0 * 16; p.eye0 = d_ray + 13; p.ray_dir = p.eye = p.z_dir = nullptr; }
        else { p.ray_dir = d_ray + (size_t)v0 * 3 * img; p.eye = d_eye + (size_t)v0 * 3; p.z_dir = d_z + (size_t)v0 * 3; p.eye0 = d_eye; }
        if (video) {
            p.video_rgb = (uint8_t*)(base + o_color) + (size_t)v0 * 3 * img;
            p.video_depth = h.video_depth ? (uint8_t*)(base + o_depth) + (size_t)v0 * img : nullptr;
            p.color = p.depth = nullptr;
        } else {
            p.color = (float*)(base + o_color) + (size_t)v0 * 3 * img;
            p.depth = (float*)(base + o_depth) + (size_t)v0 * img;
        }
        p.flags = d_flags;
        p.skipped = h.skipped ? d_skipped : nullptr;
        p.view_group = (M == 1 && h.view_group > 1) ? h.view_group : 1;
        rc = launch_fwd(p, s_run);
        if (rc) return rc;
        GMPI_CUDA_OK(cudaEventRecord(c.ev_free[slot], s_run));
        used[slot] = 1;
        slot ^= 1;
        v0 = v1;
    }
    if (video) {
        GMPI_CUDA_OK(cudaMemcpyAsync(h.video_rgb, base + o_color, (size_t)V * 3 * img, cudaMemcpyDeviceToHost, s_run));
        if (h.video_depth) GMPI_CUDA_OK(cudaMemcpyAsync(h.video_depth, base + o_depth, (size_t)V * img, cudaMemcpyDeviceToHost, s_run));
    } else {
        GMPI_CUDA_OK(cudaMemcpyAsync(h.color, base + o_color, sizeof(float) * (size_t)V * 3 * img, cudaMemcpyDeviceToHost, s_run));
        GMPI_CUDA_OK(cudaMemcpyAsync(h.depth, base + o_depth, sizeof(float) * (size_t)V * img, cudaMemcpyDeviceToHost, s_run));
    }
    GMPI_CUDA_OK(cudaMemcpyAsync(flags_out, d_flags, sizeof(uint32_t), cudaMemcpyDeviceToHost, s_run));
    unsigned long long skipped = 0;
    if (h.skipped) GMPI_CUDA_OK(cudaMemcpyAsync(&skipped, d_skipped, sizeof(skipped), cudaMemcpyDeviceToHost, s_run));
    GMPI_CUDA_OK(cudaStreamSynchronize(s_run));
    GMPI_CUDA_OK(cudaStreamSynchronize(s_copy));
    if (h.skipped) *h.skipped += skipped;      // accumulated into, like the device counter
    return GMPI_OK;
}

static int host_render(const RenderParams& h, uint32_t* flags_out, int device) {
    int rc = check_params(h, false);
    if (rc) return rc;
    if (!flags_out) return fail(GMPI_ERR_INVALID_ARGUMENT, "null output pointer");
    if (h.video_rgb ? false : (!h.color || !h.depth)) return fail(GMPI_ERR_INVALID_ARGUMENT, "null output pointer");
    if (h.n_peers > 0 || h.transmittance) return fail(GMPI_ERR_UNSUPPORTED, "the host entry point renders to host buffers only");
    if (device < 0 || device >= 64) return fail(GMPI_ERR_INVALID_ARGUMENT, "device %d out of range", device);
    for (int v = 0; v + 1 < h.V; ++v)
        if (h.view2mpi[v] > h.view2mpi[v + 1]) return fail(GMPI_ERR_INVALID_ARGUMENT, "views must be MPI-major (sorted view2mpi)");
    for (int v = 0; v < h.V; ++v)
        if (h.view2mpi[v] < 0 || h.view2mpi[v] >= h.M) return fail(GMPI_ERR_INVALID_ARGUMENT, "view2mpi[%d]=%d out of range", v, h.view2mpi[v]);
    GMPI_CUDA_OK(cudaSetDevice(device));
    std::lock_guard<std::mutex> lock(g_host_mutex[device]);
    HostCache& c = g_host_cache[device];
    rc = host_render_locked(c, h, flags_out);
    if (rc != GMPI_OK) {
        // An error may have left asynchronous copies reading the caller's host buffers or rendering from the staging slots:
        // drain both streams before returning so that the caller may free its buffers and the next call starts clean.
        char keep[sizeof(g_err)];
        memcpy(keep, g_err, sizeof(keep));
        if (c.s_run) cudaStreamSynchronize(c.s_run);
        if (c.s_copy) cudaStreamSynchronize(c.s_copy);
        cudaGetLastError();
        memcpy(g_err, keep, sizeof(keep));
    }
    return rc;
}

int gmpi_mpi_render_fwd_host(const float* rgba, const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                             const float* eye, const float* z_dir, float* color, float* depth, uint32_t* flags_out,
                             int M, int V, int N, int Ht, int Wt, int H, int W, uint32_t options, int device) {
    RenderParams h = params_classic(rgba, view2mpi, dhw, ray_dir, eye, z_dir, M, V, N, Ht, Wt, H, W, options);
    h.color = color; h.depth = depth;
    return host_render(h, flags_out, device);
}

int gmpi_mpi_render_host_ex(const gmpi_render_desc* d, int device) {
    int rc = check_desc(d);
    if (rc) return rc;
    return host_render(params_from_desc(d), d->flags, device);
}

}  // extern "C"
