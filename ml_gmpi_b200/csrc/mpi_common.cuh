// Shared device helpers of the MPI render kernels (sm_100a).
//
// The coordinate stage reproduces, bit for bit, the fp32 operation sequence of the reference
// (gmpi/core/mpi.py:74-90 + ATen grid_sampler_unnormalize) because the texel coordinate is
// amplified by (texture size x texel gradient): see DESIGN.md "Coordinates".
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

namespace gmpi {

struct RenderParams {
    const float* rgba;        // [M,N,4,Ht,Wt]
    const int32_t* view2mpi;  // [V]
    const float* dhw;         // [M,N,3]
    const float* ray_dir;     // [V,3,H,W]
    const float* eye;         // [V,3]
    const float* eye0;        // eye of the call's GLOBAL view 0 (mpi.py:70 compares every plane distance with it); == eye
                              // unless a host-side wrapper splits one call into several launches
    const float* z_dir;       // [V,3]
    float* color;             // [V,3,H,W]
    float* depth;             // [V,1,H,W]
    uint32_t* flags;          // [1]
    const float* g_color;     // bwd
    const float* g_depth;     // bwd, nullable
    float* g_rgba;            // bwd
    int M, V, N, Ht, Wt, H, W;
    uint32_t options;
    // fused all-gather (optional): frames [*,4,H,W] (RGB + depth) of view v are stored into every peer's buffer at
    // frame index frame_offset + v instead of color/depth.  peer_frames is a device array of n_peers base pointers.
    float* const* peer_frames;
    int n_peers, frame_offset;
    // training: transmittance before each plane, [V,N,H,W]; written by the forward, read by the staged backward (nullable)
    float* transmittance;
    // fast mode (opt-in): rays generated in the kernel from the pinhole camera of each view instead of read from ray_dir
    // (camera.py:182-211).  cam [V,16] = {focal as three fp32 pieces (exact fp64 sum), pixel-centre offset, R row-major (9), eye (3)}
    const float* cam;
    // video epilogue (opt-in, render_video.py:118-126): uint8 HWC colour [V,H,W,3] and depth [V,H,W,1] instead of color/depth
    uint8_t* video_rgb;
    uint8_t* video_depth;
    float depth_near, depth_range;
    // factored MPI (opt-in, networks_cond_on_pos_enc.py:950-975): shared colour rgb [M,3,Ht,Wt] (+ bg_rgb for the last plane) and
    // per-plane alpha [M,N,1,Ht,Wt] instead of rgba
    const float* rgb;
    const float* bg_rgb;
    const float* alpha;
    float* g_rgb;             // bwd, factored: [M,3,Ht,Wt] (sum over planes 0..N-1, or 0..N-2 when bg_rgb is given)
    float* g_bg_rgb;          // bwd, factored with a separate background: [M,3,Ht,Wt] of the last plane
    float* g_alpha;           // bwd, factored: [M,N,1,Ht,Wt]
    int view_group;           // > 1: every `view_group` consecutive views share one MPI (tile order hint, see TileWalk)
    // staged backward with GMPI_ZERO_GRAD: the kernel zeroes the large gradient buffer itself, one MPI slab ahead of its use
    // (GradZeroPacer, mpi_bwd_box.cuh).  zero_base = g_rgba or g_alpha, zero_slab16 = float4s per MPI, zero_flags[M] = number of
    // CTAs that have zeroed their share of MPI m (zero on entry), zero_rate = warp-wide 512-byte stores per ring stage.
    float4* zero_base;
    unsigned long long zero_slab16;
    unsigned* zero_flags;
    int zero_rate;
    // inference forward (opt-in): early ray termination.  A pixel may drop the planes behind the point where its transmittance
    // fell below stop_transmittance (0 = off); skipped (nullable, device) accumulates the pixel-planes not composited.
    float stop_transmittance;
    unsigned long long* skipped;
};

// The four channel slabs (Ht*Wt floats each) of one (MPI, plane): expanded rgba or the generator's factored form.
struct PlaneChans { const float* c[4]; };
__device__ __forceinline__ PlaneChans plane_chans(const RenderParams& p, int m, int i, size_t tex) {
    PlaneChans pc;
    if (p.alpha) {
        const float* rgb = ((p.bg_rgb && i == p.N - 1) ? p.bg_rgb : p.rgb) + (size_t)m * 3 * tex;
        pc.c[0] = rgb; pc.c[1] = rgb + tex; pc.c[2] = rgb + 2 * tex;
        pc.c[3] = p.alpha + ((size_t)m * p.N + i) * tex;
    } else {
        const float* b = p.rgba + ((size_t)m * p.N + i) * 4 * tex;
        pc.c[0] = b; pc.c[1] = b + tex; pc.c[2] = b + 2 * tex; pc.c[3] = b + 3 * tex;
    }
    return pc;
}
struct GradChans { float* c[4]; };
__device__ __forceinline__ GradChans grad_chans(const RenderParams& p, int m, int i, size_t tex) {
    GradChans gc;
    if (p.g_alpha) {
        float* rgb = ((p.g_bg_rgb && i == p.N - 1) ? p.g_bg_rgb : p.g_rgb) + (size_t)m * 3 * tex;
        gc.c[0] = rgb; gc.c[1] = rgb + tex; gc.c[2] = rgb + 2 * tex;
        gc.c[3] = p.g_alpha + ((size_t)m * p.N + i) * tex;
    } else {
        float* b = p.g_rgba + ((size_t)m * p.N + i) * 4 * tex;
        gc.c[0] = b; gc.c[1] = b + tex; gc.c[2] = b + 2 * tex; gc.c[3] = b + 3 * tex;
    }
    return gc;
}

// internal option bits (above the public GMPI_* bits of include/gmpi_mpi_render.h)
constexpr uint32_t kOptVec4Stores = 1u << 16;   // W % 4 == 0 and all output bases 16-byte aligned: float4 epilogue stores

// Pinhole ray of pixel (px, py) of a view, the arithmetic of ml_gmpi_b200.camera.PinholeCamera (camera.py:53-76,98-118,182-211
// of the reference): camera-space direction in fp64, normalised, rounded to fp32, rotated to world space in fp32.
__device__ __forceinline__ void cam_ray(const float* __restrict__ cam, int px, int py, int H, int W, float& rx, float& ry, float& rz) {
    // the focal length is an fp64 quantity on the host (w / (2 tan(fov/2))): it travels as three fp32 pieces whose exact sum it is
    const double focal = __dadd_rn(__dadd_rn((double)__ldg(cam), (double)__ldg(cam + 1)), (double)__ldg(cam + 2));
    const double off = (double)__ldg(cam + 3), cx = 0.5 * (double)W, cy = 0.5 * (double)H;     // principal point (w/2, h/2), cam_utils.py:20
    const double xs = __ddiv_rn(__dsub_rn(__dadd_rn((double)px, off), cx), focal);      // K^-1 [u v 1], camera.py:63-66
    const double ys = __ddiv_rn(__dsub_rn(__dadd_rn((double)py, off), cy), focal);
    const double nrm = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(xs, xs), __dmul_rn(ys, ys)), 1.0));   // camera.py:98-105
    const float dx = (float)__ddiv_rn(xs, nrm), dy = (float)__ddiv_rn(ys, nrm), dz = (float)__ddiv_rn(1.0, nrm);    // :116-118
    const float* R = cam + 4;
    rx = fmaf(__ldg(R + 2), dz, fmaf(__ldg(R + 1), dy, __ldg(R + 0) * dx));                 // ray_dir = R @ rays, camera.py:201
    ry = fmaf(__ldg(R + 5), dz, fmaf(__ldg(R + 4), dy, __ldg(R + 3) * dx));
    rz = fmaf(__ldg(R + 8), dz, fmaf(__ldg(R + 7), dy, __ldg(R + 6) * dx));
}

// Ray of pixel (px, py) of view v: read from ray_dir (the reference's tensor: parity mode) or generated (fast mode).
__device__ __forceinline__ void load_ray(const RenderParams& p, int v, int px, int py, size_t img, float& rx, float& ry, float& rz) {
    if (p.cam) {
        cam_ray(p.cam + 16 * (size_t)v, px, py, p.H, p.W, rx, ry, rz);
    } else
    {
        const float* rd = p.ray_dir + (size_t)v * 3 * img + (size_t)py * p.W + px;
        rx = __ldg(rd); ry = __ldg(rd + img); rz = __ldg(rd + 2 * img);
    }
}
// eye and optical axis of view v (camera.py:189-190,209)
__device__ __forceinline__ void load_eye_z(const RenderParams& p, int v, float (&ev)[3], float (&zd)[3]) {
    if (p.cam) {
        const float* c = p.cam + 16 * (size_t)v;
        ev[0] = __ldg(c + 13); ev[1] = __ldg(c + 14); ev[2] = __ldg(c + 15);
        zd[0] = __ldg(c + 6); zd[1] = __ldg(c + 9); zd[2] = __ldg(c + 12);     // R[:, 2]
    } else
    {
        ev[0] = __ldg(p.eye + 3 * v); ev[1] = __ldg(p.eye + 3 * v + 1); ev[2] = __ldg(p.eye + 3 * v + 2);
        zd[0] = __ldg(p.z_dir + 3 * v); zd[1] = __ldg(p.z_dir + 3 * v + 1); zd[2] = __ldg(p.z_dir + 3 * v + 2);
    }
}

// uint8 conversions of the reference's consumers.  Truncating: render_video.py:119-126 (numpy astype(uint8)); rounding:
// torchvision save_image(normalize=True, range=(-1,1)) as used by fid_evaluation.py:125-130 (mul(255).add_(0.5).clamp_(0,255)).
__device__ __forceinline__ uint8_t color_to_u8(float img_m11, bool round_half_up) {
    if (round_half_up) {
        const float c = fminf(fmaxf(img_m11, -1.0f), 1.0f);
        const float x = __fadd_rn(__fmul_rn(__fdiv_rn(__fadd_rn(c, 1.0f), 2.0f), 255.0f), 0.5f);
        return (uint8_t)(int)fminf(fmaxf(x, 0.0f), 255.0f);
    }
    return (uint8_t)(int)__fmul_rn(__fmul_rn(__fadd_rn(img_m11, 1.0f), 0.5f), 255.0f);       // (img + 1) / 2.0 * 255
}
__device__ __forceinline__ uint8_t depth_to_u8(float depth, float d_near, float d_range) {
    const float x = __fdiv_rn(__fsub_rn(depth, d_near), d_range);                              // render_video.py:123
    return (uint8_t)(int)__fmul_rn(fminf(fmaxf(x, 0.0f), 1.0f), 255.0f);                         // clip, * 255, astype(uint8)
}

// Store one finished pixel: plain outputs, or the same frame slot of every rank's gather buffer (NVLink peer stores).
__device__ __forceinline__ uint8_t color_to_u8(float img_m11, bool round_half_up);
__device__ __forceinline__ uint8_t depth_to_u8(float depth, float d_near, float d_range);
__device__ __forceinline__ void store_pixel(const RenderParams& p, int v, size_t img, size_t pix, float c0, float c1, float c2, float dep) {
    if (p.video_rgb) {        // uint8 HWC frame (render_video.py:118-126)
        const bool up = (p.options & GMPI_U8_ROUND_HALF_UP) != 0;
        uint8_t* c = p.video_rgb + ((size_t)v * img + pix) * 3;
        c[0] = color_to_u8(c0, up); c[1] = color_to_u8(c1, up); c[2] = color_to_u8(c2, up);
        if (p.video_depth) p.video_depth[(size_t)v * img + pix] = depth_to_u8(dep, p.depth_near, p.depth_range);
    } else if (p.n_peers > 0) {
        const size_t fo = (size_t)(p.frame_offset + v) * 4 * img + pix;
        for (int r = 0; r < p.n_peers; ++r) {
            float* f = p.peer_frames[r] + fo;
            f[0] = c0; f[img] = c1; f[2 * img] = c2; f[3 * img] = dep;
        }
    } else {
        float* co = p.color + (size_t)v * 3 * img + pix;
        co[0] = c0; co[img] = c1; co[2 * img] = c2;
        p.depth[(size_t)v * img + pix] = dep;
    }
}

// Per (view, plane) constants, staged in shared memory once per CTA.
//   a = {z_diff, pw, ph, fast}   b = {rcp(pw), rcp(ph), -, -}
// z_diff = d - e_z (mpi.py:74).  `fast` != 0 when the three divisors/dividends are in the
// exponent range where the FMA-corrected reciprocal division below is provably IEEE-exact.
struct PlaneConst {
    float z_diff, pw, ph, fast;
    float ypw, yph, pad0, pad1;
};

__device__ __forceinline__ bool in_safe_range(float x) {
    const float ax = fabsf(x);
    return ax >= 0x1p-40f && ax <= 0x1p40f;
}

// a / b, correctly rounded, given y = RN(1/b): q0 = RN(a*y); r = a - q0*b (exact in an FMA);
// q = RN(q0 + r*y).  (Markstein's theorem; verified exhaustively over all divisor mantissas
// on the CPU by tools/check_division.c and against __fdiv_rn on the GPU by
// tests/test_gpu_parity.py::test_fast_division_equals_ieee_division.)
__device__ __forceinline__ float div_by_rcp(float a, float b, float y) {
    const float q0 = __fmul_rn(a, y);
    const float r = __fmaf_rn(-q0, b, a);
    return __fmaf_rn(r, y, q0);
}

__device__ __forceinline__ PlaneConst make_plane_const(const float* __restrict__ dhw_plane, float eye_z) {
    PlaneConst c;
    const float d = dhw_plane[0], ph = dhw_plane[1], pw = dhw_plane[2];
    c.z_diff = __fsub_rn(d, eye_z);
    c.pw = pw;
    c.ph = ph;
    c.ypw = __frcp_rn(pw);
    c.yph = __frcp_rn(ph);
    const bool ok = (c.z_diff == 0.0f || in_safe_range(c.z_diff)) && in_safe_range(pw) && in_safe_range(ph);
    c.fast = ok ? 1.0f : 0.0f;
    c.pad0 = c.pad1 = 0.0f;
    return c;
}

// Per-pixel ray constants.
struct RayConst {
    float rx2, ry2;   // 2*ray_x, 2*ray_y  (exact scaling: RN(2a) = 2 RN(a))
    float rz, yrz;    // ray_z and RN(1/ray_z)
    float ex2, ey2;   // 2*eye_x, 2*eye_y
    float dz;         // ray . z_dir   (mpi.py:149)
    bool fast;
};

__device__ __forceinline__ RayConst make_ray_const(float rx, float ry, float rz, const float* e, const float* zd) {
    RayConst r;
    r.rx2 = 2.0f * rx;
    r.ry2 = 2.0f * ry;
    r.rz = rz;
    r.yrz = __frcp_rn(rz);
    r.ex2 = 2.0f * e[0];
    r.ey2 = 2.0f * e[1];
    r.dz = fmaf(rz, zd[2], fmaf(ry, zd[1], rx * zd[0]));
    r.fast = in_safe_range(rz);
    return r;
}

struct TexCoord {
    float ix, iy, scale, u, v;
};

// mpi.py:74-99 + grid_sampler_unnormalize.  Every operation rounds exactly as the reference's
// separate elementwise kernels do (no FMA contraction across reference ops).
template <bool kAlignCorners>
__device__ __forceinline__ TexCoord plane_coord(const PlaneConst& pc, const RayConst& rc, float hsx, float hsy,
                                                float fWt, float fHt) {
    TexCoord t;
    float s, u, v;
    if (pc.fast != 0.0f && rc.fast) {
        s = div_by_rcp(pc.z_diff, rc.rz, rc.yrz);                       // scale = z_diff / ray_z   (:76)
        const float X2 = __fadd_rn(rc.ex2, __fmul_rn(rc.rx2, s));      // 2*(e_x + ray_x*scale)    (:79,:90)
        const float Y2 = __fadd_rn(rc.ey2, __fmul_rn(rc.ry2, s));
        u = div_by_rcp(X2, pc.pw, pc.ypw);                             // u = 2x / width           (:90)
        v = div_by_rcp(Y2, pc.ph, pc.yph);                             // v = 2y / height          (:89)
    } else {
        s = __fdiv_rn(pc.z_diff, rc.rz);
        const float X2 = __fadd_rn(rc.ex2, __fmul_rn(rc.rx2, s));
        const float Y2 = __fadd_rn(rc.ey2, __fmul_rn(rc.ry2, s));
        u = __fdiv_rn(X2, pc.pw);
        v = __fdiv_rn(Y2, pc.ph);
    }
    if (kAlignCorners) {
        // ((u+1)/2)*(size-1) == (u+1)*((size-1)/2): the halving is exact, so both round the same
        // real product (ATen's CPU kernel uses the second form, its CUDA kernel the first).
        t.ix = __fmul_rn(__fadd_rn(u, 1.0f), hsx);
        t.iy = __fmul_rn(__fadd_rn(v, 1.0f), hsy);
    } else {
        if (u >= -1.0f && u <= 1.0f) u = __fmul_rn(u, 0.95f);            // mpi.py:95-99
        if (v >= -1.0f && v <= 1.0f) v = __fmul_rn(v, 0.95f);
        t.ix = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(u, 1.0f), fWt), -1.0f), 0.5f);   // ((u+1)*W-1)/2
        t.iy = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(v, 1.0f), fHt), -1.0f), 0.5f);
    }
    t.scale = s;
    t.u = u;
    t.v = v;
    return t;
}

// Bilinear footprint with zero padding (F.grid_sample(mode="bilinear", padding_mode="zeros")).
// Indices are clamped into the texture and the weight of an out-of-range tap is zeroed, so the
// sixteen loads are unconditional.
struct Taps {
    int o00, o01, o10, o11;      // element offsets inside one channel slab
    float w00, w01, w10, w11;    // nw, ne, sw, se
};

// Requires ix in (-1, Wt) and iy in (-1, Ht) (caller tests; anything else contributes zero).
__device__ __forceinline__ Taps make_taps(float ix, float iy, int Ht, int Wt) {
    Taps t;
    const float fx0 = floorf(ix), fy0 = floorf(iy);
    const float wx1 = ix - fx0, wy1 = iy - fy0;        // exact
    float wx0 = 1.0f - wx1, wy0 = 1.0f - wy1;          // == (x0+1) - ix rounded
    float wx1m = wx1, wy1m = wy1;
    const int x0 = (int)fx0, y0 = (int)fy0;
    if (x0 < 0) wx0 = 0.0f;
    if (y0 < 0) wy0 = 0.0f;
    if (x0 + 1 > Wt - 1) wx1m = 0.0f;
    if (y0 + 1 > Ht - 1) wy1m = 0.0f;
    const int x0c = max(x0, 0), y0c = max(y0, 0);
    const int x1c = min(x0 + 1, Wt - 1), y1c = min(y0 + 1, Ht - 1);
    t.o00 = y0c * Wt + x0c;
    t.o01 = y0c * Wt + x1c;
    t.o10 = y1c * Wt + x0c;
    t.o11 = y1c * Wt + x1c;
    t.w00 = wx0 * wy0;
    t.w01 = wx1m * wy0;
    t.w10 = wx0 * wy1m;
    t.w11 = wx1m * wy1m;
    return t;
}

__device__ __forceinline__ bool coord_hits(float ix, float iy, float fWt, float fHt) {
    return ix > -1.0f && ix < fWt && iy > -1.0f && iy < fHt;   // false for NaN
}

__device__ __forceinline__ float tap4(const float* __restrict__ ch, const Taps& t) {
    const float a = __ldg(ch + t.o00), b = __ldg(ch + t.o01), c = __ldg(ch + t.o10), d = __ldg(ch + t.o11);
    return fmaf(d, t.w11, fmaf(c, t.w10, fmaf(b, t.w01, a * t.w00)));
}

}  // namespace gmpi
