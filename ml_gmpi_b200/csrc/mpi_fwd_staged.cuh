// Forward, TMA-staged persistent variant (the fast path).
//
// One CTA per SM walks (tile, plane) pairs: a 64x30-pixel output tile, planes front to back.  A producer warp computes,
// from the tile's four corner rays, the texel footprint of the tile on the next plane and issues cp.async.bulk.tensor
// copies of exactly that footprint (all four channels, rows in units of 4 issued as a few tall copies, origin aligned to 16 bytes,
// width rounded up to one of five compile-time classes) into a 3-stage shared-memory ring; 15 consumer warps (4 pixels = 2 packed f32x2 pairs per
// thread) take their 16 bilinear taps per pixel and plane from shared memory (a warp reads 32 consecutive x of one row:
// conflict-free while the texel/pixel scale is <= 1) and composite in registers.  TMA's out-of-bounds zero fill implements
// padding_mode="zeros".  Every consumer warp verifies (one vote) that all its taps lie inside the staged box; otherwise it
// takes the generic body, which checks each pixel and samples global memory where the box does not cover it, so results
// never depend on the footprint estimate (arbitrary ray tensors stay correct, only slower).  Tiles are walked full-height
// first, partial bottom tiles last (TileWalk).  DESIGN.md section 4.1 has the measurements and what bounds the kernel.
#pragma once
#include "mpi_common.cuh"
#include "tma_utils.cuh"

namespace gmpi {

#ifndef GMPI_CONS_WARPS
#define GMPI_CONS_WARPS 15   // 15 consumer warps + producer = 16 warps = 4 per scheduler, 128 registers per thread
#endif
#ifndef GMPI_PAIRS
#define GMPI_PAIRS 2         // packed pixel pairs per thread (each pair = x and x+32 of one tile row)
#endif
constexpr int kPairs = GMPI_PAIRS, kPix = 2 * GMPI_PAIRS;
constexpr int kTileW = 64, kTileH = kPairs * GMPI_CONS_WARPS;
constexpr int kConsWarps = GMPI_CONS_WARPS, kConsThreads = kConsWarps * 32, kStagedThreads = kConsThreads + 32;
constexpr int kStages = 3;
constexpr int kRowsPerOp = 4;
constexpr int kMaxBW = 88;
constexpr int kMaxBH = (((kTileH * 5) / 4 + 6 + kRowsPerOp - 1) / kRowsPerOp) * kRowsPerOp;   // footprint rows at scale 1.25 + taps/slack, whole chunks                 // largest staged footprint (texels)
// Box widths are compile-time classes (multiples of 8: row pitch 4*bw = 0 mod 32 banks) so that the consumers'
// sixteen taps are LDS [reg + immediate]; the producer picks the narrowest class that covers the footprint.
constexpr int kMinBW = 56, kBWStep = 8;
constexpr int kNumMaps = (kMaxBW - kMinBW) / kBWStep + 1;
#ifndef GMPI_MAX_PLANES_STAGED
#define GMPI_MAX_PLANES_STAGED 512
#endif
#ifndef GMPI_CTAS_PER_SM
#define GMPI_CTAS_PER_SM 1
#endif
constexpr int kMaxPlanesStaged = GMPI_MAX_PLANES_STAGED;   // plane-constant table: 32 B per plane in shared memory
constexpr int kCtasPerSm = GMPI_CTAS_PER_SM;
constexpr int kStageFloats = kMaxBW * kMaxBH * 4;
constexpr size_t kStagedSmem = (size_t)kStages * kStageFloats * 4 + (size_t)kMaxPlanesStaged * 32;
// Factored forward: box widths 64 and 96 only.  Its boxes are [row][3][bw] (colour) and [row][bw] (alpha): row pitches of 3 bw and
// bw words, and only a pitch that is a multiple of the 32 banks keeps a warp whose 32 taps straddle two texture rows (any rotated
// view) at one wavefront per LDS -- the expanded box [row][4][bw] has that for every bw % 8 == 0.  Measured with 56..88-wide
// boxes (profiles/r02_fwdfact_ncu.txt): 121 M bank-conflict wavefronts per launch against 57 M expanded, kernel 16 % slower.
constexpr int kWideBW = 96;
constexpr int kWideStageFloats = kWideBW * kMaxBH * 4;
constexpr size_t kStagedSmemWide = (size_t)kStages * kWideStageFloats * 4 + (size_t)kMaxPlanesStaged * 32;
static_assert(kStagedSmemWide + 1024 <= 227 * 1024, "wide factored ring must fit one SM");

struct TmaMaps {
    CUtensorMap m[kNumMaps];      // expanded rgba [M*N][4][Ht][Wt] as (x, channel, y, plane), box {bw, 4, 4 rows, 1}
    CUtensorMap m8[kNumMaps], m16[kNumMaps], m32[kNumMaps];   // the same with 8-, 16- and 32-row boxes (see staged_producer: a
                                                              // footprint of r 4-row chunks goes out as the binary digits of r)
    // factored MPI: shared colour [M][3][Ht][Wt] as (x, channel, y, mpi), box {bw, 3, the ring's kColourCopyRows, 1}; the last
    // plane's own colour (torgba_sep_background) likewise; per-plane alpha [M*N][Ht][Wt] as (x, y, plane), box {bw, box height, 1}
    CUtensorMap rgb[kNumMaps], bg[kNumMaps], a[kNumMaps];
    CUtensorMap t;      // backward only: saved transmittance [V*N][H][W], box {64, 24, 1} (the backward's tile)
};

// per-stage header written by the producer before it arms the full barrier
struct __align__(16) StageMeta {
    int cx, cy;            // box origin (texel coordinates of smem element [0][.][0]) + kFloorMagicBits: bits(x + 1.5*2^23, rounded
                           // down) - cx is floor(x) relative to the box
    int rows2;             // staged rows - 2: a footprint with north-west tap (rx, ry) fits iff 0<=rx<=bw-2, 0<=ry<=rows-2
    int sel;               // bits 0-7 staged width (row pitch = 4*bw floats), bits 8-9 mode (0 staged, 1 nothing under the
                           // tile, 2 sample from global, 3 end of tile: early ray termination, see kModeEnd; the kSkip forward
                           // reads bits 8-10, 4 = empty box, see kModeEmpty), bits 16-20 width
                           // class for the packed fast body, ONE-HOT (a chain of single-bit tests, most frequent first, is
                           // shorter than a jump table), or 0 (not usable: mode != 0, or plane constants outside the
                           // exact-division range)
};
// Early ray termination (the kCut forward, inference only): after every plane each active consumer warp ORs "some pixel of mine
// still has T >= stop_transmittance" into the stage's vote word.  Before the producer reuses a stage it has waited for every
// consumer's release of the plane kStages earlier; if that plane's vote is zero the whole tile is below the threshold, and
// instead of the next plane the producer publishes a header with this mode (no copies, no tx bytes).  Consumers finish the
// planes in flight, see it in the generic body, release the stage and go to the epilogue.  The producer alone decides, so the
// ring stays in lockstep and the result does not depend on timing.
constexpr int kModeEnd = 3;
// Empty-space skipping (the kSkip forward, inference only): the producer tests the occupancy bits (one per 8x8 texels, see
// gmpi_mpi_occupancy) of exactly the box it would stage, width class x staged rows clipped to the texture.  If none is set, every
// alpha in the box is within the threshold of 0, and it publishes the box's header with this mode instead: no copies, no tx
// bytes.  A consumer warp whose taps all lie in that box composites nothing for the plane (a = 0 leaves colour, depth and T
// unchanged, bit for bit); a warp with a tap outside it, or with rays outside the fast range, takes the generic body and samples
// the plane from global memory.  Only mode-0 boxes of planes whose constants allow the packed fast body become empty.  The mode
// field is 3 bits wide in this kernel only.
constexpr int kModeEmpty = 4;

// ---- packed dual-fp32 arithmetic (sm_100 FFMA2/FADD2/FMUL2): one issue slot for two pixels, IEEE rn per element ----
typedef float2 f2;
__device__ __forceinline__ f2 splat(float a) { return make_float2(a, a); }
// Inline PTX, not the __fmul2_rn/__fadd2_rn intrinsics: the compiler contracts those into one FFMA2 (observed: texel
// coordinates off by a few ulp), which breaks the reference's separately rounded mul-then-add.  asm blocks cannot be fused.
__device__ __forceinline__ unsigned long long f2_bits(f2 a) { return *reinterpret_cast<unsigned long long*>(&a); }
__device__ __forceinline__ f2 bits_f2(unsigned long long v) { return *reinterpret_cast<f2*>(&v); }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
__device__ __forceinline__ f2 add2(f2 a, f2 b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)), "l"(f2_bits(c)));
    return bits_f2(r);
}
// floor() without the XU pipe: t = x + 1.5*2^23 rounded toward -inf has floor(x) in its mantissa (exact for |x| < 2^22):
// floor as float = t - 1.5*2^23, floor as int = bits(t) - 0x4b400000.  Anything out of range (huge, inf, NaN) yields an
// integer far outside any staged box, so the unsigned box test rejects it.
__device__ __forceinline__ f2 add2_rm(f2 a, f2 b) {
    unsigned long long r;
    asm("add.rm.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f2_bits(a)), "l"(f2_bits(b)));
    return bits_f2(r);
}
constexpr float kFloorMagic = 12582912.0f;        // 1.5 * 2^23
constexpr int kFloorMagicBits = 0x4b400000;
constexpr int kSelSlow = 0;     // class field is one-hot (bit 16 + class); 0 = packed fast body not usable

// a / b correctly rounded with y = RN(1/b), nb = -b (div_by_rcp, two pixels at once)
__device__ __forceinline__ f2 div2_by_rcp(f2 a, f2 nb, f2 y) {
    const f2 q0 = mul2(a, y);
    const f2 r = fma2(q0, nb, a);
    return fma2(r, y, q0);
}

// A thread's four pixels as two pairs: pair P = (x = lane, x = lane + 32) on tile row 2*warp + P.
struct RayPairs {
    f2 rx2[kPairs], ry2[kPairs];   // 2*ray_x, 2*ray_y
    f2 nrz[kPairs], yrz[kPairs];   // -ray_z, RN(1/ray_z)
};
struct CoordPairs {
    f2 ix[kPairs], iy[kPairs], sc[kPairs];
};

// Texel coordinates on one plane, exact-division fast form; op order of plane_coord (mpi.py:74-90 + unnormalize).
template <bool kAlignCorners>
__device__ __forceinline__ void coords_pairs(const PlaneConst& pc, const RayPairs& rp, f2 ex2, f2 ey2, f2 hsx, f2 hsy, float fWt,
                                             float fHt, CoordPairs& c) {
    const f2 zd = splat(pc.z_diff), ypw = splat(pc.ypw), yph = splat(pc.yph), npw = splat(-pc.pw), nph = splat(-pc.ph);
    const f2 one = splat(1.0f);
#pragma unroll
    for (int P = 0; P < kPairs; ++P) {
        const f2 sq = div2_by_rcp(zd, rp.nrz[P], rp.yrz[P]);                 // scale = z_diff / ray_z
        // 2*(e_x + ray_x*scale): mul, THEN add (two roundings, mpi.py:79).  Scalar on purpose: ptxas fuses
        // mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (seen in SASS even with --fmad=false), which is not the reference's
        // arithmetic; the scalar __fmul_rn/__fadd_rn intrinsics are never contracted.  (Writing the add as fma(p, 1, e) does not
        // help either: ptxas folds the multiplication by one and contracts again -- caught by the output checksum, round 2.)
        const f2 X2 = make_float2(__fadd_rn(ex2.x, __fmul_rn(rp.rx2[P].x, sq.x)), __fadd_rn(ex2.y, __fmul_rn(rp.rx2[P].y, sq.y)));
        const f2 Y2 = make_float2(__fadd_rn(ey2.x, __fmul_rn(rp.ry2[P].x, sq.x)), __fadd_rn(ey2.y, __fmul_rn(rp.ry2[P].y, sq.y)));
        f2 u = div2_by_rcp(X2, npw, ypw);                                    // (2x) / width
        f2 v = div2_by_rcp(Y2, nph, yph);
        if (kAlignCorners) {
            c.ix[P] = mul2(add2(u, one), hsx);                               // (u+1) * ((Wt-1)/2)
            c.iy[P] = mul2(add2(v, one), hsy);
        } else {
            if (u.x >= -1.0f && u.x <= 1.0f) u.x = __fmul_rn(u.x, 0.95f);
            if (u.y >= -1.0f && u.y <= 1.0f) u.y = __fmul_rn(u.y, 0.95f);
            if (v.x >= -1.0f && v.x <= 1.0f) v.x = __fmul_rn(v.x, 0.95f);
            if (v.y >= -1.0f && v.y <= 1.0f) v.y = __fmul_rn(v.y, 0.95f);
            const f2 half = splat(0.5f), m1 = splat(-1.0f);
            c.ix[P] = mul2(add2(mul2(add2(u, one), splat(fWt)), m1), half);  // ((u+1)*W - 1) / 2
            c.iy[P] = mul2(add2(mul2(add2(v, one), splat(fHt)), m1), half);
        }
        c.sc[P] = sq;
    }
}

// Sample + composite the four pixels from a staged box of compile-time width BW.  Returns false (and changes nothing)
// if any of the four footprints is not inside the box.
// AOFF == 0: expanded stage [row][4 channels][BW].  AOFF > 0 (factored MPI): colour box [row][3][BW] at the stage base and
// the alpha box [row][BW] AOFF floats further on.
template <int BW, int AOFF = 0>
__device__ __forceinline__ bool sample_pairs(const float* __restrict__ sb, int cx, int cy, int rows2, const CoordPairs& c,
                                             f2 (&T)[kPairs], f2 (&cr)[kPairs], f2 (&cg)[kPairs], f2 (&cb)[kPairs], f2 (&cws)[kPairs]) {
    constexpr int RP = AOFF ? 3 * BW : 4 * BW;       // colour row pitch
    constexpr int AP = AOFF ? BW : 4 * BW;           // alpha row pitch
    constexpr int A0 = AOFF ? AOFF : 3 * BW;         // alpha offset from the colour index (factored: separate box)
    const f2 m1 = splat(-1.0f), one = splat(1.0f);
    f2 fx0[kPairs], fy0[kPairs];
    int ia[kPairs], ib[kPairs], ja[kPairs], jb[kPairs];
    bool inbox = true;
    const f2 magic = splat(kFloorMagic), nmagic = splat(-kFloorMagic);
#pragma unroll
    for (int P = 0; P < kPairs; ++P) {
        const f2 tx = add2_rm(c.ix[P], magic), ty = add2_rm(c.iy[P], magic);         // floor without the XU pipe
        fx0[P] = add2(tx, nmagic);                                    // floor as float (exact)
        fy0[P] = add2(ty, nmagic);
        const int rxa = __float_as_int(tx.x) - cx, rxb = __float_as_int(tx.y) - cx;   // floor - box origin, as integers
        const int rya = __float_as_int(ty.x) - cy, ryb = __float_as_int(ty.y) - cy;
        inbox = inbox && (unsigned)rxa <= (unsigned)(BW - 2) && (unsigned)rxb <= (unsigned)(BW - 2) &&
                (unsigned)rya <= (unsigned)rows2 && (unsigned)ryb <= (unsigned)rows2;
        ia[P] = rya * RP + rxa;                                       // [row][channel][x], compile-time pitch
        ib[P] = ryb * RP + rxb;
        if (AOFF) { ja[P] = rya * AP + rxa + A0; jb[P] = ryb * AP + rxb + A0; }   // alpha taps (separate box)
    }
    if (!__all_sync(0xffffffffu, inbox)) return false;   // warp-uniform, so the caller's fallback needs no reconvergence scaffolding
#pragma unroll
    for (int P = 0; P < kPairs; ++P) {
        const f2 wx1 = fma2(fx0[P], m1, c.ix[P]), wy1 = fma2(fy0[P], m1, c.iy[P]);   // fractional parts (exact)
        const f2 wy0 = fma2(wy1, m1, one);
        const f2 w11 = mul2(wx1, wy1), w10 = fma2(w11, m1, wy1), w01 = fma2(w11, m1, wx1), w00 = fma2(w01, m1, wy0);
        const float* ta = sb + ia[P];
        const float* tb = sb + ib[P];
#define GMPI_TAP(ch)                                                                                           \
    fma2(make_float2(ta[RP + ch * BW + 1], tb[RP + ch * BW + 1]), w11,                                         \
         fma2(make_float2(ta[RP + ch * BW], tb[RP + ch * BW]), w10,                                            \
              fma2(make_float2(ta[ch * BW + 1], tb[ch * BW + 1]), w01, mul2(make_float2(ta[ch * BW], tb[ch * BW]), w00))))
        const f2 r = GMPI_TAP(0), g = GMPI_TAP(1), b = GMPI_TAP(2);
        f2 a;
        if (AOFF == 0) {
            a = GMPI_TAP(3);
        } else {
            const float* aa = sb + ja[P];
            const float* ab = sb + jb[P];
            a = fma2(make_float2(aa[AP + 1], ab[AP + 1]), w11,
                     fma2(make_float2(aa[AP], ab[AP]), w10, fma2(make_float2(aa[1], ab[1]), w01, mul2(make_float2(aa[0], ab[0]), w00))));
        }
#undef GMPI_TAP
        const f2 w = mul2(a, T[P]);                     // mpi.py:423
        cr[P] = fma2(w, r, cr[P]);                      // mpi.py:430
        cg[P] = fma2(w, g, cg[P]);
        cb[P] = fma2(w, b, cb[P]);
        cws[P] = fma2(w, c.sc[P], cws[P]);              // depth_i = scale * (ray . z_dir), mpi.py:150
        T[P] = fma2(w, m1, T[P]);   // T(1-a); the reference's +1e-10 changes any later weight by < 1e-10 absolute
    }
    return true;
}

// The box test of sample_pairs alone, with a run-time width (an empty box, kModeEmpty, has no taps to take): true iff the four
// bilinear footprints of every pixel of the warp lie inside the box of width bw2 + 2 and rows2 + 2 rows at (cx, cy).
__device__ __forceinline__ bool taps_in_box(const CoordPairs& c, int cx, int cy, int bw2, int rows2) {
    const f2 magic = splat(kFloorMagic);
    bool inbox = true;
#pragma unroll
    for (int P = 0; P < kPairs; ++P) {
        const f2 tx = add2_rm(c.ix[P], magic), ty = add2_rm(c.iy[P], magic);
        const int rxa = __float_as_int(tx.x) - cx, rxb = __float_as_int(tx.y) - cx;
        const int rya = __float_as_int(ty.x) - cy, ryb = __float_as_int(ty.y) - cy;
        inbox = inbox && (unsigned)rxa <= (unsigned)bw2 && (unsigned)rxb <= (unsigned)bw2 && (unsigned)rya <= (unsigned)rows2 &&
                (unsigned)ryb <= (unsigned)rows2;
    }
    return __all_sync(0xffffffffu, inbox);
}

// Rare path (a ray whose footprint is not in the staged box): sample the plane from global memory.  Out of line so
// that it does not cost registers in the hot loop.
// Expanded MPI: ONE base pointer crosses the call.  (Passing the four channel pointers of PlaneChans instead -- 8 registers that
// are live only inside the rare branch -- still shifted the register allocation of the hot loop: -3.8 % frames/s, bisected on
// the GPU in round 2.  The factored instantiation, which needs them, is a separate template instance.)
__device__ __noinline__ float4 sample_plane_direct(const float* __restrict__ plane, int Ht, int Wt, float ix, float iy) {
    const size_t tex = (size_t)Ht * Wt;
    const Taps tp = make_taps(ix, iy, Ht, Wt);
    return make_float4(tap4(plane, tp), tap4(plane + tex, tp), tap4(plane + 2 * tex, tp), tap4(plane + 3 * tex, tp));
}
__device__ __noinline__ float4 sample_chans_direct(const PlaneChans pl, int Ht, int Wt, float ix, float iy) {
    const Taps tp = make_taps(ix, iy, Ht, Wt);
    return make_float4(tap4(pl.c[0], tp), tap4(pl.c[1], tp), tap4(pl.c[2], tp), tap4(pl.c[3], tp));
}
// generic-path sample of plane i of MPI m: the instantiation decides which form crosses the call
template <bool kFactored>
__device__ __forceinline__ float4 sample_plane_any(const RenderParams& p, const float* plane, int m, int i, size_t tex, float ix, float iy) {
    if (kFactored) return sample_chans_direct(plane_chans(p, m, i, tex), p.Ht, p.Wt, ix, iy);
    return sample_plane_direct(plane, p.Ht, p.Wt, ix, iy);
}

__device__ __forceinline__ void consumer_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kConsThreads) : "memory"); }

// Tile order of the persistent grid (producer and consumers walk the same sequence): every full-height tile of every view
// first, round-robin over the CTAs; then the partial bottom-row tiles (H % kTileH valid rows), dealt only to the CTAs that
// got one full tile fewer.  Warps whose rows lie outside the image only keep the ring protocol going, so a partial tile
// costs a fraction of a full one and fills the last, incomplete round of the grid instead of stretching it
// (96 planes, 1024^2 x 4 views on 148 SMs: 16 -> 15 tile-times).
struct TileXY { int v, px0, py0; };
struct TileWalk {
    int tiles_x, full_rows, full_per_view, n_full, n_part;
    int cta, grid;               // blockIdx.x, gridDim.x (members so that the host-side test hook runs the same code)
    int n1, p_start, p_step;     // this CTA: number of full tiles; first partial tile and stride (p_step == 0: none)
    int tile_h;                  // tile height in pixels (forward: kTileH = 30, backward: 24)
    int group;                   // views per MPI when consecutive views share one (1: order tiles view by view).  With
                                 // group > 1 the views of a group are the FASTEST index: the CTAs running at the same time
                                 // work on the same tile position of different views of one MPI, i.e. on (nearly) the same
                                 // texels, which then come from L2 instead of HBM (video render: 120 views of one MPI)
    // (lives in shared memory, filled by one thread: it is read once per tile and must not cost registers in the plane loop)
    __host__ __device__ __forceinline__ void init(int tiles_x_, int H, int V, int cta_, int grid_, int tile_h_ = kTileH, int group_ = 1) {
        tiles_x = tiles_x_;
        cta = cta_; grid = grid_;
        tile_h = tile_h_;
        group = (group_ > 1 && V % group_ == 0) ? group_ : 1;
        full_rows = H / tile_h;
        full_per_view = tiles_x * full_rows;
        n_full = full_per_view * V;
        n_part = (H % tile_h) ? tiles_x * V : 0;
        const int b = cta, G = grid, r = n_full % G;
        n1 = b < n_full ? (n_full - b + G - 1) / G : 0;
        if (r == 0) { p_start = b; p_step = G; }
        else if (b >= r) { p_start = b - r; p_step = G - r; }
        else { p_start = 0; p_step = 0; }
    }
    // index t of a sequence of `per_view` positions x V views -> (view, position): view-major, or group-minor
    __host__ __device__ __forceinline__ void split(int t, int per_view, int& v, int& pos) const {
        if (group == 1) { v = t / per_view; pos = t - v * per_view; return; }
        const int per_group = per_view * group, g = t / per_group, rem = t - g * per_group;
        pos = rem / group;
        v = g * group + (rem - pos * group);
    }
    // j-th tile of this CTA; false when done
    __host__ __device__ __forceinline__ bool at(int j, TileXY& r) const {
        int pos;
        if (j < n1) {
            split(cta + j * grid, full_per_view, r.v, pos);
            r.px0 = (pos % tiles_x) * kTileW; r.py0 = (pos / tiles_x) * tile_h;
            return true;
        }
        if (p_step == 0) return false;
        const int u = p_start + (j - n1) * p_step;
        if (u >= n_part) return false;
        split(u, tiles_x, r.v, pos);
        r.px0 = pos * kTileW; r.py0 = full_rows * tile_h;
        return true;
    }
};

// A consumer warp without a single row inside the image: hand every stage of this tile straight back to the producer (kCut: up to
// and including an end-of-tile header; such a warp does not vote).  kModeMask: the width of the header's mode field.
template <bool kCut = false, int kModeMask = 3>
__device__ __forceinline__ void consumer_idle_tile(uint64_t* s_full, uint64_t* s_empty, int N, int lane, int& c_stage, uint32_t& c_phase,
                                                   const StageMeta* s_meta = nullptr) {
    for (int i = 0; i < N; ++i) {
        const int s = c_stage;
        const uint32_t ph = c_phase;
        if (++c_stage == kStages) { c_stage = 0; c_phase ^= 1u; }
        mbar_wait(&s_full[s], ph);
        bool end = false;
        if constexpr (kCut) end = ((s_meta[s].sel >> 8) & kModeMask) == kModeEnd;
        __syncwarp();
        mbar_arrive_if(&s_empty[s], lane == 0);
        if (end) break;
    }
}

// Producer warp, shared by the forward (front-to-back) and backward (back-to-front) kernels: for every (tile, plane) of
// this CTA, estimate the tile's texel footprint from its four corner rays, pick the narrowest box class, publish the stage
// header and issue the TMA copies.
// Ring geometry of a kernel: tile height, ring depth, the largest staged box and what a stage holds.
struct FwdRing {
    static constexpr int kTileRows = kTileH, kRingStages = kStages, kBoxMaxH = kMaxBH;
    static constexpr int kPlaneFloats = kStageFloats;      // floats of one staged plane box
    static constexpr int kStride = kStageFloats;           // floats per ring stage
    static constexpr bool kReverse = false;                // planes front to back; no transmittance box
#ifndef GMPI_FWD_SLEEP
#define GMPI_FWD_SLEEP 0      // measured: sleeping between polls costs the forward 1 % (the 3-stage ring wants its producer prompt)
#endif
    static constexpr bool kSleepPolls = GMPI_FWD_SLEEP != 0;   // producer sleeps between polls of a full ring (see mbar_wait_sleep)
    static constexpr bool kWideFact = false;
    static constexpr bool kBinaryCopies = true;            // expanded MPI: copies of 32/16/8/4 rows (see staged_producer)
    static constexpr int kColourCopyRows = kMaxBH;         // factored MPI (only with GMPI_FWD_WIDE_FACT=0): one colour copy
};
#ifndef GMPI_FWD_WIDE_FACT
#define GMPI_FWD_WIDE_FACT 1
#endif
static_assert(kMaxBH % 2 == 0 && kMaxBH / kRowsPerOp < 16, "half-height colour copies; binary digits of the chunk count");
struct FwdRingWide {      // the factored forward's ring: 64- or 96-wide boxes (see kWideBW)
    static constexpr int kTileRows = kTileH, kRingStages = kStages, kBoxMaxH = kMaxBH;
    static constexpr int kPlaneFloats = kWideStageFloats, kStride = kWideStageFloats;
    static constexpr bool kReverse = false;
    static constexpr bool kSleepPolls = GMPI_FWD_SLEEP != 0;
    static constexpr bool kWideFact = true;
    static constexpr bool kBinaryCopies = true;
    // factored MPI: colour box = 2 copies of 22 rows.  A copy lands at row offset r * 3 * bw * 4 bytes, which must be a multiple
    // of 128 (TMA destination alignment): any r for bw = 64 / 96.
    static constexpr int kColourCopyRows = kMaxBH / 2;
};
// factored MPI: the colour box [row][3][bw] starts the stage, the alpha box [row][bw] follows after 3/4 of the stage

// kFact: factored MPI (compile time: a run-time test of p.alpha in this loop cost the forward 1 %, the producer's per-stage latency
// being on the critical path of a three-stage ring).
// The expanded forward's copies of one stage: the footprint's n_chunks 4-row chunks as the binary digits of n_chunks.  Lane 0..3
// owns the digit 8, 4, 2, 1: returns the copy's height in chunks (0: this lane issues nothing) and, in `before`, the chunks
// covered by the taller copies, i.e. where this copy starts.  (Host-evaluable: gmpi_debug_copy_plan, tests/test_tile_walk.py.)
__host__ __device__ __forceinline__ int binary_copy_of_lane(int n_chunks, int lane, int& before) {
    const int bit = 3 - lane;
    before = (n_chunks >> (bit + 1)) << (bit + 1);
    return ((n_chunks >> bit) & 1) << bit;
}

struct NoPacer { static constexpr bool kActive = false; };      // the forward's producer has no side job

// Pacer: an optional side job of the producer warp (the backward's gradient zeroing): before_tile(mpi) ahead of a tile's first
// copy; new_stage() then chunk() between the polls of the wait for a free ring stage (chunk() returns false when there is nothing
// to do); at_end() after the last tile.
// kCut (forward only): early ray termination, see kModeEnd.  s_vote[kStages] are the stages' vote words; `skipped` (nullable)
// accumulates the pixel-planes of the tiles it cuts short.
// kSkip (forward only): empty-space skipping, see kModeEmpty.  occ is the occupancy map of the MPI ([M][N][ceil(Ht/8)][ceil(Wt/512)]
// words); `skipped_empty` (nullable) accumulates the in-image pixels of a tile times the planes published empty.
template <bool kAlignCorners, class Ring, bool kFact, class Pacer, bool kCut = false, bool kSkip = false>
__device__ __forceinline__ void staged_producer(const RenderParams& p, const TmaMaps& maps, float* s_buf, StageMeta* s_meta,
                                            uint64_t* s_full, uint64_t* s_empty, const TileWalk* s_walk, int lane, Pacer& pacer,
                                            uint32_t* s_vote = nullptr, unsigned long long* skipped = nullptr,
                                            const uint64_t* __restrict__ occ = nullptr, unsigned long long* skipped_empty = nullptr) {
    static_assert(!(kSkip && Ring::kReverse), "empty-space skipping is a forward-only mode");
    // the words a box can touch: lane = 2 * (block row - first) + (word - first); a box spans at most 2 words of 64 blocks
    static_assert((Ring::kBoxMaxH + 7) / 8 + 1 <= 16 && kWideBW / 8 + 1 <= 64, "a staged box spans <= 16 block rows x 2 words");
    const int occ_wy = (p.Ht + 7) >> 3, occ_wx = (p.Wt + 511) >> 9;      // words per plane: block rows x words per row
    constexpr bool kReverse = Ring::kReverse;
    constexpr int kStride = Ring::kStride;      // floats per ring stage
    constexpr int kTileH = Ring::kTileRows, kStages = Ring::kRingStages, kMaxBH = Ring::kBoxMaxH, kStageFloats = Ring::kPlaneFloats;
    constexpr uint32_t kTBytes = kReverse ? (uint32_t)(kTileW * kTileH * 4) : 0u;
    const int Ht = p.Ht, Wt = p.Wt, N = p.N;
    const float fWt = (float)Wt, fHt = (float)Ht;
    const float hsx = 0.5f * (float)(Wt - 1), hsy = 0.5f * (float)(Ht - 1);
    const size_t img = (size_t)p.H * p.W;
    if (lane < kNumMaps) {
        if (kFact) { tma_prefetch_desc(&maps.rgb[lane]); tma_prefetch_desc(&maps.a[lane]); }
        else { tma_prefetch_desc(&maps.m[lane]); tma_prefetch_desc(&maps.m8[lane]); tma_prefetch_desc(&maps.m16[lane]); tma_prefetch_desc(&maps.m32[lane]); }
    }
    int p_stage = 0;
    uint32_t p_phase = 0;
    TileXY txy;
    for (int j = 0; s_walk->at(j, txy); ++j) {
        const int v = txy.v, px0 = txy.px0, py0 = txy.py0;
        const int m = __ldg(p.view2mpi + v);
        if constexpr (Pacer::kActive) pacer.before_tile(m);
        float ev[3], zd[3];
        load_eye_z(p, v, ev, zd);
        // the four corner pixels of the tile (replicated over the warp), clamped into the image
        const int cx = min(px0 + ((lane & 1) ? kTileW - 1 : 0), p.W - 1);
        const int cy = min(py0 + ((lane & 2) ? kTileH - 1 : 0), p.H - 1);
        float crx, cry, crz;
        load_ray(p, v, cx, cy, img, crx, cry, crz);
        const RayConst rc = make_ray_const(crx, cry, crz, ev, zd);
        unsigned n_empty = 0;       // kSkip: planes of this tile published empty
        for (int ii = 0; ii < N; ++ii) {
            const int i = kReverse ? N - 1 - ii : ii;
            const int s = p_stage;
            const uint32_t ph = p_phase;
            if (++p_stage == kStages) { p_stage = 0; p_phase ^= 1u; }
            const PlaneConst pc = make_plane_const(p.dhw + ((size_t)m * N + i) * 3, ev[2]);
            const TexCoord tc = plane_coord<kAlignCorners>(pc, rc, hsx, hsy, fWt, fHt);
            // footprint of the tile = bounding box of the corner coordinates (the pixel -> texel map is projective,
            // hence monotone along image rows and columns), +-1 texel of slack for rounding
            const bool finite = fabsf(tc.ix) < 1e9f && fabsf(tc.iy) < 1e9f;
            const bool all_finite = __all_sync(0xffffffffu, finite);
            const int fx = finite ? (int)floorf(tc.ix) : 0, fy = finite ? (int)floorf(tc.iy) : 0;
            const int xmin = __reduce_min_sync(0xffffffffu, fx), xmax = __reduce_max_sync(0xffffffffu, fx);
            const int ymin = __reduce_min_sync(0xffffffffu, fy), ymax = __reduce_max_sync(0xffffffffu, fy);
            // TMA needs a 16-byte aligned start in the innermost dimension: the box origin is a multiple of 4 texels
            const int bx0 = ((xmin - 1) >> 2) << 2, by0 = ymin - 1;
            const int need_w = xmax - bx0 + 3, need_h = ymax - ymin + 4;      // +1 east/south tap, +-1 slack
            int mode = 0;
            constexpr bool kWide = kFact && Ring::kWideFact;
            constexpr int kBoxMaxW = kWide ? kWideBW : kMaxBW;
            if (!all_finite || need_w > kBoxMaxW || ((need_h + kRowsPerOp - 1) / kRowsPerOp) * kRowsPerOp > kMaxBH) mode = 2;   // would not fit a ring stage
            else if (bx0 > Wt - 1 || bx0 + need_w - 1 < 0 || by0 > Ht - 1 || by0 + need_h - 1 < 0) mode = 1;
            // width class k (tensor-map slot, one-hot bit 16 + k of the header); wide rings: slot 1 = 64, slot 4 = kWideBW
            const int k = mode != 0 ? 0 : kWide ? (need_w <= 64 ? 1 : 4) : max(0, (need_w - kMinBW + kBWStep - 1) / kBWStep);
            const int bw = (kWide && k == 4) ? kWideBW : kMinBW + k * kBWStep;
            int n_ops = mode == 0 ? (need_h + kRowsPerOp - 1) / kRowsPerOp : 0;
            const int rows = n_ops * kRowsPerOp;
            uint64_t occ_w = 0;     // kSkip: this lane's occupancy word of the box, masked to the box's blocks
            if constexpr (kSkip) {
                // Issued before the wait for a free stage, consumed after it: the load is off the ring's critical path.
                const int x0 = max(bx0, 0), x1 = min(bx0 + bw, Wt) - 1;      // the published box, clipped to the texture
                const int y0 = max(by0, 0), y1 = min(by0 + rows, Ht) - 1;
                const int br = (y0 >> 3) + (lane >> 1), bxl = x0 >> 3, bxh = x1 >> 3, wx = (bxl >> 6) + (lane & 1);
                if (mode == 0 && x0 <= x1 && y0 <= y1 && br <= (y1 >> 3) && wx <= (bxh >> 6)) {
                    const int lo = max(bxl - 64 * wx, 0), hi = min(bxh - 64 * wx, 63);
                    occ_w = __ldg(occ + ((size_t)(m * N + i) * occ_wy + br) * occ_wx + wx) & ((~0ull >> (63 - hi)) & (~0ull << lo));
                }
                // ... and it hits L1: a box drifts by a few texels from plane to plane, so the words of plane i + kOccAhead around this
                // box are fetched now.  (Without it a prompt producer waits a full L2 round trip per stage: -25 % on a white-noise MPI,
                // where nothing is empty, and no gain where almost everything is.)
                if (mode == 0 && x0 <= x1 && y0 <= y1) {
                    constexpr int kOccAhead = 4;
                    const int ia = min(i + kOccAhead, N - 1);
                    asm volatile("prefetch.global.L1 [%0];" ::"l"(occ + ((size_t)(m * N + ia) * occ_wy + min(br, occ_wy - 1)) * occ_wx +
                                                                     min(wx, occ_wx - 1)));
                }
            }
            if constexpr (Pacer::kActive) {      // the side job fills the wait for a free stage, a few stores between polls
                pacer.new_stage();
                while (!mbar_try_wait(&s_empty[s], ph ^ 1))
                    if (!pacer.chunk()) __nanosleep(96);
            } else if (Ring::kSleepPolls) {
                mbar_wait_sleep(&s_empty[s], ph ^ 1);
            } else {
                mbar_wait(&s_empty[s], ph ^ 1);
            }
            if constexpr (kCut) {
                // every consumer has released plane ii - kStages of this tile, so its vote is complete (lane 0 reads it: the
                // decision must be warp-uniform, and lane 0 clears the word below)
                const uint32_t vote = __shfl_sync(0xffffffffu, lane == 0 ? *(volatile uint32_t*)&s_vote[s] : 0u, 0);
                if (ii >= kStages && vote == 0) {
                    if (lane == 0) {
                        StageMeta mt;
                        mt.cx = mt.cy = mt.rows2 = 0;
                        mt.sel = kModeEnd << 8;
                        s_meta[s] = mt;
                        mbar_arrive(&s_full[s]);
                        if (skipped) {
                            const int tile_pix = min(kTileW, p.W - px0) * min(kTileH, p.H - py0);
                            atomicAdd(skipped, (unsigned long long)(N - ii) * (unsigned long long)tile_pix);
                        }
                    }
                    __syncwarp();
                    break;
                }
                if (lane == 0) s_vote[s] = 0u;      // published below with the header (the arrive releases both)
            }
            if constexpr (kSkip) {
                // nothing above the threshold in the box; and the plane constants are in the exact-division range, where the
                // consumers' packed coordinates (their box test) are bit-exact -- the same condition as the class bits
                if (mode == 0 && pc.fast != 0.0f && !__any_sync(0xffffffffu, occ_w != 0)) {
                    mode = kModeEmpty;
                    n_ops = 0;
                    ++n_empty;
                }
            }
            if (lane == 0) {
                StageMeta mt;
                mt.cx = kFloorMagicBits + bx0; mt.cy = kFloorMagicBits + by0;
                mt.rows2 = rows - 2;
                mt.sel = bw | (mode << 8) | ((mode == 0 && pc.fast != 0.0f ? (1 << k) : kSelSlow) << 16);
                s_meta[s] = mt;
                // bytes the copies of this stage will deliver (a box counts whole, zero-filled parts included)
                const uint32_t tx = (uint32_t)((kFact ? kMaxBH : rows) * bw * 16);
                if (n_ops > 0 || kTBytes) mbar_arrive_expect_tx(&s_full[s], (n_ops > 0 ? tx : 0u) + kTBytes);
                else mbar_arrive(&s_full[s]);
                if (kReverse)   // the tile's saved transmittance for this plane rides in the same stage
                    tma_load_3d(s_buf + (size_t)s * kStride + kStageFloats, &maps.t, &s_full[s], px0, py0, v * N + i);
            }
            __syncwarp();
            // Few, tall copies.  UTMALDG takes uniform operands, so the lanes of a warp issue their copies ONE AFTER ANOTHER: with a
            // 4-row copy per lane (9-11 per stage, twice that for the factored MPI) the producer was the bottleneck of its own ring
            // (profiles/README.md, round 2: factored forward 1.61 -> 1.41 ms with three copies per stage).
            if (n_ops > 0) {
                float* stage = s_buf + (size_t)s * kStride;
                if (kFact) {
                    // factored MPI: the colour box (shared image, or the last plane's own) as two or three copies that tile the
                    // ring's box height, the alpha box as one copy of the full height.  Rows beyond the footprint are fetched and never
                    // read: the colour image is shared by all planes and comes from L2, alpha is a quarter of the bytes.
                    constexpr int kCR = Ring::kColourCopyRows;      // (a copy's destination must be 128-byte aligned, see the rings)
                    static_assert(kMaxBH % kCR == 0, "colour copies tile the box");
                    const CUtensorMap* cmap = (p.bg_rgb && i == N - 1) ? &maps.bg[k] : &maps.rgb[k];
                    if (lane < kMaxBH / kCR) tma_load_4d(stage + (size_t)lane * kCR * 3 * bw, cmap, &s_full[s], bx0, 0, by0 + lane * kCR, m);
                    if (lane == 31) tma_load_3d(stage + (kStageFloats / 4) * 3, &maps.a[k], &s_full[s], bx0, by0, m * N + i);
                } else if (!Ring::kBinaryCopies) {
                    // expanded MPI, backward: one 4-row copy per lane (measured: taller copies make its 2-stage ring 0.5 % slower)
                    if (lane < n_ops)
                        tma_load_4d(stage + (size_t)lane * kRowsPerOp * 4 * bw, &maps.m[k], &s_full[s], bx0, 0, by0 + lane * kRowsPerOp, m * N + i);
                } else if (lane < 4) {
                    // expanded MPI, forward (HBM-bound: no over-fetch): the n_ops 4-row chunks go out as the binary digits of n_ops,
                    // one copy of 32, 16, 8 and 4 rows each where the digit is set -- at most three copies for up to 44 rows (-1.1 %)
                    int before;
                    const int h = binary_copy_of_lane(n_ops, lane, before);
                    if (h) {
                        const CUtensorMap* mp = h == 8 ? &maps.m32[k] : h == 4 ? &maps.m16[k] : h == 2 ? &maps.m8[k] : &maps.m[k];
                        tma_load_4d(stage + (size_t)before * kRowsPerOp * 4 * bw, mp, &s_full[s], bx0, 0, by0 + before * kRowsPerOp, m * N + i);
                    }
                }
            }
        }
        if constexpr (kSkip) {
            if (skipped_empty && n_empty && lane == 0)
                atomicAdd(skipped_empty, (unsigned long long)n_empty * (unsigned long long)(min(kTileW, p.W - px0) * min(kTileH, p.H - py0)));
        }
    }
    if constexpr (Pacer::kActive) pacer.at_end();
}

// 4x4 transpose inside every quad of lanes (4 q .. 4 q + 3): on entry lane k of a quad holds a[c] = M[k][c], on return
// a[t] = M[t][k].  Two butterfly steps, four shuffles.
__device__ __forceinline__ void quad_transpose(float (&a)[4], int lane) {
    const bool hi2 = (lane & 2) != 0, hi1 = (lane & 1) != 0;
    {   // exchange 2x2 blocks with lane ^ 2
        const float s0 = hi2 ? a[0] : a[2], s1 = hi2 ? a[1] : a[3];
        const float r0 = __shfl_xor_sync(0xffffffffu, s0, 2), r1 = __shfl_xor_sync(0xffffffffu, s1, 2);
        if (hi2) { a[0] = r0; a[1] = r1; } else { a[2] = r0; a[3] = r1; }
    }
    {   // exchange inside the 2x2 blocks with lane ^ 1
        const float s0 = hi1 ? a[0] : a[1], s1 = hi1 ? a[2] : a[3];
        const float r0 = __shfl_xor_sync(0xffffffffu, s0, 1), r1 = __shfl_xor_sync(0xffffffffu, s1, 1);
        if (hi1) { a[0] = r0; a[2] = r1; } else { a[1] = r0; a[3] = r1; }
    }
}

// Epilogue of one consumer warp: rows py, py + 1 of the tile, 64 pixels each; out[q] = (R, G, B, depth) of pixel
// (px0 + lane + 32 (q & 1), py + (q >> 1)).  Three destinations:
//   * uint8 video frames (HWC colour + normalised depth, render_video.py:118-126) when video_rgb is set;
//   * float4 stores after a quad transpose (lane k of a quad ends up with channel k of four consecutive x): 4 x STG.128 per
//     thread instead of 16 x STG.32 -- and 4 per peer in the fused all-gather, or 4 in total through a multicast address;
//   * the scalar store_pixel path for odd widths / unaligned outputs.
// Epilogue of one consumer warp, one pixel set at a time: o = (R, G, B, depth) of pixel (pxb + lane, py) of view v; all 32 lanes
// call this (the quad transpose shuffles).  Destinations:
//   * float4 stores after a quad transpose (lane k of a quad ends up with channel k of four consecutive x): 4 x STG.128 per
//     thread and tile instead of 16 x STG.32 -- and 4 per peer in the fused all-gather, or 4 in total through a multicast address;
//   * store_pixel for odd widths / unaligned outputs and for the uint8 video frames (render_video.py:118-126).
// (Collecting the four pixel sets in a [4][4] array first costs the plane loop 8 instructions per iteration through register
// pressure -- measured: -5 % frames/s -- so each set is stored as soon as it is formed.)
__device__ __forceinline__ void store_tile_pixels(const RenderParams& p, int v, size_t img, int pxb, int py, int lane, float (&o)[4]) {
    if (p.options & kOptVec4Stores) {      // (never set together with the video outputs)
        quad_transpose(o, lane);               // lane k of a quad now holds channel k of four consecutive x
        const int k = lane & 3, px = pxb + 4 * (lane >> 2);
        if (px >= p.W || py >= p.H) return;     // W % 4 == 0: a quad is inside or outside as a whole
        const float4 val = make_float4(o[0], o[1], o[2], o[3]);
        const size_t pix = (size_t)py * p.W + px;
        if (p.n_peers > 0) {
            const size_t fo = ((size_t)(p.frame_offset + v) * 4 + k) * img + pix;
            for (int r = 0; r < p.n_peers; ++r) *reinterpret_cast<float4*>(p.peer_frames[r] + fo) = val;
        } else {
            float* dst = k < 3 ? p.color + ((size_t)v * 3 + k) * img + pix : p.depth + (size_t)v * img + pix;
            *reinterpret_cast<float4*>(dst) = val;
        }
        return;
    }
    const int px = pxb + lane;
    if (px >= p.W || py >= p.H) return;
    store_pixel(p, v, img, (size_t)py * p.W + px, o[0], o[1], o[2], o[3]);
}

template <bool kFactored>
using FwdRingFor = typename std::conditional<kFactored && GMPI_FWD_WIDE_FACT != 0, FwdRingWide, FwdRing>::type;

// The staged forward, body of the kernels below.  kCut: early ray termination at T < tau (never with kEmitT); s_vote [kStages]
// and `skipped` (nullable) as in staged_producer.  kSkip: empty-space skipping (never with kEmitT); occ and `skipped_empty`
// (nullable) as in staged_producer.  With kCut == kSkip == false the extra arguments are unused and the code is that of the
// kernel before either existed.
template <bool kAlignCorners, bool kEmitT, bool kFactored, bool kCut, bool kSkip = false>
__device__ __forceinline__ void fwd_staged_body(const RenderParams& p, const TmaMaps& maps, const int tiles_x, const int tiles_y,
                                                float tau, uint32_t* s_vote, unsigned long long* skipped,
                                                const uint64_t* occ = nullptr, unsigned long long* skipped_empty = nullptr) {
    static_assert(!(kCut && kEmitT), "the training forward saves every T: no termination");
    static_assert(!(kSkip && kEmitT), "the training forward is exact: no empty-space skipping");
    constexpr int kModeMask = kSkip ? 7 : 3;      // the header's mode field: 3 bits with kModeEmpty
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* s_buf = reinterpret_cast<float*>(smem_raw);   // the ring starts the dynamic segment (1024-byte aligned)
    using Ring = FwdRingFor<kFactored>;
    constexpr int kRingFloats = Ring::kPlaneFloats;         // floats per ring stage
    constexpr int kAOff = kFactored ? 3 * (kRingFloats / 4) : 0;      // factored: alpha box behind the colour box
    PlaneConst* s_pc = reinterpret_cast<PlaneConst*>(smem_raw + (size_t)kStages * kRingFloats * 4);   // [N] of the current view
    __shared__ StageMeta s_meta[kStages];
    __shared__ __align__(8) uint64_t s_full[kStages], s_empty[kStages];
    __shared__ TileWalk s_walk;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        s_walk.init(tiles_x, p.H, p.V, (int)blockIdx.x, (int)gridDim.x, kTileH, p.view_group);
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&s_full[s], 1);
            mbar_init(&s_empty[s], kConsWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();

    const int Ht = p.Ht, Wt = p.Wt, N = p.N;
    const float fWt = (float)Wt, fHt = (float)Ht;
    float hsx = 0.5f * (float)(Wt - 1), hsy = 0.5f * (float)(Ht - 1);
    // Opaque to the optimiser: otherwise ptxas, short of registers, re-derives these two constants from the kernel parameters in
    // EVERY plane iteration (2 x LDCU + UIADD3 + I2FP + FMUL, the I2FP on the XU pipe behind the tap loads' MIO queue) -- seen
    // in the round-2 profile after unrelated prologue/epilogue changes: +3 % kernel time.
    asm volatile("" : "+f"(hsx), "+f"(hsy));
    int lane_ = lane;
    asm volatile("" : "+r"(lane_));     // likewise: no S2R + LOP3 per plane for the `lane == 0` of the arrive
    const size_t img = (size_t)p.H * p.W;

    if (warp == kConsWarps) {
        NoPacer np;
        if constexpr (kSkip) staged_producer<kAlignCorners, Ring, kFactored, NoPacer, kCut, true>(p, maps, s_buf, s_meta, s_full, s_empty, &s_walk,
                                                                                                 lane, np, s_vote, skipped, occ, skipped_empty);
        else if constexpr (kCut) staged_producer<kAlignCorners, Ring, kFactored, NoPacer, true>(p, maps, s_buf, s_meta, s_full, s_empty, &s_walk, lane, np,
                                                                                               s_vote, skipped);
        else staged_producer<kAlignCorners, Ring, kFactored>(p, maps, s_buf, s_meta, s_full, s_empty, &s_walk, lane, np);
    } else {
        // ================================ consumer warps ================================
        // warp w owns rows kPairs*w .. kPairs*w + kPairs-1 of the tile; a lane owns x = lane and lane+32 on each of them
        const bool check_last = (p.options & GMPI_CHECK_LAST_PLANE) != 0;
        const bool minus1_1 = (p.options & GMPI_COLOR_MINUS1_1) != 0;
        int c_stage = 0;            // ring position of this warp: stage index and mbarrier phase parity
        uint32_t c_phase = 0;
        uint32_t flag = 0;
        if (blockIdx.x == 0) {          // mpi.py:70: every plane distance against view 0's eye
            const float eye0_z = __ldg(p.eye0 + 2);
            for (int j = threadIdx.x; j < p.M * N; j += kConsThreads)
                if (!(__ldg(p.dhw + (size_t)j * 3) >= eye0_z)) flag |= GMPI_FLAG_PLANE_BEHIND_EYE;
        }
        const size_t tex = (size_t)Ht * Wt;
        int v_table = -1;
        TileXY txy;
        for (int j = 0; s_walk.at(j, txy); ++j) {
            const int v = txy.v, px0 = txy.px0, py0 = txy.py0;
            const int m = __ldg(p.view2mpi + v);
            float ev[3], zd[3];
            load_eye_z(p, v, ev, zd);
            if (v != v_table) {          // (view, plane) constants, once per view and CTA
                consumer_bar_sync();     // everyone is done with the previous view's table
                for (int i = threadIdx.x; i < N; i += kConsThreads) s_pc[i] = make_plane_const(p.dhw + ((size_t)m * N + i) * 3, ev[2]);
                consumer_bar_sync();
                v_table = v;
            }
            if (py0 + kPairs * warp >= p.H) {      // warp-uniform: no row of this warp is inside the image
                consumer_idle_tile<kCut, kModeMask>(s_full, s_empty, N, lane, c_stage, c_phase, s_meta);
                continue;
            }
            RayConst rc[kPix];   // scalar copies, only for the generic (rare) body and the epilogue
            RayPairs rp;
            bool rays_fast = (in_safe_range(ev[0]) || ev[0] == 0.0f) && (in_safe_range(ev[1]) || ev[1] == 0.0f);
#pragma unroll
            for (int q = 0; q < kPix; ++q) {
                const int px = min(px0 + lane + 32 * (q & 1), p.W - 1), py = min(py0 + kPairs * warp + (q >> 1), p.H - 1);
                float qx, qy, qz;
                load_ray(p, v, px, py, img, qx, qy, qz);
                rc[q] = make_ray_const(qx, qy, qz, ev, zd);
                rays_fast = rays_fast && rc[q].fast && fabsf(rc[q].rx2) <= 0x1p40f && fabsf(rc[q].ry2) <= 0x1p40f;
            }
#pragma unroll
            for (int P = 0; P < kPairs; ++P) {
                rp.rx2[P] = make_float2(rc[2 * P].rx2, rc[2 * P + 1].rx2);
                rp.ry2[P] = make_float2(rc[2 * P].ry2, rc[2 * P + 1].ry2);
                rp.nrz[P] = make_float2(-rc[2 * P].rz, -rc[2 * P + 1].rz);
                rp.yrz[P] = make_float2(rc[2 * P].yrz, rc[2 * P + 1].yrz);
            }
            const f2 ex2 = splat(rc[0].ex2), ey2 = splat(rc[0].ey2), hsx2 = splat(hsx), hsy2 = splat(hsy);
            // warp-uniform: every ray of this warp is in the range where the reciprocal+FMA division is exact and no
            // coordinate can be NaN, so the per-plane body needs no per-pixel range checks
            const bool warp_fast = __all_sync(0xffffffffu, rays_fast);
            f2 T[kPairs], cr[kPairs], cg[kPairs], cb[kPairs], cws[kPairs];
#pragma unroll
            for (int P = 0; P < kPairs; ++P) { T[P] = splat(1.f); cr[P] = cg[P] = cb[P] = cws[P] = splat(0.f); }
            PlaneConst pc_next = s_pc[0];
            for (int i = 0; i < N; ++i) {
                const int s = c_stage;
                const uint32_t ph = c_phase;
                if (++c_stage == kStages) { c_stage = 0; c_phase ^= 1u; }
                const PlaneConst pcc = pc_next;            // loaded one plane ahead: no shared-memory latency in front of the
                pc_next = s_pc[min(i + 1, N - 1)];         // coordinate chain (+1.3 %)
                CoordPairs cc;
                // Coordinates before the wait.  (Computing plane i+1's coordinates in the shadow of plane i's tap loads was
                // measured twice: -3 to -4 %; warps in their arithmetic phase leave the shared-memory pipe to the others.)
                if (warp_fast) coords_pairs<kAlignCorners>(pcc, rp, ex2, ey2, hsx2, hsy2, fWt, fHt, cc);
                if (kEmitT) {              // training: save T_i (before plane i) for the backward sweep, [V,N,H,W]
                    float* ts = p.transmittance + ((size_t)v * N + i) * img;
#pragma unroll
                    for (int q = 0; q < kPix; ++q) {
                        const int px = px0 + lane + 32 * (q & 1), py = py0 + kPairs * warp + (q >> 1);
                        if (px < p.W && py < p.H) ts[(size_t)py * p.W + px] = (q & 1) ? T[q >> 1].y : T[q >> 1].x;
                    }
                }
                mbar_wait(&s_full[s], ph);
                const StageMeta mt = s_meta[s];
                const float* sb = s_buf + s * kRingFloats;
                const int sel = mt.sel;                  // warp-uniform; the producer already folded mode and plane range in
                bool done = false;
                bool empty = false;
                if constexpr (kSkip) empty = ((sel >> 8) & kModeMask) == kModeEmpty;
                // (exclusive of the tap chain: testing the empty box in front of the chain instead cost the kSkip kernels a spill)
                if (empty) {                             // all taps in the empty box: a = 0, nothing to add
                    if (warp_fast) done = taps_in_box(cc, mt.cx, mt.cy, (sel & 0xff) - 2, mt.rows2);
                } else if (warp_fast) {
                    if (Ring::kWideFact) {               // factored: two widths, both with bank-aligned row pitches
                        if (sel & (1 << 20)) done = sample_pairs<kWideBW, kAOff>(sb, mt.cx, mt.cy, mt.rows2, cc, T, cr, cg, cb, cws);
                        else if (sel & (1 << 17)) done = sample_pairs<64, kAOff>(sb, mt.cx, mt.cy, mt.rows2, cc, T, cr, cg, cb, cws);
                    } else {                             // most frequent classes first (FFHQ poses: 72 > 64 > 80 >> 56, 88)
                        if (sel & (1 << 18)) done = sample_pairs<72, kAOff>(sb, mt.cx, mt.cy, mt.rows2, cc, T, cr, cg, cb, cws);
                        else if (sel & (1 << 17)) done = sample_pairs<64, kAOff>(sb, mt.cx, mt.cy, mt.rows2, cc, T, cr, cg, cb, cws);
                        else if (sel & (1 << 19)) done = sample_pairs<80, kAOff>(sb, mt.cx, mt.cy, mt.rows2, cc, T, cr, cg, cb, cws);
                        else if (sel & (1 << 16)) done = sample_pairs<56, kAOff>(sb, mt.cx, mt.cy, mt.rows2, cc, T, cr, cg, cb, cws);
                        else if (sel & (1 << 20)) done = sample_pairs<88, kAOff>(sb, mt.cx, mt.cy, mt.rows2, cc, T, cr, cg, cb, cws);
                    }
                }
                if (!done) {
                    // ---- generic body: per-pixel range / box checks, direct sampling when not staged ----
                    // (kModeEmpty: nothing is staged, mode != 0 sends every pixel to global memory)
                    const int bw = mt.sel & 0xff, mode = (mt.sel >> 8) & kModeMask, bw4 = 4 * bw;
                    if constexpr (kCut) {
                        if (mode == kModeEnd) {          // the producer cut the tile short: release the stage, go to the epilogue
                            __syncwarp();
                            mbar_arrive_if(&s_empty[s], lane_ == 0);
                            break;
                        }
                    }
                    const float fbw2 = (float)(bw - 2), fbh2 = (float)mt.rows2;
                    const float fbx0 = (float)(mt.cx - kFloorMagicBits), fby0 = (float)(mt.cy - kFloorMagicBits);
                    const float* plane = kFactored ? nullptr : p.rgba + ((size_t)m * N + i) * 4 * tex;
                    float* Ts = reinterpret_cast<float*>(T);
                    float* crs = reinterpret_cast<float*>(cr);
                    float* cgs = reinterpret_cast<float*>(cg);
                    float* cbs = reinterpret_cast<float*>(cb);
                    float* cwss = reinterpret_cast<float*>(cws);
#pragma unroll
                    for (int q = 0; q < kPix; ++q) {
                        RayConst rg = rc[q];
                        rg.fast = false;            // rare path: plain IEEE divisions, no per-plane range checks in the hot loop
                        const TexCoord tc = plane_coord<kAlignCorners>(pcc, rg, hsx, hsy, fWt, fHt);
                        const float fx = floorf(tc.ix), fy = floorf(tc.iy);
                        const float rxx = fx - fbx0, ryy = fy - fby0;
                        float r, g, b, a;
                        if (!kFactored && mode == 0 && rxx >= 0.0f && rxx <= fbw2 && ryy >= 0.0f && ryy <= fbh2) {
                            const float wx1 = tc.ix - fx, wy1 = tc.iy - fy;
                            const float wx0 = 1.0f - wx1, wy0 = 1.0f - wy1;
                            const float w00 = wx0 * wy0, w01 = wx1 * wy0, w10 = wx0 * wy1, w11 = wx1 * wy1;
                            const float* t0 = sb + ((int)ryy * bw4 + (int)rxx);
                            const float* t1 = t0 + bw4;
                            r = fmaf(t1[1], w11, fmaf(t1[0], w10, fmaf(t0[1], w01, t0[0] * w00)));
                            g = fmaf(t1[bw + 1], w11, fmaf(t1[bw], w10, fmaf(t0[bw + 1], w01, t0[bw] * w00)));
                            b = fmaf(t1[2 * bw + 1], w11, fmaf(t1[2 * bw], w10, fmaf(t0[2 * bw + 1], w01, t0[2 * bw] * w00)));
                            a = fmaf(t1[3 * bw + 1], w11, fmaf(t1[3 * bw], w10, fmaf(t0[3 * bw + 1], w01, t0[3 * bw] * w00)));
                        } else if (coord_hits(tc.ix, tc.iy, fWt, fHt)) {   // mode 1 ("nothing under the tile") is only the
                            // producer's corner-ray estimate: every pixel is still tested on its own
                            const float4 sv = sample_plane_any<kFactored>(p, plane, m, i, tex, tc.ix, tc.iy);
                            r = sv.x; g = sv.y; b = sv.z; a = sv.w;
                        } else {
                            continue;   // no texel under this ray on this plane: contributes exactly nothing
                        }
                        const float w = a * Ts[q];
                        crs[q] = fmaf(w, r, crs[q]);
                        cgs[q] = fmaf(w, g, cgs[q]);
                        cbs[q] = fmaf(w, b, cbs[q]);
                        cwss[q] = fmaf(w, tc.scale, cwss[q]);
                        Ts[q] -= w;
                    }
                }
                if constexpr (kCut) {         // the vote (see kModeEnd): one ballot, one shared OR, before the release
                    bool alive = false;
#pragma unroll
                    for (int P = 0; P < kPairs; ++P) alive = alive || T[P].x >= tau || T[P].y >= tau;
                    if (__any_sync(0xffffffffu, alive) && lane_ == 0) atomicOr(&s_vote[s], 1u);
                }
                __syncwarp();
                mbar_arrive_if(&s_empty[s], lane_ == 0);    // predicated, no branch
            }
            if (check_last) {     // assert_not_out_of_last_plane, mpi.py:103-109 (once per tile)
                const PlaneConst pcl = s_pc[N - 1];
#pragma unroll
                for (int q = 0; q < kPix; ++q) {
                    RayConst rg = rc[q];
                    rg.fast = false;
                    const TexCoord tc = plane_coord<kAlignCorners>(pcl, rg, hsx, hsy, fWt, fHt);
                    if (!(tc.u >= -1.0f && tc.u <= 1.0f && tc.v >= -1.0f && tc.v <= 1.0f)) flag |= GMPI_FLAG_LAST_PLANE_OOB;
                }
            }
            // ---- epilogue: the warp's 2 rows x 64 pixels, (R, G, B, depth) per pixel, one pixel set at a time ----
#pragma unroll
            for (int q = 0; q < kPix; ++q) {
                float o[4];
                o[0] = (q & 1) ? cr[q >> 1].y : cr[q >> 1].x; o[1] = (q & 1) ? cg[q >> 1].y : cg[q >> 1].x;
                o[2] = (q & 1) ? cb[q >> 1].y : cb[q >> 1].x;
                o[3] = ((q & 1) ? cws[q >> 1].y : cws[q >> 1].x) * rc[q].dz;
                if (minus1_1) {
                    o[0] = fmaf(2.0f, o[0], -1.0f); o[1] = fmaf(2.0f, o[1], -1.0f); o[2] = fmaf(2.0f, o[2], -1.0f);
                }
                store_tile_pixels(p, v, img, px0 + 32 * (q & 1), py0 + kPairs * warp + (q >> 1), lane, o);
            }
        }
        if (flag) atomicOr(p.flags, flag);
    }
}

template <bool kAlignCorners, bool kEmitT, bool kFactored>
__global__ void __launch_bounds__(kStagedThreads, kCtasPerSm)
mpi_fwd_staged_kernel(const RenderParams p, const __grid_constant__ TmaMaps maps, const int tiles_x, const int tiles_y) {
    fwd_staged_body<kAlignCorners, kEmitT, kFactored, false>(p, maps, tiles_x, tiles_y, 0.0f, nullptr, nullptr);
}

// Inference forward with early ray termination at T < tau (0 < tau < 1); skipped (nullable) accumulates the pixel-planes not
// composited.  Same ring, same epilogues as mpi_fwd_staged_kernel<kAlignCorners, false, kFactored>.
template <bool kAlignCorners, bool kFactored>
__global__ void __launch_bounds__(kStagedThreads, kCtasPerSm)
mpi_fwd_cut_kernel(const RenderParams p, const __grid_constant__ TmaMaps maps, const int tiles_x, const int tiles_y, const float tau,
                   unsigned long long* skipped) {
    __shared__ uint32_t s_vote[kStages];
    fwd_staged_body<kAlignCorners, false, kFactored, true>(p, maps, tiles_x, tiles_y, tau, s_vote, skipped);
}

// Inference forward with empty-space skipping (see kModeEmpty): occupancy is the map of gmpi_mpi_occupancy for the MPI of p;
// empty_pixel_planes (nullable) accumulates the pixel-planes of the boxes published empty.  kCut: together with early ray
// termination (tau, skipped as in mpi_fwd_cut_kernel).  Same ring, same epilogues as mpi_fwd_staged_kernel<kAlignCorners, false,
// kFactored>.
template <bool kAlignCorners, bool kFactored, bool kCut>
__global__ void __launch_bounds__(kStagedThreads, kCtasPerSm)
mpi_fwd_skip_kernel(const RenderParams p, const __grid_constant__ TmaMaps maps, const int tiles_x, const int tiles_y, const float tau,
                    unsigned long long* skipped, const uint64_t* __restrict__ occupancy, unsigned long long* empty_pixel_planes) {
    __shared__ uint32_t s_vote[kStages];
    fwd_staged_body<kAlignCorners, false, kFactored, kCut, true>(p, maps, tiles_x, tiles_y, tau, s_vote, skipped, occupancy,
                                                                 empty_pixel_planes);
}

}  // namespace gmpi
