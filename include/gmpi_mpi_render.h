/*
 * gmpi_mpi_render.h -- C ABI of the B200 (sm_100a) multiplane-image renderer.
 *
 * Drop-in boundary for ONE path of apple/ml-gmpi: the over-composite render of
 * gmpi/core/mpi.py (MPI.forward :308-436 + homography :26-153) as driven by
 * MPIRenderer.render (gmpi/core/mpi_renderer.py:387-469).  The reference has no FFI for this
 * path (it is a chain of ~30 ATen kernels); these entry points are what a binding for it binds.
 * INTEGRATION.md shows the ctypes stub and the two-line patch on the reference side.
 *
 * Conventions
 *   - plain C, plain pointers and sizes; no torch types.  All tensors fp32, contiguous,
 *     row-major, on the CUDA device that is current on the calling thread (except *_host).
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream).  All device
 *     entry points are asynchronous on that stream and allocate nothing.
 *   - return value: GMPI_OK, or an error code with a message available from gmpi_last_error()
 *     (thread-local).  The library never exits the process (the reference calls sys.exit(1) when
 *     rays leave the last plane, mpi.py:122-128; here that is a flag bit).
 *
 * Layouts (names follow the reference)
 *   rgba      [M, N, 4, Ht, Wt]  MPI textures in [0,1], planes ordered near -> far (mpi.py:413)
 *   dhw       [M, N, 3]          per plane: distance, metric height, metric width (mpi.py:59-63)
 *   view2mpi  [V] int32          MPI index of every rendered view.  Replaces the expand+cat of
 *                                mpi.py:334-346 (no copy of the MPI per view); views are
 *                                MPI-major like the reference's concatenation.
 *   ray_dir   [V, 3, H, W]       world-space unit rays per pixel (camera.py:182-211)
 *   eye       [V, 3]             camera position (camera.py:189)
 *   z_dir     [V, 3]             optical axis (camera.py:209)
 *   color     [V, 3, H, W]       composited colour in [0,1] (or 2c-1 if GMPI_COLOR_MINUS1_1)
 *   depth     [V, 1, H, W]       transmittance-weighted z-depth (mpi.py:434)
 *   flags     [1] uint32         OR-ed GMPI_FLAG_* bits (device memory; caller zeroes it)
 */
#ifndef GMPI_MPI_RENDER_H_
#define GMPI_MPI_RENDER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GMPI_ABI_VERSION 2

/* return codes */
#define GMPI_OK 0
#define GMPI_ERR_INVALID_ARGUMENT 1
#define GMPI_ERR_CUDA 2
#define GMPI_ERR_UNSUPPORTED 3

/* flag bits written to *flags: the reference's data-dependent asserts, reported instead of raised */
#define GMPI_FLAG_RGBA_RANGE 1u        /* rgba outside [0,1]            mpi_renderer.py:447-449 */
#define GMPI_FLAG_ALPHA_RANGE 2u       /* alpha outside [0,1]           mpi.py:185-187          */
#define GMPI_FLAG_LAST_PLANE_OOB 4u    /* |u| or |v| > 1 on last plane  mpi.py:103-109,381-395  */
#define GMPI_FLAG_PLANE_BEHIND_EYE 8u  /* distance < z_eye[0]           mpi.py:70-72            */

/* option bits for `options` */
#define GMPI_ALIGN_CORNERS 1u          /* MPI(align_corners=True), configs/gmpi.yml:74          */
#define GMPI_CHECK_LAST_PLANE 2u       /* assert_not_out_of_last_plane, mpi.py:317              */
#define GMPI_COLOR_MINUS1_1 4u         /* fuse "2*color-1" of mpi_renderer.py:467 into the store */
#define GMPI_ZERO_GRAD 8u              /* bwd: zero the gradient buffers on the stream before accumulating */
#define GMPI_U8_ROUND_HALF_UP 16u       /* uint8 epilogue: clamp, x*255+0.5 (torchvision save_image, fid_evaluation.py:125-130)
                                          instead of numpy's truncating astype (render_video.py:119-126) */

int gmpi_abi_version(void);
const char* gmpi_last_error(void);

/* Name of the kernel variant a forward call with these shapes would launch (diagnostics). */
const char* gmpi_mpi_render_fwd_variant(int N, int Ht, int Wt, int H, int W);

/*
 * Which forward/backward kernels a call with these shapes launches: GMPI_PLAN_STAGED (persistent TMA-staged kernels, the fast
 * path) or GMPI_PLAN_DIRECT (one thread per pixel, any shape, several times slower).  *why (nullable) receives the GMPI_WHY_*
 * bits of every reason the staged path is not taken, so a caller can surface the performance cliff instead of finding it in a
 * profile.  rgba may be NULL (alignment unknown: not checked).
 */
#define GMPI_PLAN_DIRECT 1
#define GMPI_PLAN_STAGED 2
#define GMPI_WHY_TEX_WIDTH 1u    /* Wt % 4 != 0: rows are not 16-byte multiples, no tensor map                     */
#define GMPI_WHY_FEW_TILES 2u    /* fewer than 120 tiles of 64x30 pixels over all views: the persistent grid would idle */
#define GMPI_WHY_MANY_PLANES 4u  /* N > 512: the per-view plane-constant table does not fit next to the ring        */
#define GMPI_WHY_ALIGNMENT 8u    /* rgba base not 16-byte aligned                                                   */
#define GMPI_WHY_FORCED 16u      /* gmpi_debug_set_fwd_variant(1)                                                    */
int gmpi_mpi_render_fwd_plan(int V, int N, int Ht, int Wt, int H, int W, const void* rgba, uint32_t* why);

/*
 * Forward: replaces MPI.forward (mpi.py:308-436) for all V views in one launch.
 * Per output pixel the planes are walked front to back; colour, depth and transmittance stay in
 * registers; no [V*N, c, H, W] intermediate is written.
 * Numerics: texel coordinates are bit-identical to the reference's fp32 op sequence.  The transmittance is updated as
 * T <- T - a*T in the TMA-staged kernels and as T <- T*((1-a)+1e-10) (the reference's form, mpi.py:421) in the direct kernels:
 * the two differ by < 1e-10 absolute per plane, far below the fp32 resolution of the outputs; both are within 1e-6 (relative
 * to the largest output) of the reference, and so is the transmittance saved for the backward.  Up to 65535 views per launch
 * on the direct kernels (gmpi_mpi_render_fwd_plan tells which kernel a shape gets); the staged kernels have no such limit.
 */
int gmpi_mpi_render_fwd(const float* rgba, const int32_t* view2mpi, const float* dhw,
                        const float* ray_dir, const float* eye, const float* z_dir,
                        float* color, float* depth, uint32_t* flags,
                        int M, int V, int N, int Ht, int Wt, int H, int W,
                        uint32_t options, void* stream);

/*
 * Forward with the all-gather of frames fused into the epilogue (multi-GPU, SURVEY.md section 8e).  Instead of
 * color/depth, every finished pixel of view v is stored as a packed frame [4,H,W] = (R,G,B,depth) at frame index
 * frame_offset + v of EVERY buffer in peer_frames: a DEVICE array of n_peers base pointers to [F,4,H,W] fp32 buffers,
 * one per rank, peer-mapped over NVLink (e.g. torch symmetric memory, cudaIpc).  The stores are posted writes that overlap
 * the remaining compute; the caller makes them visible with a barrier across ranks after the kernel.  Replaces the
 * render + ncclAllGather pair; the reference has no counterpart (its renderer is single-GPU, gloo barriers only).
 */
int gmpi_mpi_render_fwd_gather(const float* rgba, const int32_t* view2mpi, const float* dhw,
                               const float* ray_dir, const float* eye, const float* z_dir,
                               float* const* peer_frames, int n_peers, int frame_offset, uint32_t* flags,
                               int M, int V, int N, int Ht, int Wt, int H, int W,
                               uint32_t options, void* stream);

/*
 * Backward: d(sum(color*g_color) + sum(depth*g_depth)) / d rgba, what torch autograd produces for
 * MPI.forward (only the sampled rgba carries gradient: mpi.py:65,148 run under no_grad).
 * g_depth may be NULL.  Views of one MPI accumulate into the same g_rgba slab (the `expand` of
 * train.py:733-738).  g_rgba must be zero, or pass GMPI_ZERO_GRAD.
 * If options has GMPI_COLOR_MINUS1_1 the upstream g_color is w.r.t. 2*color-1.
 */
int gmpi_mpi_render_bwd(const float* rgba, const int32_t* view2mpi, const float* dhw,
                        const float* ray_dir, const float* eye, const float* z_dir,
                        const float* g_color, const float* g_depth, float* g_rgba,
                        int M, int V, int N, int Ht, int Wt, int H, int W,
                        uint32_t options, void* stream);

/*
 * Training pair.  gmpi_mpi_render_fwd_train = gmpi_mpi_render_fwd that additionally saves the transmittance in front of
 * every plane, transmittance [V,N,H,W] (T_i = prod_{j<i}(1 - alpha_j), mpi.py:421-423) -- what torch autograd keeps alive as
 * `weights`/`cumprod` tensors, here 4 bytes per (pixel, plane).  gmpi_mpi_render_bwd_saved consumes it: one staged
 * back-to-front sweep instead of the two-pass kernel (falls back to gmpi_mpi_render_bwd for shapes the staged path skips).
 */
int gmpi_mpi_render_fwd_train(const float* rgba, const int32_t* view2mpi, const float* dhw,
                              const float* ray_dir, const float* eye, const float* z_dir,
                              float* color, float* depth, float* transmittance, uint32_t* flags,
                              int M, int V, int N, int Ht, int Wt, int H, int W,
                              uint32_t options, void* stream);
int gmpi_mpi_render_bwd_saved(const float* rgba, const int32_t* view2mpi, const float* dhw,
                              const float* ray_dir, const float* eye, const float* z_dir,
                              const float* transmittance, const float* g_color, const float* g_depth,
                              float* g_rgba, int M, int V, int N, int Ht, int Wt, int H, int W,
                              uint32_t options, void* stream);

/*
 * Descriptor form of the render calls: every optional input/output of the path in one struct, so that the variants below
 * compose (factored MPI x in-kernel rays x video epilogue x fused all-gather x training).  Zero-initialise it, set
 * struct_bytes = sizeof(gmpi_render_desc) and fill what applies; every pointer is DEVICE memory for gmpi_mpi_render_fwd_ex /
 * gmpi_mpi_render_bwd_ex and HOST memory for gmpi_mpi_render_host_ex.
 *
 *   MPI, one of
 *     rgba   [M,N,4,Ht,Wt]                       the expanded stack MPI.forward receives (mpi.py:309)
 *     rgb    [M,3,Ht,Wt] + alpha [M,N,1,Ht,Wt]   the generator's FACTORED output: one colour image shared by all planes and one
 *            (+ bg_rgb [M,3,Ht,Wt], optional)    alpha per plane, before the reference expands and concatenates them
 *                                                (networks_cond_on_pos_enc.py:950-975,984,1313; bg_rgb = the last plane's own
 *                                                colour under torgba_sep_background).  4x fewer HBM / PCIe bytes; output
 *                                                identical to rendering the expanded stack.
 *   camera, one of
 *     ray_dir [V,3,H,W] + eye [V,3] + z_dir [V,3]   the reference's tensors (parity mode: bit-exact texel coordinates)
 *     cam [V,16] = {f0, f1, f2 (the fp64 focal length as three fp32 pieces with f0 + f1 + f2 == focal exactly), pixel-centre
 *                   offset (0.5), R row-major (9), eye (3)}; the principal point is (W/2, H/2) (cam_utils.py:20)
 *                                                fast mode: rays generated in the kernel with camera.py:53-118,182-211's
 *                                                arithmetic (fp64 camera ray -> fp32 -> fp32 rotation); saves the [V,3,H,W]
 *                                                tensor and its upload.  Forward only.
 *   view_group  > 1 when every view_group consecutive views share one MPI (V % view_group == 0): tiles are then ordered so that
 *               concurrently running CTAs work on the same texels (L2 reuse; video render, multi-view search).  0/1 otherwise.
 *   outputs, one of
 *     color [V,3,H,W] + depth [V,1,H,W]          fp32 (2c-1 with GMPI_COLOR_MINUS1_1)
 *     peer_frames / n_peers / frame_offset       fused all-gather, see gmpi_mpi_render_fwd_gather.  A single NVLS multicast
 *                                                address with n_peers = 1 makes the switch replicate the stores.
 *     video_rgb [V,H,W,3] uint8 + video_depth [V,H,W,1] uint8 (optional), depth_near / depth_range
 *                                                the conversion lines of render_video.py:118-126 fused into the store:
 *                                                ((2c-1)+1)/2*255 truncated; clip((d - near)/range, 0, 1)*255 truncated
 *                                                (GMPI_U8_ROUND_HALF_UP: torchvision save_image rounding instead)
 *   transmittance [V,N,H,W]                      training forward: saved for gmpi_mpi_render_bwd_ex
 *   backward: g_color [V,3,H,W], g_depth (nullable), and g_rgba [M,N,4,Ht,Wt]  or  g_rgb [M,3,Ht,Wt] (+ g_bg_rgb) + g_alpha
 *             [M,N,1,Ht,Wt]; zeroed by the callee with GMPI_ZERO_GRAD, else accumulated into
 *   stop_transmittance  tau in [0, 1): early ray termination of the INFERENCE forward (0 = off, the default).
 *               A pixel's colour and depth may drop the contributions of the planes behind the point where its transmittance
 *               T = prod_{j<i}(1 - alpha_j) is already below tau.  Hence every output lies in [full - tau * max(value), full]
 *               (colour in [0,1], and depth; plus fp32 rounding; twice that for 2c-1 colour), a pixel whose T stays >= tau up
 *               to the last plane is bit-identical to the tau = 0 render, and tau = 0 is bit-identical to a descriptor without
 *               the field.  Deterministic: the same inputs give the same bytes and the same skip count.  The staged kernels
 *               stop a 64x30 tile once all its pixels are below tau (a few planes later: the planes already in flight are
 *               composited); the direct kernel stops each pixel on its own.  Rejected (GMPI_ERR_INVALID_ARGUMENT, before any
 *               CUDA call): tau NaN, < 0 or >= 1; tau > 0 together with `transmittance` (the training forward saves every T);
 *               tau > 0 in gmpi_mpi_render_bwd_ex (gradients stay exact).
 *   skipped_pixel_planes  nullable uint64 [1], device memory (host memory for gmpi_mpi_render_host_ex): accumulated into, the
 *               number of (pixel, plane) pairs not composited because of stop_transmittance.  Not zeroed by the callee.
 *   The last two fields were appended without changing GMPI_ABI_VERSION: struct_bytes = offsetof(gmpi_render_desc,
 *   stop_transmittance), the size of the descriptor before them, is still accepted and means both fields absent (tau = 0).
 *   A caller that sets them against an older library gets the struct_bytes error, never a silently exact render.
 */
typedef struct gmpi_render_desc {
    uint32_t struct_bytes;
    uint32_t options;
    int32_t M, V, N, Ht, Wt, H, W;
    int32_t view_group;
    int32_t n_peers, frame_offset;
    float depth_near, depth_range;
    const float* rgba;
    const float* rgb;
    const float* alpha;
    const float* bg_rgb;
    const int32_t* view2mpi;
    const float* dhw;
    const float* ray_dir;
    const float* eye;
    const float* z_dir;
    const float* cam;
    float* color;
    float* depth;
    float* transmittance;
    float* const* peer_frames;
    uint8_t* video_rgb;
    uint8_t* video_depth;
    const float* g_color;
    const float* g_depth;
    float* g_rgba;
    float* g_rgb;
    float* g_bg_rgb;
    float* g_alpha;
    uint32_t* flags;
    void* stream;
    float stop_transmittance;
    uint64_t* skipped_pixel_planes;
} gmpi_render_desc;

/* cudaMemsetAsync(ptr, 0, bytes) on `stream`, for callers that accumulate into their own buffers (no GMPI_ZERO_GRAD).  Note that a
 * memset cannot overlap the staged kernels, on whatever stream (they own every SM: measured, tools/zero_overlap_probe.py). */
int gmpi_mpi_zero_async(void* ptr, size_t bytes, void* stream);

int gmpi_mpi_render_fwd_ex(const gmpi_render_desc* desc);
int gmpi_mpi_render_bwd_ex(const gmpi_render_desc* desc);
/* Host-buffer form (end-to-end entry point, see gmpi_mpi_render_fwd_host): all pointers of *desc are HOST memory, `stream` is
 * ignored, *flags receives the flag word.  Forward only; supports the factored MPI, cam and the video outputs. */
int gmpi_mpi_render_host_ex(const gmpi_render_desc* desc, int device);

/*
 * Empty-space skipping of the INFERENCE forward: planes whose alpha is (near) zero under a whole 64x30 tile are not fetched and
 * not composited.  Two steps on the same stream:
 *
 * gmpi_mpi_occupancy: one bit per 8x8-texel block of every alpha plane, set iff some alpha of the block has !(|alpha| <=
 *   threshold) (so NaN counts as occupied, -0.0 does not).  occupancy [M][N][ceil(Ht/8)][ceil(Wt/512)] uint64 (device memory):
 *   bit b of word w of block row r covers texels x in [8(64w+b), 8(64w+b)+8), y in [8r, 8r+8); texels outside the texture do not
 *   exist and never set a bit.  gmpi_mpi_occupancy_plane_words(Ht, Wt) = ceil(Ht/8) * ceil(Wt/512), the words of one plane (0 for
 *   sizes < 1).  Alpha of plane i of MPI m is read at alpha[m * mpi_stride + i * plane_stride + texel] as in gmpi_mpi_alpha_depth_fwd:
 *   the expanded stack (alpha = rgba + 3*Ht*Wt, plane_stride = 4*Ht*Wt, mpi_stride = N*4*Ht*Wt) or the factored alpha [M,N,1,Ht,Wt]
 *   (plane_stride = Ht*Wt).  Every word is written (no zeroing needed).  A streaming read of the alpha planes only.  Rejected
 *   (GMPI_ERR_INVALID_ARGUMENT, before any CUDA call): threshold NaN, < 0 or >= 1.
 *
 * gmpi_mpi_render_fwd_skip_ex: gmpi_mpi_render_fwd_ex on the same descriptor (every option composes: expanded or factored MPI,
 *   ray_dir or cam, fp32 / 2c-1 / uint8 video outputs, fused gather, view_group, stop_transmittance), except that the staged
 *   kernel may skip a (tile, plane) whose staged box (the footprint estimate of the tile, rounded up to the box the kernel would
 *   fetch) has no bit set in `occupancy`, built for the same MPI tensors.  A warp whose taps all lie in such a box composites
 *   nothing for that plane; any other pixel samples the plane as usual, so results never depend on the footprint estimate.
 *   The direct kernel ignores the map (exact render, nothing counted).
 *   empty_pixel_planes: nullable uint64 [1], device memory: accumulated into (not zeroed), the in-image pixels of each tile times
 *   the planes published empty for it.  Deterministic.
 *   Contract.  For finite inputs, threshold 0 gives output bit-identical to gmpi_mpi_render_fwd_ex with the same descriptor,
 *   including with stop_transmittance > 0: a plane whose taps all have alpha = 0 adds fma(0, x, acc) = acc and leaves T unchanged,
 *   so the termination votes, decisions and count are identical too.  With threshold eps > 0, for MPIs with alpha and colour in
 *   [0, 1] (the range the reference asserts), every output moves by at most N * eps * max(value) plus fp32 rounding (twice that
 *   for 2c-1 colour): skipping plane j changes the composite by T_j * alpha_j * (c_j - C_behind).
 *   Rejected (GMPI_ERR_INVALID_ARGUMENT, before any CUDA call): a NULL occupancy; a non-NULL transmittance (the training forward
 *   stays exact).
 */
size_t gmpi_mpi_occupancy_plane_words(int Ht, int Wt);
int gmpi_mpi_occupancy(const float* alpha, long long mpi_stride, long long plane_stride, int M, int N, int Ht, int Wt, float threshold,
                       uint64_t* occupancy, void* stream);
int gmpi_mpi_render_fwd_skip_ex(const gmpi_render_desc* desc, const uint64_t* occupancy, uint64_t* empty_pixel_planes);

/*
 * LightRenderer (gmpi/core/light_renderer.py), the lighting augmentation applied to the MPI right before the render call in
 * training (train.py:534-541,702-709).  Two streaming kernels replace what the reference materialises:
 *
 * gmpi_mpi_alpha_depth_fwd = LightRenderer.compute_depth (light_renderer.py:82-100): the over-composite of the UN-warped alpha,
 *   depth[m] = sum_i a_i prod_{j<i}(1 - a_j + 1e-10) plane_d[i]  -> depth [M,1,Ht,Wt].  alpha of plane i of MPI m is read at
 *   alpha[m * mpi_stride + i * plane_stride + texel] (strides in floats): the expanded stack (alpha = rgba + 3*Ht*Wt, plane_stride
 *   = 4*Ht*Wt, mpi_stride = N*4*Ht*Wt) or the factored alpha [M,N,1,Ht,Wt] (plane_stride = Ht*Wt).  transmittance [M,N,Ht,Wt] is
 *   optional (training: saved for the backward).  gmpi_mpi_alpha_depth_bwd: d sum(depth * g_depth) / d alpha into g_alpha with its
 *   own strides (e.g. channel 3 of a g_rgba stack).
 * gmpi_mpi_apply_shading_fwd = the last step of LightRenderer.render (light_renderer.py:190-199): out[m,i,c] =
 *   clip(rgba[m,i,c] * shade[m], 0, 1) for the colour channels, alpha copied: the new [M,N,4,Ht,Wt] MPI in one pass.
 *   _bwd: gradients w.r.t. rgba and shade [M,1,Ht,Wt] (torch.clip's closed-interval mask).
 */
int gmpi_mpi_alpha_depth_fwd(const float* alpha, long long mpi_stride, long long plane_stride, const float* plane_d,
                             float* depth, float* transmittance, int M, int N, int Ht, int Wt, void* stream);
int gmpi_mpi_alpha_depth_bwd(const float* alpha, long long mpi_stride, long long plane_stride, const float* plane_d,
                             const float* transmittance, const float* g_depth, float* g_alpha, long long g_mpi_stride,
                             long long g_plane_stride, int M, int N, int Ht, int Wt, void* stream);
int gmpi_mpi_apply_shading_fwd(const float* rgba, const float* shade, float* out, int M, int N, int Ht, int Wt, void* stream);
int gmpi_mpi_apply_shading_bwd(const float* rgba, const float* shade, const float* g_out, float* g_rgba, float* g_shade,
                               int M, int N, int Ht, int Wt, void* stream);

/*
 * Range checks of MPIRenderer.render (mpi_renderer.py:447-449) and MPI.check_shapes
 * (mpi.py:185-187) in one streaming pass: sets GMPI_FLAG_RGBA_RANGE / GMPI_FLAG_ALPHA_RANGE.
 */
int gmpi_mpi_check_range(const float* rgba, int M, int N, int Ht, int Wt, uint32_t* flags,
                         void* stream);

/*
 * Host-buffer forward (end-to-end entry point): all pointers are HOST memory (pinned memory
 * overlaps best).  Copies inputs to `device`, renders, copies colour/depth/flags back and
 * synchronises.  MPIs are streamed through a double-buffered device staging area so the copy of
 * MPI m+1 overlaps the render of MPI m.  *flags_out receives the OR of all flag bits.  The staging buffers, streams and
 * events are cached per device (grow-only) across calls; gmpi_mpi_release_host_cache() frees them.
 */
int gmpi_mpi_render_fwd_host(const float* rgba, const int32_t* view2mpi, const float* dhw,
                             const float* ray_dir, const float* eye, const float* z_dir,
                             float* color, float* depth, uint32_t* flags_out,
                             int M, int V, int N, int Ht, int Wt, int H, int W,
                             uint32_t options, int device);

int gmpi_mpi_release_host_cache(void);

/* Test hook: texel coordinates (ix, iy) of every (view, plane, pixel), out [V,N,2,H,W]; the
 * bit-exact stage of the path (must equal torch's fp32 op sequence, DESIGN.md "coordinates"). */
int gmpi_debug_plane_coords(const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                            const float* eye, float* out, int V, int N, int Ht, int Wt, int H,
                            int W, uint32_t options, void* stream);

/* Test hook: same as gmpi_debug_plane_coords through the staged kernel's packed (f32x2) coordinate code (H*W even). */
int gmpi_debug_plane_coords_packed(const int32_t* view2mpi, const float* dhw, const float* ray_dir,
                                   const float* eye, float* out, int V, int N, int Ht, int Wt, int H,
                                   int W, uint32_t options, void* stream);

/* Test hook: force the forward kernel variant: 0 auto (default), 1 direct-gather, 2 TMA-staged. */
int gmpi_debug_set_fwd_variant(int variant);

/* GMPI_ZERO_GRAD of the staged backward as stream memsets before the kernel (0, default) or inside the kernel, one MPI slab
 * ahead of use (1: correct for any view order, measured 4.5 % slower on B200 -- see mpi_bwd_box.cuh). */
int gmpi_debug_set_bwd_zero(int in_kernel);

/* Test hook (host only): the TMA copies the expanded forward issues for a footprint of n_rows staged rows, as (first row, rows)
 * pairs: the binary digits of n_rows / 4 (copies of 32, 16, 8, 4 rows).  Returns the number of copies. */
int gmpi_debug_copy_plan(int n_rows, int* out_row_rows, int max_copies);

/* Test hook (host only): tile order for a tile height (30 forward, 24 backward) and view grouping (gmpi_render_desc.view_group). */
int gmpi_debug_tile_walk_ex(int H, int W, int V, int tile_h, int view_group, int grid, int cta, int* out_v_px0_py0, int max_tiles);

/* Test hook: the rays the fast mode generates from cam [V,16] -> ray_dir [V,3,H,W] (device memory). */
int gmpi_debug_cam_rays(const float* cam, float* ray_dir, int V, int H, int W, void* stream);

/* Test hook (host only, no GPU work): the persistent kernels' tile order.  Writes the (view, px0, py0) of the tiles that
 * CTA `cta` of a `grid`-CTA launch walks, in order, into out_v_px0_py0[3 * max_tiles]; returns their number (>= 0) or a
 * negative GMPI_ERR_* code.  Tile size: 64 x 30 pixels. */
int gmpi_debug_tile_walk(int H, int W, int V, int grid, int cta, int* out_v_px0_py0, int max_tiles);

/* Test hook: out_fast[i] = the kernels' reciprocal+FMA division a[i]/b[i]; out_ieee[i] = div.rn.f32. */
int gmpi_debug_division(const float* a, const float* b, float* out_fast, float* out_ieee, size_t n,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GMPI_MPI_RENDER_H_ */
