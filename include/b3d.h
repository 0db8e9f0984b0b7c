/*
 * libb3d — C ABI of the B200-native hot path of NikolaZubic/2dimageto3dmodel.
 *
 * The reference has no FFI of its own: its boundary is the Python call surface
 * (SURVEY.md §8b).  Every entry point below is what a reference-side binding for
 * that call would wrap; the reference function it replaces is cited as
 * /root/reference/code/<file>:<lines>.  INTEGRATION.md shows the ctypes stubs.
 *
 * Conventions (all entry points)
 *   - plain pointers + sizes, no torch types; every pointer is DEVICE memory,
 *     contiguous, fp32 unless stated, base pointers 16-byte aligned;
 *   - the caller owns every buffer (inputs, outputs, workspaces); the library never
 *     allocates or frees persistent device memory;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no
 *     internal synchronisation;
 *   - return 0 on success, a negative B3D_E* code otherwise; b3d_last_error()
 *     returns a thread-local message.  Nothing throws or exits across the ABI;
 *   - stateless and re-entrant.
 */
#ifndef B3D_H_
#define B3D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B3D_API __attribute__((visibility("default")))
#else
#define B3D_API
#endif

#define B3D_OK 0
#define B3D_EINVAL (-1)  /* bad argument (null pointer, negative size, unsupported shape) */
#define B3D_EALIGN (-2)  /* pointer not 16-byte aligned */
#define B3D_ECUDA (-3)   /* CUDA runtime error (message in b3d_last_error) */

/* semantics switch of the point-cloud path, SURVEY.md App. A */
#define B3D_MODE_REFERENCE 0 /* "R": the reference as written (quirks D3,D4,D5,D10 kept) */
#define B3D_MODE_PAPER 1     /* "P": paper-intended */

B3D_API const char* b3d_last_error(void);
B3D_API int b3d_version(void);
/* ';'-joined names of the kernel template instances launched by the calling thread's most recent convolution
 * entry point (b3d_conv2d_tf32 / _flat_tf32 / _wgrad_tf32 / _thin_*), e.g. "conv_tf32_persistent<256,4,0,1>":
 * the parity tests assert WHICH variant they exercised, so dispatch drift cannot silently un-test a kernel. */
B3D_API const char* b3d_last_variant(void);
/* number of kernels this library has launched in the calling process (bench.py's gpu_launches) */
B3D_API uint64_t b3d_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Point-cloud "effective loss" path
 *   EffectiveLossFunction.forward            utils/effective_loss_function.py:58-81
 * ------------------------------------------------------------------------------------------ */

/* Rotate by the normalised quaternion, perspective-project, map to grid coordinates, and sort the
 * in-bounds points of every sample by the (8 x 16)-cell bin of their base voxel (y, x).
 *   PointsQuaternionsRotator.rotate_points   quaternions/points_quaternions.py:41-81
 *   QuaternionOperations.quaternion_multiplication / _conjugate   quaternions/operations.py:68-97,120-136
 *   CameraUtilities.transformation_3d_coord_to_camera_coord       camera/coordinate_system_transformation.py:20-39
 *   TrilinearInterpolation.get_grid / get_point_cloud_object_borders  utils/trilinear_interpolation.py:17-35
 * points [B,N,3] (columns z,y,x), quat [B,4] (w,x,y,z); fov / cam_dist are the reference's
 * field_of_view = 1.875 and camera_view_distance = 2.0 (effective_loss_function.py:69-70).
 * pg        [B,N,4]  out: grid coords (gz,gy,gx) = (V-1)(c+0.5) and flag 1.0/0.0 = in bounds
 * coords    [B,N,3]  out, nullable: camera coords c
 * base      [B,N,3]  out, nullable, int32: floor(g) — the reference's index buffer for corner (0,0,0)
 *                    (trilinear_interpolation.py:47-52); bit-exact target
 * inb       [B,N]    out, nullable, uint8: in-bounds mask (bit-exact target)
 * sorted    [B,N,4]  out, nullable: (gz,gy,gx, bits(point index)) of the in-bounds points, bin-sorted
 * bin_start [B, b3d_pc_bin_count(V)+1] out, int32 (with sorted): start of every bin in `sorted`      */
B3D_API int b3d_pc_bin_count(int V);
/* 1 when the silhouette kernels stage the bin records through shared memory with cp.async.bulk (the TMA's 1-D bulk copy,
 * mbarrier byte-count completion; the first stages are in flight while the patch is zero-filled), 0 when they read them with
 * plain loads.  Process-wide, read once: environment B3D_PC_TMA=0/1 overrides the built-in default. */
B3D_API int b3d_pc_tma_staging(void);
/* Host-only view of that staging (CPU tests): records per ring stage, and the contiguous runs of `sorted` that bulk copies
 * bring in for chunk `chunk` of the record sequence "bins [bx_lo, bx_hi] of bin rows by_lo .. by_hi" given one sample's
 * bin_start (HOST memory): run r copies count[r] records starting at record src_first[r] to offset dst_off[r] of the stage.
 * Returns the number of runs (the arrays hold the first `cap`), negative on bad arguments. */
B3D_API int b3d_pc_stage_records(void);
B3D_API int b3d_pc_stream_plan(const int32_t* bin_start_host, int nbx, int by_lo, int by_hi, int bx_lo, int bx_hi, int chunk,
                               int* dst_off, int* src_first, int* count, int cap);
B3D_API int b3d_pc_project(const float* points, const float* quat, int B, int N, int V, float fov,
                           float cam_dist, float* pg, float* coords, int32_t* base, uint8_t* inb,
                           float* sorted, int32_t* bin_start, void* stream);

/* Splat + z-blur + scale/clamp + ray termination + silhouette in ONE kernel (mode R): the V^3 grid lives
 * only in shared memory.
 *   TrilinearInterpolation.trilinear_interpolation / positions_update  utils/trilinear_interpolation.py:37-74
 *   VoxelsSmooth.smooth                                                utils/smooth_voxels.py:44-84
 *   EffectiveLossFunction.termination_probs + sum + flip               utils/effective_loss_function.py:18-56,79-81
 * (sorted, bin_start) from b3d_pc_project; taps [ktaps] the 1-D smoothing kernel (the host computes it with
 * the reference's expression, smooth_voxels.py:24-31); scale [B] nullable; sil [B,V,V] out.
 * workspace: b3d_pc_silhouette_workspace_bytes(B,V,mode) bytes (0 for mode R; may be NULL then).
 * The *_hosttaps variants take the taps from HOST memory (no device->host read of 21 floats); they are what
 * the Python wrapper calls.                                                                           */
B3D_API size_t b3d_pc_silhouette_workspace_bytes(int B, int V, int mode);
B3D_API int b3d_pc_silhouette_fwd(const float* sorted, const int32_t* bin_start, const float* taps, int ktaps,
                                  const float* scale, int B, int N, int V, int mode, float* sil,
                                  void* workspace, size_t workspace_bytes, void* stream);
B3D_API int b3d_pc_silhouette_fwd_hosttaps(const float* sorted, const int32_t* bin_start,
                                           const float* taps_host, int ktaps, const float* scale, int B,
                                           int N, int V, int mode, float* sil, void* workspace,
                                           size_t workspace_bytes, void* stream);

/* Backward of the above: dsil [B,V,V] -> dpg [B,N,4] (d/d grid coords, indexed by ORIGINAL point index,
 * written for in-bounds points only; .w unused), dscale [B] (nullable iff scale is NULL; zeroed by the call). */
B3D_API int b3d_pc_silhouette_bwd(const float* sorted, const int32_t* bin_start, const float* taps, int ktaps,
                                  const float* scale, const float* dsil, int B, int N, int V, int mode,
                                  float* dpg, float* dscale, void* workspace, size_t workspace_bytes,
                                  void* stream);
B3D_API int b3d_pc_silhouette_bwd_hosttaps(const float* sorted, const int32_t* bin_start,
                                           const float* taps_host, int ktaps, const float* scale,
                                           const float* dsil, int B, int N, int V, int mode, float* dpg,
                                           float* dscale, void* workspace, size_t workspace_bytes,
                                           void* stream);

/* Backward of b3d_pc_project: (pg, dpg) [B,N,4] -> dpoints [B,N,3], dquat [B,4] (zeroed by the call). */
B3D_API int b3d_pc_project_bwd(const float* points, const float* quat, const float* pg, const float* dpg,
                               int B, int N, int V, float fov, float cam_dist, float* dpoints,
                               float* dquat, void* stream);

/* Materialised occupancy grid [B,V,V,V] (clamped to [0,1]) — the tensor
 * TrilinearInterpolation.trilinear_interpolation returns (trilinear_interpolation.py:74).
 * Used by mode P and by the parity tests; grid is zeroed by the call. */
B3D_API int b3d_pc_splat_grid(const float* pg, int B, int N, int V, int mode, float* grid, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense voxel-grid kernels: the stand-alone VoxelsSmooth / termination_probs surface and mode P.
 *   b3d_vox_blur_axis        one separable kernel of VoxelsSmooth.smooth (utils/smooth_voxels.py:62-73): zero-padded
 *                            cross-correlation of in [B,V,V,V] along axis 1 (z), 2 (y) or 3 (x); taps in HOST memory;
 *                            reversed = 1 applies the adjoint.
 *   b3d_vox_scale_clamp(+_bwd)  clamp(in * scale[b], 0, 1) (smooth_voxels.py:80-82) and its adjoint (dscale zeroed by the call)
 *   b3d_vox_termination(+_bwd)  termination_probs [B,V+1,V,V] (nullable) and/or the silhouette [B,V,V] = sum of the first V
 *                            terms flipped along y (effective_loss_function.py:18-56,79-81); mode selects the epsilon pads
 *   b3d_vox_splat_sorted     raw (unclamped) trilinear scatter of the bin-sorted points (grid zeroed by the call)
 *   b3d_vox_clamp01          in-place clamp to [0,1] (trilinear_interpolation.py:74)
 *   b3d_vox_gather           adjoint of clamp + splat: dgrid masked by 0 <= raw <= 1, gathered at the 8 corners -> dpg
 * ------------------------------------------------------------------------------------------ */
B3D_API int b3d_vox_blur_axis(const float* in, float* out, const float* taps_host, int ktaps, int axis, int reversed,
                              int B, int V, void* stream);
B3D_API int b3d_vox_scale_clamp(const float* in, const float* scale, float* out, int B, int V, void* stream);
B3D_API int b3d_vox_scale_clamp_bwd(const float* in, const float* scale, const float* gout, float* gin, float* dscale,
                                    int B, int V, void* stream);
B3D_API int b3d_vox_termination(const float* vox, int B, int V, int mode, float* probs, float* sil, void* stream);
B3D_API int b3d_vox_termination_bwd(const float* vox, const float* dsil, int B, int V, int mode, float* dvox, void* stream);
B3D_API int b3d_vox_splat_sorted(const float* sorted, const int32_t* bin_start, int B, int N, int V, int mode, float* grid,
                                 void* stream);
B3D_API int b3d_vox_clamp01(float* x, long long n, void* stream);
B3D_API int b3d_vox_gather(const float* sorted, const int32_t* bin_start, const float* raw, float* dgrid, int B, int N, int V,
                           int mode, float* dpg, void* stream);

/* ------------------------------------------------------------------------------------------
 * Textured-mesh render path (replaces the kaolin dependency)
 *   Renderer.forward                          rendering/renderer.py:39-77
 * ------------------------------------------------------------------------------------------ */

/* ortho_projection + per-face gathers          rendering/renderer.py:9-28,52-58
 *   (kaolin dib_renderer.utils.datanormalize for normal1, renderer.py:52)
 * verts [B,P,3]; faces [F,3] int32; uv [B,T,2] (uv_batched=1) or [T,2] (0); ft [F,3] int32.
 * fgeo    [B,F,12] out: (ax,ay,bx,by,cx,cy)*multiplier, az,bz,cz, normal_z, 0,0
 * fuv     [B,F,6]  out, nullable: per-face-corner uv
 * normal1 [B,F,3]  out, nullable: unit face normals (the third value Renderer.forward returns)   */
B3D_API int b3d_mesh_face_setup(const float* verts, const int32_t* faces, const float* uv,
                                int uv_batched, const int32_t* ft, int B, int P, int F, int T,
                                float* fgeo, float* fuv, float* normal1, void* stream);

/* kaolin.graphics.dib_renderer.rasterizer.linear_rasterizer (renderer.py:60-67; defaults expand=0.02,
 * knum=30, multiplier=1000, delta=7000, restated from SURVEY.md App. B — parity unpinned) fused with
 * fragmentshader (rendering/fragment_shader.py:22-37, bilinear, align_corners=True).
 * tex [B,3,Th,Tw] : imout = shaded image [B,H,W,3] (tex*hardmask, or lerp(bg,tex,hardmask) with bg [B,H,W,3])
 * tex NULL        : imout = imfeat [B,H,W,3] = interpolated (u,v,1), what linear_rasterizer returns
 * imidx [B,H,W] int32 face index + 1 (0 = background; bit-exact target), imwei [B,H,W,3] barycentrics,
 * improb [B,H,W] soft silhouette (1 inside).                                                      */
B3D_API int b3d_mesh_render_fwd(const float* fgeo, const float* fuv, const float* tex, const float* bg,
                                int B, int F, int H, int W, int Th, int Tw, int32_t* imidx,
                                float* imwei, float* imout, float* improb, void* stream);

/* Adjoint: d_imout [B,H,W,3], d_improb [B,H,W] (nullable) -> dfp2d [B,F,6] (w.r.t. the UNSCALED 2-D
 * face vertices), dfuv [B,F,6], dtex [B,3,Th,Tw] (all zeroed by the call).  No gradient to depth or
 * normal_z (kaolin semantics).                                                                     */
B3D_API int b3d_mesh_render_bwd(const float* fgeo, const float* fuv, const float* tex, int has_bg, int B,
                                int F, int H, int W, int Th, int Tw, const int32_t* imidx,
                                const float* imwei, const float* d_imout, const float* d_improb,
                                float* dfp2d, float* dfuv, float* dtex, void* stream);

/* MeshTemplate.compute_normals                  rendering/mesh_template.py:113-123
 * verts [B,V,3], faces [F,3] int32 -> normals [B,F,3] = normalize((v_b - v_a) x (v_c - v_a)) (F.normalize: n / max(|n|, 1e-12)).
 * bwd: gnormals [B,F,3] -> dverts [B,V,3] (zeroed by the call, accumulated with atomics).  Vertex ids must lie in [0, V). */
B3D_API int b3d_face_normals_fwd(const float* verts, const int32_t* faces, int B, int V, int F, float* normals, void* stream);
B3D_API int b3d_face_normals_bwd(const float* verts, const int32_t* faces, const float* gnormals, int B, int V, int F,
                                 float* dverts, void* stream);

/* loss_flat(mesh, norms)                        utils/losses.py:5-17
 * norms [B,F,3]; ff [F,K] int32 face adjacency (negative ids index from the end, as torch does);
 * loss [1] out (zeroed by the call).  bwd: gloss [1] upstream gradient -> dnorms [B,F,3].        */
B3D_API int b3d_flat_loss_fwd(const float* norms, const int32_t* ff, int B, int F, int K, float* loss,
                              void* stream);
B3D_API int b3d_flat_loss_bwd(const float* norms, const int32_t* ff, int B, int F, int K,
                              const float* gloss, float* dnorms, void* stream);

/* nn.MSELoss()(cat(image, alpha).permute(0,3,1,2), X_real) + the counts mean_iou thresholds
 *                                               run_reconstruction.py:225-231,429-431
 * image [B,H,W,3], alpha [B,H,W], target [B,4,H,W]; loss [1] out; counts [B,2] int32 out, nullable:
 * {|pred&real|, |pred|real|} at threshold 0.5.  bwd writes d_image, d_alpha (= 2 (x - t) gloss / n).  */
B3D_API int b3d_rgba_mse_iou_fwd(const float* image, const float* alpha, const float* target, int B, int H,
                                 int W, float* loss, int32_t* counts, void* stream);
B3D_API int b3d_rgba_mse_bwd(const float* image, const float* alpha, const float* target, int B, int H,
                             int W, const float* gloss, float* d_image, float* d_alpha, void* stream);

/* ------------------------------------------------------------------------------------------
 * Chamfer / pairwise nearest neighbour (north-star kernel; no reference implementation exists —
 * the reference's only pairwise-NN site is rendering/mesh_template.py:33-39).
 * query [B,N,3], cand [B,M,3] -> dist [B,N] = min_j |q_i - c_j|^2, idx [B,N] int32 = argmin (lowest index on
 * ties; bit-exact target).  bwd ACCUMULATES into dquery [B,N,3] and dcand [B,M,3] (caller zeroes them).
 * ------------------------------------------------------------------------------------------ */
B3D_API int b3d_chamfer_nn(const float* query, const float* cand, int B, int N, int M, float* dist,
                           int32_t* idx, void* stream);
B3D_API int b3d_chamfer_bwd(const float* query, const float* cand, const int32_t* idx, const float* gdist,
                            int B, int N, int M, float* dquery, float* dcand, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense 2-D convolution of the conv-GAN (nn.Conv2d call sites models/gan.py:57-65,163-177,294-302,359,364)
 * as a tcgen05 / TMA implicit GEMM (tf32 inputs, fp32 accumulate — cuDNN's default TF32 class, SURVEY §2.2).
 *   out[n, osy*y+ooy, osx*x+oox, co] = leaky( bias[co] + sum_t sum_ci x[n, sy*y+dy[t], sx*x+dx[t], ci] * wt[t, co, ci] )
 * x [N,H,W,Cin] NHWC fp32 (Cin % 32 == 0; reads outside [0,H)x[0,W) are zero = the conv's zero padding),
 * wt [ntaps,Cout,Cin] (w_cin_major = 0) or [ntaps,Cin,Cout] (w_cin_major = 1: N-major B operand, Cout % 4 == 0),
 * bias [Cout] nullable, out [N,OH,OW,OC]; (y,x) run over [0,Hout)x[0,Wout).
 * fprop: dy = r - pad_y, dx = s.  dgrad: dy = pad_y - r, dx = -s with wt[t] = W[:,:,r,s]^T (strided dgrad = one
 * call per output parity class with osy = osx = 2).  leaky = negative slope of the fused LeakyReLU (1 = none).
 * ------------------------------------------------------------------------------------------ */
/* Optional extras of b3d_conv2d_tf32 (all zero = none).  They exist for the discriminators' backward pass
 * (models/gan.py:163-177,294-302: conv -> bias -> LeakyReLU -> wrap-around x padding -> next conv), where the input
 * gradient of layer L+1 IS the gradient of layer L's padded, activated output:
 *   mask        tensor with the geometry of `out` (the activated forward tensor the gradient belongs to): the epilogue
 *               stores acc * (mask >= 0 ? 1 : mask_slope) — the LeakyReLU adjoint without a pass of its own; `stats`
 *               then receives the sums of the masked values (stats_sum_only = 1: the sum of squares is skipped), i.e. the
 *               bias gradient once the pad columns are folded back (b3d_wrap_x_bwd_inplace).
 *   x_row_pitch x is a W-pixel-wide window of rows that are x_row_pitch pixels apart in memory (image n at
 *               n * H * x_row_pitch pixels): the interior of a padded gradient buffer is read in place; columns outside
 *               [0, W) read as zero even though the memory behind them is valid.
 *   nclass      2..4: ONE launch computes nclass outputs that share x, the strides and the logical extent (Hout, Wout) —
 *               the output-parity classes of a stride-2 input gradient.  dy / dx / wtap hold nclass consecutive groups of
 *               ntaps / nclass taps; class c is written at (osy*y + class_ooy[c], osx*x + class_oox[c]) (ooy / oox are
 *               ignored).  Classes are the fastest-varying work index, so the CTAs that read the same pixel tiles of x
 *               run at the same time and share them in L2 (four separate launches re-read x four times from HBM).           */
typedef struct b3d_conv_opts {
    const float* mask;
    float mask_slope;
    int stats_sum_only;
    int x_row_pitch;
    int nclass;
    int class_ooy[4];
    int class_oox[4];
} b3d_conv_opts;
B3D_API int b3d_conv2d_tf32(const float* x, const float* wt, const float* bias, float* out, int N, int H, int W,
                            int Cin, int Hout, int Wout, int Cout, int ntaps, const int* dy, const int* dx,
                            int sy, int sx, int OH, int OW, int OC, int osy, int osx, int ooy, int oox,
                            float leaky, int w_cin_major, const int* wtap, int wtaps_total, double* stats, int fold_kh,
                            int fold_pad, const b3d_conv_opts* opts, void* stream);
/* wtap (nullable): loop tap t reads weight tap wtap[t] of a tap-major array that holds wtaps_total taps — the stride-2
 * input-gradient parity classes address their tap subsets of the full weight array without a gathered copy.
 * stats (nullable): [2][Cout] fp64, ACCUMULATED into by the epilogue: per-channel sum and sum of squares of the output
 * before bias / activation — the BatchNorm statistics of the generator's layers without a second pass over the tensor
 * (models/gan.py:264-286; the caller zeroes the buffer; dense outputs only, or nclass = 4 parity classes of a stride-2
 * output, which together cover it).
 * fold_kh > 0: thin 8-channel stems (models/gan.py:163-166, 5x5 on 8 channels): x is the RAW input [N,H,W,8]; the kh vertical
 * taps are folded into the K dimension ON THE FLY by the TMA boxes (four image rows x 8 channels = one 32-channel K slice, rows
 * outside the image = the zero padding fold_pad) — Cin is the folded channel count (32 * ceil(8 kh / 32)), the taps are the kw
 * horizontal ones, wt is the folded tap-major layout [kw][Cout][Cin] (b3d/bank.py `fold`).  Needs Wout % 128 == 0.            */

/* Stride-1 variant with a halo-staged input and R stacked accumulators (csrc/tc_conv2.cu): x [N,H,P,Cin] with P the
 * padded width (row pitch), taps (dy, dx >= 0); same weights / bias / LeakyReLU semantics as b3d_conv2d_tf32, output
 * out[n,y,x,co] for y < Hout, x < Wout of a tensor [N,OH,OW,OC].  Returns B3D_EINVAL ("does not fit") when the halo
 * (max tap offset - min tap offset rows of 128 B) exceeds shared memory; callers then use b3d_conv2d_tf32.          */
B3D_API int b3d_conv2d_flat_tf32(const float* x, const float* wt, const float* bias, float* out, int N, int H, int P,
                                 int Cin, int Hout, int Wout, int Cout, int ntaps, const int* dy, const int* dx,
                                 int OH, int OW, int OC, float leaky, void* stream);

/* Weight gradient of the same convolution (split-K tcgen05 GEMM over the output pixels, M/N-major operands
 * straight from the NHWC tensors):
 *   dw[co, ci, r, s] += sum_{n,y,x} dy[n, y, x, co] * x[n, stride*y + r - pad_y, stride*x + s + x_off, ci]
 * dy [N,Hout,Wout,Cout], x [N,H,W,Cin] (x already padded along x; Cin, Cout multiples of 4; x_off > -kw: columns left
 * of x read as zero),
 * dw [Cout,Cin,kh,kw] is ACCUMULATED into (caller zeroes it).                                          */
B3D_API int b3d_conv2d_wgrad_tf32(const float* dy, const float* x, float* dw, int N, int H, int W, int Cin,
                                  int Hout, int Wout, int Cout, int kh, int kw, int pad_y, int stride,
                                  int x_off, int tap_major, int fold_kh, int dy_row_pitch, void* stream);
/* dy_row_pitch > 0: dy is a Wout-pixel-wide window of rows dy_row_pitch pixels apart (the interior of a padded gradient
 * buffer, read in place); 0 = dense [N,Hout,Wout,Cout].                                                                   */
/* tap_major != 0: dw is the tap-major array [kh*kw][Cout][Cin] (the layout b3d_conv2d_tf32 reads, 16-byte vector
 * reductions) instead of [Cout][Cin][kh][kw].  fold_kh > 0: x is the raw 8-channel stem input, folded on the fly as in
 * b3d_conv2d_tf32 (kh = 1, kw = the horizontal taps, Cin = folded channel count, pad_y = the fold's y padding).              */

/* Thin heads: 5x5 / stride-1 convolutions with 1..4 output channels (generator conv_final, models/gan.py:359;
 * discriminator heads :177, :302) on the fp32 CUDA cores, channels across the lanes of a warp.  Cin % 64 == 0.
 *   _fwd:   x [N,H,W,Cin], wt [25][Cout][Cin] (tap-major, as b3d_conv2d_tf32), bias [Cout] or NULL ->
 *           out[n, y, x, co] = leaky(bias + sum ...) written with pixel pitch OW and channel pitch OC.
 *   _wgrad: dw [Cout,Cin,5,5] += sum dy[n,y,x,co] * x[n, y + r - pad_y, x + s + x_off, ci]   (dy dense [N,Hout,Wout,Cout]). */
B3D_API int b3d_conv2d_thin_fwd(const float* x, const float* wt, const float* bias, float* out, int N, int H, int W, int Cin,
                                int Hout, int Wout, int Cout, int kh, int kw, int pad_y, int x_off, int OW, int OC,
                                float leaky, void* stream);
B3D_API int b3d_conv2d_thin_wgrad(const float* dy, const float* x, float* dw, int N, int H, int W, int Cin, int Hout,
                                  int Wout, int Cout, int kh, int kw, int pad_y, int x_off, int tap_major, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused vertex pipeline (csrc/vertex_kernels.cu; SURVEY §8f rank 1): displacement map -> template vertices -> camera
 * space in one launch (and one for the backward).
 *   MeshTemplate.get_vertex_positions / deform / adjust_uv_and_texture   rendering/mesh_template.py:106-111,125-170
 *   transform_vertices                                                    run_reconstruction.py:237-252
 *   qrot                                                                  rendering/utils.py:36-46
 * dmap [B,3,h,w] addressed through element strides (sn, sc, sy, sx); rec [V] per-vertex records of
 * b3d_vertex_record_bytes() bytes (int32 tap[4] texel offsets y*w+x of the unpadded map with the wrap-around column
 * resolved, float wgt[4] bilinear weights, float frame[9] tangent frame rows, float v0[3]); sgn [V] float4 (x factor:
 * -1 mirrored vertex, 0 on the symmetry plane, +1).  Pose (nullable together with vtx): scale [B], trans [B,3], rot
 * [B,4] (w,x,y,z), z0 [B] (nullable: perspective correction).  raw / vtx [B,V,3].
 * _bwd: g_raw / g_vtx [B,V,3] (either nullable) -> d_dmap [B,3,h,w] (NCHW contiguous), d_scale [B], d_trans [B,3],
 * d_z0 [B] (all nullable, ACCUMULATED into: the caller zeroes them).
 * ------------------------------------------------------------------------------------------ */
B3D_API int b3d_vertex_record_bytes(void);
B3D_API int b3d_vertex_pipeline_fwd(const float* dmap, long long sn, long long sc, long long sy, long long sx, int h, int w,
                                    const void* rec, const void* sgn, int B, int V, const float* scale, const float* trans,
                                    const float* rot, const float* z0, float* raw, float* vtx, void* stream);
B3D_API int b3d_vertex_pipeline_bwd(const float* g_raw, const float* g_vtx, const float* raw, const void* rec, const void* sgn,
                                    int B, int V, int h, int w, const float* scale, const float* trans, const float* rot,
                                    const float* z0, float* d_dmap, float* d_scale, float* d_trans, float* d_z0, void* stream);

/* ------------------------------------------------------------------------------------------
 * Weight bank (csrc/sn_kernels.cu): spectral normalisation (torch.nn.utils.spectral_norm as applied at
 * models/gan.py:57-65,163-177,294-302: one power iteration in training mode, sigma = u.(W v), W / sigma) and the
 * kernel weight layouts of ALL convolutions of a network in four launches; backward maps the tap-major weight
 * gradients back to weight_orig's layout through d(W / sigma).  `layers` is a device array of records of
 * b3d_bank_layer_bytes() bytes each (field order: csrc/sn_kernels.cu BankLayer; packed by b3d/bank.py), `items_*` device
 * arrays of int4 work items, `scratch` a per-bank buffer (zeroed here), `out` / `df` / `dw` per-call flat buffers.
 * `training`: bit 0 = training mode (power iteration), bit 1 = round the emitted weights to the nearest tf32 value.
 * ------------------------------------------------------------------------------------------ */
B3D_API int b3d_bank_layer_bytes(void);
B3D_API int b3d_bank_forward(const void* layers, const void* items_wtu, int n_wtu, const void* items_wv, int n_wv,
                             const void* items_emit, int n_emit, float* scratch, size_t scratch_bytes, float* out,
                             int training, void* stream);
B3D_API int b3d_bank_backward(const void* layers, const void* items_dot, int n_dot, const void* items_emit, int n_emit,
                              float* out, const float* df, float* dw, void* stream);
/* up2 layers (BankLayer.up2: a 3x3 convolution run on the input of its x2 nearest upsample as four 2x2 parity-class
 * convolutions, class taps UF / UD written by b3d_bank_forward): the adjoint of the 3x3 -> class-tap map.  dk [4x4][Cin][Cout]
 * is the up-convolution's weight gradient as b3d_conv2d_wgrad_tf32 (tap-major) leaves it; it is ACCUMULATED into df
 * [9][Cout][Cinp], the layer's F-layout gradient sink. */
B3D_API int b3d_bank_up2_grad(const float* dk, float* df, int Cout, int Cin, int Cinp, void* stream);

/* ------------------------------------------------------------------------------------------
 * One-pass NHWC helpers between the GAN's convolutions.
 * b3d_pad_x_*: padding along x of x [rows = N*H, W, C] -> out [rows, W + 2*amount, C]; mode 0 = replicate
 *   (F.pad(..., mode='replicate'), models/gan.py:329), 1 = circular (circpad, rendering/utils.py:29-33); C % 4 == 0.
 * b3d_leaky_bwd: out = gy * (y >= 0 ? 1 : slope) — gradient of the LeakyReLU fused into the conv epilogue.
 * ------------------------------------------------------------------------------------------ */
B3D_API int b3d_pad_x_fwd(const float* x, float* out, long long rows, int W, int C, int amount, int mode, void* stream);
B3D_API int b3d_pad_x_bwd(const float* gout, float* gx, long long rows, int W, int C, int amount, int mode, void* stream);
/* Discriminator stem input (models/gan.py:102-111 `_with_positions`, :95-96 wrap-around padding, then conv1 :163-166) in one
 * pass: out [N, H, W + 2*amount, C1 + C2] (NHWC) = x-padding (mode 0 replicate / 1 circular) of concat(x [N,C1,H,W] (NCHW
 * planes), pos [C2,H,W] broadcast over N).  C1 + C2 = 4 or 8.  _bwd: gx [N,C1,H,W] = adjoint w.r.t. x (pos is a constant). */
B3D_API int b3d_stem_input_fwd(const float* x, const float* pos, float* out, int N, int C1, int C2, int H, int W, int amount,
                               int mode, void* stream);
B3D_API int b3d_stem_input_bwd(const float* gout, float* gx, int N, int C1, int C2, int H, int W, int amount, int mode,
                               void* stream);
/* Thin-stem fold in front of the 5x5 discriminator stems (models/gan.py:163, :294 — 8 / 11 input channels): the kh
 * vertical taps become channels, out [N, H + 2*pad_y - kh + 1, W, Cp][.., r*C + c] = x [N,H,W,C][n, y + r - pad_y, x, c]
 * (zero rows = the y padding, zero channels up to Cp), so the tensor cores see kw taps of kh*C real channels.  _bwd is
 * the adjoint (gx [N,H,W,C] from gout [N,Hout,W,Cp]). */
B3D_API int b3d_fold_rows_fwd(const float* x, float* out, int N, int H, int W, int C, int kh, int pad_y, int Cp, void* stream);
B3D_API int b3d_fold_rows_bwd(const float* gout, float* gx, int N, int H, int W, int C, int kh, int pad_y, int Cp, void* stream);
/* In-place x padding of buf [rows, W + 2*amount, C] whose interior columns were written by a convolution epilogue
 * (b3d_conv2d_tf32 with OW = W + 2*amount, oox = amount): fills the 2*amount pad columns (mode 0 replicate / 1 circular).
 * Replaces circpad (rendering/utils.py:29-33) / F.pad (models/gan.py:329) after a conv without a full-tensor copy. */
B3D_API int b3d_wrap_x_inplace(float* buf, long long rows, int W, int C, int amount, int mode, void* stream);
/* Adjoint of b3d_wrap_x_inplace, in place: the gradients of the 2*amount pad columns of g [rows, W + 2*amount, C] are
 * added to the interior columns they were copied from (mode 1: column W + j += column j, column amount + j += column
 * W + amount + j; mode 0: the edge columns collect their side's pad columns).  The pad columns keep their values: consumers
 * read the interior through x_row_pitch / dy_row_pitch.  amount <= W, C % 4 == 0. */
B3D_API int b3d_wrap_x_bwd_inplace(float* g, long long rows, int W, int C, int amount, int mode, void* stream);
/* Backward of conv -> bias -> LeakyReLU(slope) -> x padding in one pass (models/gan.py discriminators :163-177,
 * :294-302): gy [rows, W, C] = pad^T(gout_pad [rows, W + 2*amount, C]) * leaky'(y_pad interior); gbias [C] (nullable)
 * accumulates sum(gy) (caller zeroes it).  C = 4 * power of two. */
B3D_API int b3d_pad_leaky_bias_bwd(const float* gout_pad, const float* y_pad, float* gy, float* gbias, long long rows, int W,
                                   int C, int amount, int mode, float slope, void* stream);
B3D_API int b3d_leaky_bwd(const float* gy, const float* y, float* out, long long n, float slope, void* stream);

/* Batch-norm statistics of an NHWC activation y [rows = N*H*W, C] in one pass: mean[c] and invstd[c] = 1/sqrt(biased
 * variance + eps) — what F.batch_norm / torch.batch_norm_stats compute for the generator's BatchNorm2d(affine=False)
 * layers (models/gan.py:211-232).  workspace: 2*C doubles (zeroed by the call).  C = 4 * a divisor of 256. */
B3D_API int b3d_bn_stats(const float* y, long long rows, int C, float eps, float* mean, float* invstd, double* workspace,
                         void* stream);

/* Fused generator glue between two convolutions (models/gan.py:282-286 ConditionalBatchNorm2d, :309-311 LeakyReLU and
 * residual add, :319 nearest x2 upsample, :329 replicate pad), NHWC, C % 4 == 0:
 *   out[n, yo, xo, :] = post( leaky(y[n,ys,xs,:] * scale[n,:] + shift[n,:]) + skip[n,ys,xs,:] ),
 *   (ys, xs) = (yo / up, clamp(xo - pad, 0, up*W-1) / up);  out [N, up*H, up*W + 2*pad, C];  scale = inv_std*(1+gamma),
 *   shift = beta - mean*scale ([N,C]); skip (nullable) is read at row pitch skip_pitch, pixel offset skip_off.
 *   skip_half = 1 (even H, W): the skip is at half resolution [N,H/2,..] and read at (ys/2, xs/2) — the residual of a block
 *   whose input arrives before the x2 upsample (nearest upsampling commutes with the identity and the 1x1 shortcut).
 * bwd1: gout -> ga = d/d(pre-activation) [N,H,W,C], gskip (nullable; skip_half: the 2x2 sums, at half resolution),
 *       S1[n,c] = sum ga, S2[n,c] = sum ga*xhat: rows of
 *       pitch s_pitch floats (>= C; slices of the batched d(gamma, beta) buffer), zeroed by the call
 * bwd2 (in place on ga): dy = inv_std * (ga * gamma_t - m1 - xhat * m2), (m1, m2) [C] = inv_m * (sums of d xhat, d xhat * xhat)
 * b3d_cbn_prepare / b3d_cbn_bwd_reduce / b3d_bn_sums: the per-layer scalar math around these passes, one launch each
 *       (statistics -> mean / inv_std / running buffers / scale / shift; coupling-term reduction; fp64 channel sums).       */
B3D_API int b3d_cbn_act_fwd(const float* y, const float* scale, const float* shift, const float* skip, int skip_pitch,
                            int skip_off, float* out, int N, int H, int W, int C, int up, int pad, float slope,
                            int post_leaky, int skip_half, void* stream);
B3D_API int b3d_cbn_act_bwd1(const float* gout, const float* y, const float* scale, const float* shift, const float* skip,
                             int skip_pitch, int skip_off, const float* mean, const float* invstd, float* ga, float* gskip,
                             int gskip_pitch, int gskip_off, float* S1, float* S2, int s_pitch, int N, int H, int W, int C,
                             int up, int pad, float slope, int post_leaky, int skip_half, void* stream);
B3D_API int b3d_cbn_act_bwd2(float* ga, const float* y, const float* gamma_t, const float* mean, const float* invstd,
                             const float* m1, const float* m2, float inv_m, int N, int H, int W, int C, void* stream);
B3D_API int b3d_bn_sums(const float* y, long long rows, int C, double* sums, void* stream);
B3D_API int b3d_cbn_prepare(const float* gb, int gb_pitch, int gamma_off, int beta_off, const double* sums, double count,
                            float eps, float momentum, int mode, float* running_mean, float* running_var,
                            long long* num_batches_tracked, float* mean, float* invstd, float* scale, float* shift, float* gt,
                            int N, int C, void* stream);
B3D_API int b3d_cbn_bwd_reduce(const float* S1, const float* S2, int s_pitch, const float* gt, float* red, int N, int C,
                               void* stream);
/* SyncBN (sync_batchnorm/batchnorm.py:68-150: statistics over all replicas) with the collective FUSED into the consuming
 * kernel: a one-shot all-reduce over NVLink / NVSwitch peer memory (csrc/ew_kernels.cu peer_allreduce) instead of a
 * separate NCCL all-reduce per layer.  peer_data / peer_flag: host arrays of `world` device pointers (rank order) into every
 * rank's symmetric buffer (b3d_sync_buffer_bytes(world) bytes, zeroed once; flags start at b3d_sync_flag_offset(world));
 * epoch / err: this rank's own device counters (zeroed once; *err != 0 after a peer timed out).  Same maths as
 * b3d_cbn_prepare mode 2 / b3d_cbn_bwd_reduce on the global sums.  world <= 8, C <= 512; every rank issues the same calls. */
B3D_API size_t b3d_sync_buffer_bytes(int world);
B3D_API size_t b3d_sync_flag_offset(int world);
B3D_API int b3d_cbn_prepare_sync(const void* const* peer_data, const void* const* peer_flag, int rank, int world,
                                 unsigned* epoch, int* err, const float* gb, int gb_pitch, int gamma_off, int beta_off,
                                 const double* sums_local, double count, float eps, float momentum, float* running_mean,
                                 float* running_var, long long* num_batches_tracked, float* mean, float* invstd, float* scale,
                                 float* shift, float* gt, int N, int C, void* stream);
B3D_API int b3d_cbn_bwd_reduce_sync(const void* const* peer_data, const void* const* peer_flag, int rank, int world,
                                    unsigned* epoch, int* err, const float* S1, const float* S2, int s_pitch, const float* gt,
                                    float* red, int N, int C, void* stream);

/* ---- FID evaluation (SURVEY §8f rank 4; reference: main.py:188-412 evaluate_fid, utils/fid.py, utils/inception.py) ----------
 * The Inception-v3 convolutions run on b3d_conv2d_tf32 (BatchNorm folded into weights and bias, ReLU = leaky slope 0 in the
 * epilogue, every branch written into its channel slice of the concatenated tensor through OC / the output pointer); 3x3
 * average pools are folded into the 1x1 convolution that follows them (nine taps of w / 9).  The rest:
 * b3d_inception_input   utils/inception.py:123-131: img [B,3,H,W] planes in (0,1) -> bilinear resize to OH x OW
 *                       (align_corners=False; identity when the size already matches), 2x - 1 when normalize != 0, written
 *                       as NHWC [B,OH,OW,OC] with channels 3..OC-1 zero (OC % 4 == 0: one 32-channel K slice for the stem)
 * b3d_maxpool3x3s2_nhwc nn.MaxPool2d(3, stride=2) on x [N,H,W,C]; `out` points at the first channel of the destination slice
 *                       of a tensor with OC channels per pixel ([N,(H-3)/2+1,(W-3)/2+1,OC]); C, OC multiples of 4
 * b3d_mean_hw_nhwc      AdaptiveAvgPool2d((1,1)): x [N,HW,C] -> out [N,C]
 * b3d_fid_accumulate    utils/fid.py:27-30 calculate_stats as running sums: sum [D] += sum_k feat[k,:],
 *                       outer [D,D] += feat^T feat, both fp64 (feat [n,D] fp32); mu = sum / n,
 *                       sigma = (outer - n mu mu^T) / (n - 1) afterwards (np.cov's unbiased estimate).                        */
B3D_API int b3d_inception_input(const float* img, int B, int H, int W, int OH, int OW, int OC, int normalize, float* out,
                                void* stream);
B3D_API int b3d_maxpool3x3s2_nhwc(const float* x, int N, int H, int W, int C, float* out, int OC, void* stream);
B3D_API int b3d_mean_hw_nhwc(const float* x, int N, int HW, int C, float* out, void* stream);
B3D_API int b3d_fid_accumulate(const float* feat, int n, int D, double* sum, double* outer, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B3D_H_ */
