/* vpn_b200 - C ABI of the B200 (sm_100a) primitive-assembly + loss kernels.
 *
 * Drop-in boundary for the hot path of hank-kuo-cs/Volumetric-Primitives-Net (SURVEY.md section 8b).
 * The reference has no FFI layer for this path - its boundary is the Python call surface of
 * modules/{transform,sampling,loss,render,meshing} - so the convention copied here is the one of its
 * only native op (modules/loss/emd/emd_module.py:32-59, emd.cpp:6-23): the caller allocates every output
 * and scratch buffer, native code only fills them and returns an int status.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous fp32 / int32 data unless stated otherwise;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous, stream ordered, never
 *     allocate, never synchronise (the *_timed / probe measurement helpers excepted) and keep no state between calls
 *     (process-wide: an atomic launch counter, per-device caches of immutable device properties, and the
 *     vpn_set_tuning overrides; every device of a multi-GPU process is handled independently);
 *   - return 0 on success, negative on error (VPN_ERR_*); vpn_last_error_string() describes the last
 *     error of the calling thread;
 *   - "nprim" is B*K: one pose (v,q,t) per primitive, primitives laid out sample-major (b*K + k).
 */
#ifndef VPN_B200_H
#define VPN_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VPN_OK 0
#define VPN_ERR_CUDA (-1)
#define VPN_ERR_SHAPE (-2)
#define VPN_ERR_ARG (-3)
#define VPN_ERR_WORKSPACE (-4)

/* kinds for vpn_pose_points_* */
#define VPN_KIND_SPHERE 0   /* src = uniforms (nprim, N, 2): [elev draw, azim draw]  (sampling/sphere.py:26-27) */
#define VPN_KIND_CUBOID 1   /* src = uniforms (nprim, N, 3)                           (sampling/cuboid.py:66)     */
#define VPN_KIND_TEMPLATE 2 /* src = template vertices (N, 3), shared by all primitives (meshing/sphere.py:17)   */
#define VPN_KIND_POINTS 3   /* src = caller points (nprim, N, 3); v ignored          (transform/transform.py:6)  */

const char* vpn_last_error_string(void);
int vpn_abi_version(void);
int vpn_device_info(int* sm_count, int* cc_major, int* cc_minor, int* clock_khz);
/* kernels launched by this library in this process so far (bench.py reports the per-step delta) */
unsigned long long vpn_launch_count(void);
/* Test / probe hook: force a launch-plan choice.  key "tiled_r" | "tc_nb" (4, 8, 16), "emd_cluster" (1, 2, 4, 8),
 * "tc_prune" (2 = tensor-core Chamfer filter without the spatial pruning), "tc_hunits" (1 + the 32-column units of a
 * block reduced on the FP16 pipe, 1..5), "serial_recovery" (1 = row and column recovery on one stream),
 * "prep_near_rows" | "prep_near_cols" (1..32) and "prep_reps_rows" | "prep_reps_cols" (1, 2, 4): near blocks and
 * representatives of the pruning bounds, "prep_deterministic" (1 = reproducible sort permutation), "prep_probe" (1 =
 * phase timers of the sort kernel in the statistics words), "ar_variant" | "ar_ctas" | "ar_threads" | "ar_grid_div"
 * (all-reduce launch shape); value 0 restores the automatic choice.  Results never depend on it (tests check exactly
 * that); unknown keys return VPN_ERR_ARG. */
int vpn_set_tuning(const char* key, int value);

/* ---- primitive instantiation: canonical sample -> scale -> rotate -> translate, one kernel ------------
 * Replaces Sampling.{sphere,cuboid}_sampling (modules/sampling/sampling.py:12-38), transform_points /
 * rotate_points / translate_points (modules/transform/transform.py:6-18, rotate.py:7-25, translate.py:4-8)
 * and Meshing.{sphere,cuboid}_meshing's vertex math (modules/meshing/sphere.py:8-27, cuboid.py:8-27).
 * v (nprim,3), q (nprim,4) = (axis, turn fraction), t (nprim,3) or NULL (rotate only), out (nprim,N,3). */
int vpn_pose_points_fwd(int kind, const float* v, const float* q, const float* t, const float* src,
                        float* out, int nprim, int N, void* stream);
/* Measurement variant: `reps` launches back to back, launch i reading srcs[i % nsrc] (HOST array of device pointers),
 * one CUDA-event pair around the stream of launches; *ms_per_launch is a HOST float.  Synchronises. */
int vpn_pose_points_fwd_timed(int kind, const float* v, const float* q, const float* t, const float* const* srcs,
                              int nsrc, float* out, int nprim, int N, int reps, float* ms_per_launch, void* stream);
int vpn_pose_bwd_workspace_floats(int nprim, int N, size_t* floats);
/* grad_out (nprim,N,3) -> grad_v (nprim,3), grad_q (nprim,4), grad_t (nprim,3); any may be NULL.
 * grad_points (nprim,N,3) is written for VPN_KIND_POINTS only (may be NULL). */
int vpn_pose_points_bwd(int kind, const float* v, const float* q, const float* src, const float* grad_out,
                        float* grad_v, float* grad_q, float* grad_t, float* grad_points,
                        float* workspace, size_t workspace_floats, int nprim, int N, void* stream);
/* get_faces_points (modules/sampling/cuboid.py:30-53): counts (nprim,6) int32. */
int vpn_cuboid_face_counts(const float* v, int* counts, int nprim, int N, void* stream);

/* ---- camera frame changes: view_to_obj_points / obj_to_view_points (modules/transform/transform.py:21-73)
 * mode 0 = view_to_obj (angles required), 1 = obj_to_view.  transpose 1 = gradient w.r.t. the points. */
int vpn_view_workspace_bytes(int B, size_t* bytes);
int vpn_view_points(int mode, int transpose, const float* in, const float* dists, const float* elevs,
                    const float* azims, const float* angles, float* out, void* workspace,
                    size_t workspace_bytes, int B, int n, void* stream);

/* ---- Chamfer nearest neighbours, both directions (modules/loss/chamfer_distance.py:14-23) ------------
 * p1 (B,P,3), p2 (B,M,3) -> min1 (B,P) = min_j sqrt(d_ij), idx1 (B,P) int32 = first arg-min, min2 (B,M),
 * idx2 (B,M).  Arg-mins are bit-exact to torch.min over the reference's dense distance tensor.
 * impl: 0 auto (tensor-core filter when the shape allows, else the CUDA-core tiled kernel, else generic),
 * 1 generic kernel, 2/3/4 CUDA-core tiled kernel with exact / FMA-difference / centred-expansion hot-loop
 * arithmetic, 5 tcgen05 tensor-core filter (fp16-split operands, fp32 accumulate).  Results are identical for
 * every impl: the hot loop only selects candidates, the recovery kernels redo them with the reference's arithmetic. */
int vpn_chamfer_workspace_bytes(int B, int P, int M, int impl, size_t* bytes);
int vpn_chamfer_fwd(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                    int B, int P, int M, void* workspace, size_t workspace_bytes, int impl, void* stream);
/* Name of the kernel the forward spends its time in for this shape and impl (static string; measurement label). */
const char* vpn_chamfer_main_kernel(int B, int P, int M, int impl);
/* Measurement variant: `reps` forwards with CUDA events between the stages; stage_ms is a HOST float[4]
 * (main kernel, fall-back launch, row recovery, column recovery), mean ms per stage.  Synchronises. */
int vpn_chamfer_fwd_timed(const float* p1, const float* p2, float* min1, int* idx1, float* min2, int* idx2,
                          int B, int P, int M, void* workspace, size_t workspace_bytes, int impl, int reps,
                          float* stage_ms, void* stream);
/* Pruning statistics of the last vpn_chamfer_fwd that used `workspace` (tensor-core filter only, else zeros): the sweep's
 * 128 x 256 stages (both directions counted) and how many of them the spatial pruning skipped.  Synchronises. */
int vpn_chamfer_prune_stats(const void* workspace, int B, int P, int M, int impl, unsigned long long* stages,
                            unsigned long long* skipped, void* stream);
/* Probe: the filter's 16 counters - [0] stages, [1] skipped, [2..5] cycles of one epilogue warp summed over the CTAs
 * (prologue, row phase, column phase, tail), [6] / [7] live stages per phase, [8] live chunks, [9] operand passes built. */
int vpn_chamfer_tc_counters(const void* workspace, int B, int P, int M, int impl, unsigned long long* out16, void* stream);
/* g1 (B,P), g2 (B,M): upstream gradients of min1 / min2.  grad_p1 (B,P,3) overwritten; grad_p2 (B,M,3)
 * overwritten when not NULL.  Same result as autograd through the reference's dense graph. */
int vpn_chamfer_bwd(const float* p1, const float* p2, const float* min1, const int* idx1,
                    const float* min2, const int* idx2, const float* g1, const float* g2,
                    float* grad_p1, float* grad_p2, int B, int P, int M, void* stream);

/* Fused loss head/tail of ChamferDistanceLoss (chamfer_distance.py:25-28): loss[b] = w1*mean(min1[b]) + w2*mean(min2[b]);
 * the backward takes the per-sample upstream gradient grad_loss (B) instead of full (B,P)/(B,M) tensors. */
int vpn_chamfer_loss_fwd(const float* min1, const float* min2, float w1, float w2, float* loss,
                         float* scratch /* >= 64*B floats */, int B, int P, int M, void* stream);
int vpn_chamfer_loss_bwd(const float* p1, const float* p2, const float* min1, const int* idx1,
                         const float* min2, const int* idx2, const float* grad_loss, float w1, float w2,
                         float* grad_p1, float* grad_p2, int B, int P, int M, void* stream);

/* ---- soft silhouette (modules/loss/silhouette.py:13-23 -> render/vertex_renderer.py:15-26 -> kaolin DIB-R)
 * verts (B,V,3), faces (F,3) int32 shared topology, cam_rot (B,3,3), cam_pos (B,3), proj = (px,py,pz).
 * alpha (B,H,W); covered (B,H,W) uint8; normals (B,F,3) or NULL.  bwd needs the workspace as fwd left it.
 * soft_cull_backfaces: 0 = DIB-R as recalled in SURVEY.md 8(a-R): back faces (normal.z < 0) are skipped by the coverage
 * (hard) pass only and still count among the first `knum` soft candidates; 1 = they are skipped by the soft pass too. */
int vpn_silhouette_workspace_bytes(int B, int V, int F, size_t* bytes);
int vpn_silhouette_fwd(const float* verts, const int* faces, const float* cam_rot, const float* cam_pos,
                       float proj_x, float proj_y, float proj_z, float expand, int knum, float multiplier,
                       float delta, int soft_cull_backfaces, float* alpha, unsigned char* covered, float* normals,
                       void* workspace, size_t workspace_bytes, int B, int V, int F, int H, int W, void* stream);
int vpn_silhouette_bwd(const int* faces, const float* cam_rot, float proj_x, float proj_y, float proj_z,
                       float expand, int knum, float multiplier, float delta, int soft_cull_backfaces, const float* grad_alpha,
                       const unsigned char* covered, float* grad_verts, void* workspace, size_t workspace_bytes,
                       int B, int V, int F, int H, int W, void* stream);

/* ---- area-weighted mesh surface sampling: kaolin TriangleMesh.sample at train_sphere.py:71-80, dataset/dataset.py:162-165
 * verts (B,V,3), faces (F,3) int32 shared topology, u (B,n,3) uniforms in [0,1): [face draw, u1, u2].
 * points (B,n,3) = (1-sqrt(u1)) v0 + sqrt(u1)(1-u2) v1 + sqrt(u1) u2 v2 of face_idx (B,n) int32 = first face whose
 * cumulative area share exceeds the face draw.  cdf: scratch (B,F) floats.  bwd overwrites grad_verts (B,V,3). */
int vpn_mesh_sample_fwd(const float* verts, const int* faces, const float* u, float* points, int* face_idx,
                        float* cdf, int B, int V, int F, int n, void* stream);
int vpn_mesh_sample_bwd(const int* faces, const float* u, const int* face_idx, const float* grad_points,
                        float* grad_verts, int B, int V, int F, int n, void* stream);
/* The same gradient as a gather with a fixed summation order (what the autograd Function uses): the samples of each mesh
 * are stably counting-sorted by face, each face sums w * grad over its run, each vertex sums its incident (face, corner)
 * terms in CSR order.  No atomics and no memset; a mesh's grad_verts is the same bits in every run and in any batch.
 * adj_offsets (V+1) int32 / adj_entries (3F) int32: vertex -> (3 * face + corner) CSR of `faces`, entries of a vertex in
 * the order the caller chooses (vpn_b200: a stable argsort of faces.flatten()).  face_idx as vpn_mesh_sample_fwd wrote
 * it.  workspace: vpn_mesh_sample_bwd_workspace_bytes(B, F, n) bytes of scratch. */
int vpn_mesh_sample_bwd_workspace_bytes(int B, int F, int n, size_t* bytes);
int vpn_mesh_sample_bwd_sorted(const int* faces, const float* u, const int* face_idx, const float* grad_points,
                               float* grad_verts, const int* adj_offsets, const int* adj_entries, void* workspace,
                               size_t workspace_bytes, int B, int V, int F, int n, void* stream);

/* ---- EMD approximation by auction: modules/loss/emd (emd_module.py:29-79, emd_cuda.cu:227-316)
 * xyz1 (B,n,3) predicted (bidders), xyz2 (B,n,3) ground truth (objects), coordinates normalised to [0,1].
 * dist (B,n) = squared distance to the assigned object, assignment (B,n) int32 (not necessarily a bijection).
 * One launch (thread-block cluster per sample); ties resolved deterministically (lowest index). */
int vpn_emd_workspace_bytes(int B, int n, size_t* bytes);
int vpn_emd_fwd(const float* xyz1, const float* xyz2, float* dist, int* assignment, void* workspace,
                size_t workspace_bytes, int B, int n, float eps, int iters, void* stream);
/* grad_xyz1 (B,n,3) = 2 grad_dist (xyz1 - xyz2[assignment]); xyz2 receives no gradient (emd_module.py:66-67). */
int vpn_emd_bwd(const float* xyz1, const float* xyz2, const int* assignment, const float* grad_dist,
                float* grad_xyz1, int B, int n, void* stream);
/* Fused loss head of train.py:188-195 / train_gcn.py:91-95: loss[b] = weight * mean_j sqrt(dist[b,j]) (IEEE sqrt), summed in an
 * order that depends on n only, so a sample's value does not depend on the batch it is computed in.  The backward takes
 * the per-sample upstream gradient grad_loss (B) and overwrites grad_xyz1 (B,n,3) in one pass, in the operation order of
 * autograd through the head followed by vpn_emd_bwd (dist == 0 gives NaN, as in the reference). */
int vpn_emd_loss_fwd(const float* dist, float weight, float* loss, float* scratch /* >= 32*B floats */, int B, int n,
                     void* stream);
int vpn_emd_loss_bwd(const float* xyz1, const float* xyz2, const int* assignment, const float* dist,
                     const float* grad_loss, float weight, float* grad_xyz1, int B, int n, void* stream);

/* ---- GCN vertex-feature pooling: modules/network/gcn.py:84-164 (train_gcn.py:121; SURVEY.md section 8f-4)
 * vpn_image_bounds: GCNModel.get_bound_of_images (gcn.py:90-133).  imgs (B,C,H,W) -> bounds (B,4) = [x lo, x hi, y lo,
 *   y hi] of the pixels whose channel sum exceeds `threshold` (0.03), as x / w * 2 - 1; the lower bound skips index 0
 *   and unset bounds stay 0 / w, as the reference's scan does.
 * vpn_points_yz_range: the per-sample max / min of gcn.py:146-150.  range (B,4) = [min z, max z, min y, max y],
 *   arg (B,4) int32 = first vertex attaining each (the backward pass routes the range's gradient there).
 * vpn_feature_pool_fwd: GCNModel.perceptual_feature_pooling (gcn.py:135-164) for ONE feature map feat (B,C,H,W):
 *   bilinear grid_sample (zeros padding, align_corners=True) at grid x = f(z), grid y = f(y), written to
 *   out[:, :, coff : coff + C] of out (B,N,Ctot) - the reference's cat + view + permute layout.  One call per map.
 * vpn_feature_pool_bwd: grad_feat (B,C,H,W) fully written; grad_grid (B,N,2) ACCUMULATED over the maps (zero it first).
 * vpn_feature_pool_points_bwd: grad_grid -> grad_pts (B,N,3) (x component 0), including the arg-min / arg-max terms. */
int vpn_image_bounds(const float* imgs, float* bounds, int B, int C, int H, int W, float threshold, void* stream);
int vpn_points_yz_range(const float* pts, float* range, int* arg, int B, int N, void* stream);
int vpn_feature_pool_fwd(const float* feat, const float* pts, const float* bounds, const float* range, float* out,
                         int B, int C, int H, int W, int N, int Ctot, int coff, void* stream);
int vpn_feature_pool_bwd(const float* feat, const float* pts, const float* bounds, const float* range,
                         const float* grad_out, float* grad_feat, float* grad_grid,
                         int B, int C, int H, int W, int N, int Ctot, int coff, void* stream);
/* The same gradient through the cell-sorted kernels (what the autograd Function uses): the vertices are counting-sorted by
 * bilinear cell once per map, a warp accumulates a cell's four texel gradients in registers and flushes them with global
 * float atomics into the zero-filled grad_feat (so the summation order, hence the last bits, can differ between runs).
 * workspace: vpn_feature_pool_bwd_workspace_bytes(B, N) bytes of scratch, reusable for every map. */
int vpn_feature_pool_bwd_workspace_bytes(int B, int N, size_t* bytes);
int vpn_feature_pool_bwd_sorted(const float* feat, const float* pts, const float* bounds, const float* range,
                                const float* grad_out, float* grad_feat, float* grad_grid, void* workspace,
                                size_t workspace_bytes, int B, int C, int H, int W, int N, int Ctot, int coff, void* stream);
int vpn_feature_pool_points_bwd(const float* pts, const float* bounds, const float* range, const int* arg,
                                const float* grad_grid, float* grad_pts, int B, int N, void* stream);

/* ---- gradient all-reduce over NVSwitch multicast (NVLS): in-place SUM of a symmetric fp32 buffer (SURVEY.md 8e)
 * multicast_ptr: multicast virtual address of the buffer (numel % 4 == 0, 16-byte aligned).  The caller brackets the
 * call with cross-rank barriers on the stream.  The reference is single process: no counterpart. */
int vpn_allreduce_nvls(void* multicast_ptr, size_t numel, int rank, int world, void* stream);
/* Self-synchronising variant: ONE launch, cross-rank barriers inside the kernel (multimem.red arrive counters in the
 * buffer tail, bounded spins), epoch in device memory - no per-call host state, capturable in a CUDA graph.  The
 * symmetric buffer is numel payload floats followed by vpn_allreduce_nvls_flag_floats() flag words that are zero on
 * every rank before the first call; multicast_ptr / local_ptr address the same buffer.  A wait that times out (4 s)
 * sets flag word vpn_allreduce_nvls_error_word() instead of hanging the GPU. */
int vpn_allreduce_nvls_flag_floats(size_t* floats);
int vpn_allreduce_nvls_error_word(void);
int vpn_allreduce_nvls_sync(void* multicast_ptr, void* local_ptr, size_t numel, int rank, int world, void* stream);

/* ---- measurement helper: achieved FP32 FMA throughput (the Chamfer roofline denominator) ----------------
 * scratch: >= 64 device floats, the first 16 finite and near 1.0.  Synchronises the stream. */
int vpn_fp32_peak_probe(float* scratch, int reps, double* tflops_ffma, double* tflops_ffma2, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VPN_B200_H */
