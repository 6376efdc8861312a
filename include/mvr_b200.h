/*
 * mvr_b200.h -- C ABI of libmvr_b200.so: the sm_100a implementation of MVTN's MVRenderer hot path.
 *
 * Boundary.  The reference (ajhamdi/MVTN, Python) reaches its native code through PyTorch3D's
 * `pytorch3d._C` extension; the entry points below are what a maintainer would bind with ctypes
 * in place of those calls (see INTEGRATION.md).  Each function cites the reference call site /
 * upstream operator it replaces.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer owned by the caller unless the comment says "host";
 *  - fp32 / int32 unless stated; row-major, innermost dimension last;
 *  - `stream` is a cudaStream_t passed as void*; every call is asynchronous on that stream, does
 *    no host synchronisation and no allocation (scratch comes from the caller's workspace);
 *  - return value: 0 ok; <0 invalid argument (see mvr_last_error_string); >0 a cudaError_t;
 *  - view n = b*M + m (flat order of util.py:509-534 batch_tensor / Meshes.extend(M));
 *  - R (n,3,3), T (n,3): PyTorch3D row-vector convention X_view = X_world R + T.
 *  - arithmetic contract for fragments: IEEE fp32, written operation order, no FMA contraction
 *    (DESIGN.md "Parity"), so pix_to_face / idx agree bit-for-bit with oracle/mvr_oracle.c.
 */
#ifndef MVR_B200_H
#define MVR_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVR_ABI_VERSION 16

/* flags */
#define MVR_PERSPECTIVE_CORRECT 1  /* [upstream] RasterizationSettings.perspective_correct (FoV persp.: True) */
#define MVR_CULL_BACKFACES 2       /* renderer.py:52,97 cull_backfaces */
#define MVR_COMPOSITE_ALPHA 4      /* AlphaCompositor instead of NormWeightedCompositor (renderer.py:11,138) */
#define MVR_RGB_PER_ELEMENT 8      /* per-vertex / per-point colours (object_color == "custom") */
#define MVR_FACES_I64 16           /* faces given as int64 (F,3) -- the reference's layout, renderer.py:68 */
#define MVR_IMAGES_BF16 32         /* images (forward) / grad_images (backward) are bfloat16 instead of float32 */
#define MVR_SCALE_IS_DIST 64       /* points: the per-view scale array holds dist, not 1/dist (see mvr_points_forward) */
/* workspace reuse hints of the mesh path (the caller vouches for them; all optional, off = always safe):             */
#define MVR_WS_KEYS_ARMED 128      /* mvr_mesh_forward: the key plane of this workspace was left re-armed by a previous
                                      mvr_mesh_forward with the SAME (B, M, H, W, K, total_verts) and MVR_WS_REARM_KEYS, and
                                      nothing but mvr_mesh_backward has touched the workspace since: skip the plane memset */
#define MVR_WS_REARM_KEYS 256      /* mvr_mesh_forward: the shade pass writes EMPTY back over every key it consumed */
#define MVR_WS_PROJECTED 512       /* mvr_mesh_backward: projected vertices / pixel table / clip flag in the workspace are
                                      those of the matching mvr_mesh_forward (same geometry, R, T): skip the re-projection */
#define MVR_IDX_SPARSE 1024        /* mvr_points_forward (K in {1,2,4,8}, hit_mask given, no zbuf / dists2 wanted): idx is written
                                      only where the pixel's hit_mask bit is set -- 4 K bytes per background pixel (~90 % of a
                                      point image) are not stored; mvr_points_backward never reads them */
#define MVR_FACES_U16 8192         /* mvr_mesh_prepare: faces given as uint16 (F,3) -- every mesh of the batch has at most 65536 vertices; half
                                      the bytes of int32 on the host-to-device copy (mvtn_b200.collate_meshes narrows when it can) */
#define MVR_CLIP_BARYCENTRIC 4096  /* [upstream] RasterizationSettings.clip_barycentric_coords (default: True iff blur_radius > 0): the
                                      fragment's barycentrics are clamped below at 0 and renormalised (BarycentricClipForward) */
#define MVR_TEST_TINY_QUEUES 0x40000000 /* tests only: shrink the scatter kernel's work queues to force their fallbacks */

/* Phong constants of DirectionalLights() / Materials() as constructed at renderer.py:190-191 */
#define MVR_AMBIENT 0.5f
#define MVR_DIFFUSE 0.3f
#define MVR_SPECULAR 0.2f
#define MVR_SHININESS 64

/* counters[] slots written by mvr_mesh_forward (device int64[MVR_NUM_COUNTERS]; the call zeroes them first) */
#define MVR_CNT_STRADDLE 0     /* faces straddling the near clip plane (clipped against it, [upstream] clip.py) */
#define MVR_CNT_BIG_FACES 1    /* faces whose pixel bbox exceeded 1024 pixels (walked by a whole CTA) */
#define MVR_NUM_COUNTERS 4

int mvr_abi_version(void);
/* thread-local description of the last non-zero return value (host string) */
const char* mvr_last_error_string(void);

/* -- measurement hooks (bench.py) ------------------------------------------------------------ */
/* number of kernels this library has launched in this process */
long long mvr_launch_count(void);
/* bracket every following launch of the named kernel (e.g. "mesh_fine_kernel") with CUDA events on
 * its launch stream; NULL disables.  mvr_profile_collect synchronises those events, returns the summed
 * device time and the number of launches, and disables collection. */
int mvr_profile_enable(const char* kernel_name);
int mvr_profile_collect(double* total_ms, int* n_launches);

/* -- host staging (renderer.py:67-68 replacement, SURVEY 8f N1) -------------------------------- */
/* HOST pointers: gather n arrays (counts[i] elements of elem_bytes each) back to back into dst with all
 * host cores; narrow_i64_to_i32 converts int64 sources to int32 on the way (faces).  No CUDA calls. */
/* number of host threads mvr_host_gather may use (0 = all); set it to cores / ranks under torchrun */
int mvr_host_set_threads(int n);
int mvr_host_gather(const void* const* srcs, const int64_t* counts, int n, void* dst, int elem_bytes,
                    int narrow_i64_to_i32);

/* One-call staging of a batch of meshes: gather the n vertex arrays (vert_counts[i] FLOATS each) into pinned_verts and
 * the n face arrays (face_counts[i] INDICES each; int64 when face_elem_bytes == 8, narrowed to int32, else int32) into
 * pinned_faces inside one parallel region, enqueueing the H2D copy of the vertices (to dev_verts, on `stream`) while the
 * faces are still being gathered, then the faces' copy (to dev_faces).  dev_* may be NULL (gather only: no CUDA call). */
int mvr_host_stage_meshes(const void* const* vert_srcs, const int64_t* vert_counts,
                          const void* const* face_srcs, const int64_t* face_counts, int n,
                          int face_elem_bytes, float* pinned_verts, int32_t* pinned_faces,
                          float* dev_verts, int32_t* dev_faces, void* stream);

/* The same, plus: the faces optionally narrowed (saturating) to uint16 ids (face_out_bytes 2: pinned_faces / dev_faces hold 2-byte
 * elements; for batches whose meshes all have at most 65536 vertices, then prepare with MVR_FACES_U16 -- a third fewer H2D bytes than
 * the int32 form), and the batch's offset table written to pinned_offs and copied to dev_offs (either may be NULL): 2n + 2 int32,
 * vertex offsets (n + 1) | face offsets (n + 1), the vert_off / face_off arguments of mvr_mesh_prepare. */
int mvr_host_stage_meshes_packed(const void* const* vert_srcs, const int64_t* vert_counts,
                                 const void* const* face_srcs, const int64_t* face_counts, int n,
                                 int face_elem_bytes, int face_out_bytes, float* pinned_verts, void* pinned_faces,
                                 int32_t* pinned_offs, float* dev_verts, void* dev_faces, int32_t* dev_offs, void* stream);

/* Asynchronous variant: _begin hands the same work to a persistent native worker thread (which selects CUDA device
 * `device` before enqueueing the copies) and returns a job id > 0 at once, so the caller can build the rest of the step
 * while the meshes are staged; _end(job) waits for it and returns its status.  Every array passed to _begin must stay
 * alive until _end returns.  One job in flight at a time (-10 otherwise). */
int mvr_host_stage_meshes_begin(const void* const* vert_srcs, const int64_t* vert_counts,
                                const void* const* face_srcs, const int64_t* face_counts, int n,
                                int face_elem_bytes, float* pinned_verts, int32_t* pinned_faces,
                                float* dev_verts, int32_t* dev_faces, int device, void* stream);
int mvr_host_stage_meshes_packed_begin(const void* const* vert_srcs, const int64_t* vert_counts,
                                       const void* const* face_srcs, const int64_t* face_counts, int n,
                                       int face_elem_bytes, int face_out_bytes, float* pinned_verts, void* pinned_faces,
                                       int32_t* pinned_offs, float* dev_verts, void* dev_faces, int32_t* dev_offs,
                                       int device, void* stream);      /* mvr_host_stage_meshes_packed on the worker */
int mvr_host_stage_meshes_end(int job);

/* -- cameras ------------------------------------------------------------------------------ */
/* look_at_view_transform(dist, elev, azim) + camera_position_from_spherical_angles
 * (renderer.py:79-80,122-123,168; ops.py:160) fused with util.py:403-420
 * check_valid_rotation_matrix: *invalid_count = number of matrices failing the check (the call owns the word: up to 4096 views one
 * CTA counts and stores it, no memset; above, memset + atomics).  azim/elev in degrees, n = B*M.  C (n,3) = camera centres (may be NULL). */
int mvr_look_at_forward(const float* azim, const float* elev, const float* dist, int n, float* R,
                        float* T, float* C, int* invalid_count, void* stream);
/* The same with the flag sent to the host behind the kernel: host_flag (pinned int) receives *invalid_count -- stored by the kernel
 * itself when n <= 4096 and the word is device-addressable (pinned memory under unified addressing), by an asynchronous copy
 * otherwise -- and `event` (cudaEvent_t) is recorded behind it: the rotation guard (ops.py:156-165) waits for that event only. */
int mvr_look_at_forward_flagged(const float* azim, const float* elev, const float* dist, int n, float* R, float* T, float* C,
                                int* invalid_count, int* host_flag, void* event, void* stream);
/* autograd backward of the above: (gR, gT, gC) -> (g_azim, g_elev, g_dist); any g* input may be NULL */
int mvr_look_at_backward(const float* azim, const float* elev, const float* dist, int n,
                         const float* gR, const float* gT, const float* gC, float* g_azim,
                         float* g_elev, float* g_dist, void* stream);

/* -- consumer side: the regulariser applied to the rendered views ------------------------------ */
/* ops.py:138-178 regualarize_rendered_views (called right behind the renderer: run_mvtn.py:186,244, Trainer_mvt.py:104) as ONE
 * gather: view dropout (dropout2d on the 5-D (B,M,3,H,W) tensor = a per-view factor 0 or 1/(1-p): view_scale (N) or NULL),
 * batchwise horizontal flip, and ReplicationPad2d(pad) + RandomCrop(H) = a shift by (shift_y, shift_x) = crop offset - pad with
 * edge replication:  out[n,c,y,x] = view_scale[n] * in[n,c,clamp(y+shift_y), fx(clamp(x+shift_x))], fx(u) = flip ? W-1-u : u.
 * images / out: (N,C,H,W) contiguous, fp32 or bfloat16 [MVR_IMAGES_BF16], out != images.  The caller draws the random decisions
 * (mvtn_b200/augment.py draws them with the reference's own torch calls). */
int mvr_images_regularize_forward(const void* images, int N, int C, int H, int W, const float* view_scale, int flip,
                                  int shift_y, int shift_x, int flags, void* out, void* stream);
/* its adjoint: grad_out (N,C,H,W) -> grad_in (N,C,H,W), fully written */
int mvr_images_regularize_backward(const void* grad_out, int N, int C, int H, int W, const float* view_scale, int flip,
                                   int shift_y, int shift_x, int flags, void* grad_in, void* stream);

/* -- meshes ------------------------------------------------------------------------------- */
/* Device-resident packed geometry built once per batch of objects (replaces Meshes(...),
 * Textures(verts_rgb) and verts_normals_packed(): renderer.py:67-77 + [upstream] meshes.py). */
size_t mvr_mesh_geometry_bytes(int64_t total_verts, int64_t total_faces);
/* verts (Vtot,3); faces (Ftot,3) int32, int64 [MVR_FACES_I64] or uint16 [MVR_FACES_U16], mesh-local vertex ids;
 * vert_off / face_off (B+1) int32 prefix sums (device); vert_rgb (Vtot,3) or NULL. */
int mvr_mesh_prepare(const float* verts, const void* faces, const int* vert_off, const int* face_off,
                     int B, int64_t total_verts, int64_t total_faces, int max_faces,
                     const float* vert_rgb, int flags, void* geometry, size_t geometry_bytes,
                     void* stream);
/* copy of the per-vertex unit normals (Vtot,3) out of a prepared geometry (tests / callers) */
int mvr_mesh_get_normals(const void* geometry, int64_t total_verts, int64_t total_faces,
                         float* normals, void* stream);

/* backward of the vertex normals ([upstream] meshes.py Meshes._compute_vertex_normals: per-corner area-weighted cross
 * products, index_add, F.normalize(eps 1e-6)) for callers that want gradients w.r.t. mesh vertices: grad_normals (Vtot,3)
 * = d loss / d unit normals (as accumulated by mvr_mesh_backward; CONSUMED -- overwritten with the gradient w.r.t. the
 * un-normalised sums), grad_verts (Vtot,3) ACCUMULATED with atomics.  `geometry` as left by mvr_mesh_prepare. */
int mvr_mesh_normals_backward(const void* geometry, const int* vert_off, const int* face_off, int B,
                              int64_t total_verts, int64_t total_faces, int max_faces, float* grad_normals,
                              float* grad_verts, void* stream);

/* scratch for one forward or backward call: projected vertices of every view (16 B * M * total_verts), the
 * pixel-centre table, the 64-bit key plane(s) (one for K == 1, two for K > 1) and the backward partial sums */
size_t mvr_mesh_workspace_bytes(int B, int M, int H, int W, int K, int64_t total_verts, int64_t total_faces);
/* MeshRenderer(MeshRasterizer, HardPhongShader)(meshes.extend(M), cameras, lights)
 * (renderer.py:89-113; [upstream] _C.rasterize_meshes + interp_face_attrs + phong_shading +
 * hard_rgb_blend).
 *   blur_radius >= 0 ([upstream] RasterizationSettings.blur_radius, squared NDC units; renderer.py:91 passes 0): with a positive
 *   radius a face is also a fragment of the pixels closer than it to one of its edges, `dists` carries the SIGNED squared edge
 *   distance (negative inside) and, with MVR_CLIP_BARYCENTRIC, `bary` the clipped barycentrics -- the fragments the soft
 *   shaders blend (mvr_mesh_soft_blend_forward); the image written here stays the hard-shaded nearest fragment.
 *   Cc (n,3) camera centres; light (1,3) if light_stride == 0 else (n,3) with stride 3;
 *   obj_rgb (3) uniform colour (ignored when the geometry holds per-vertex colours); bg_rgb (3);
 *   k00,k11: FoV projection scale (1/tan(fov/2)); z_clip: near clip plane in view space ([upstream] MeshRasterizer:
 *   znear / 2) -- faces entirely behind it are culled, faces crossing it are clipped into one or two triangles and their
 *   fragments mapped back to the original face ([upstream] clip.py); z_clip < 0 disables both;
 *   K = faces_per_pixel; max_verts / max_faces = largest per-object counts (grid sizing).
 *   out_mean_std: HOST float[6] = per-channel mean[3], std[3], or NULL.  Consumer-side fusion (SURVEY 8f N2):
 *   the images are written as (x - mean_c) / std_c -- viewGCN/tools/Trainer_mvt.py:41-49 Normalize -- and, with
 *   MVR_IMAGES_BF16, rounded to bfloat16, i.e. in the layout and dtype the CNN consumes; NULL + fp32 = the reference.
 * outputs: images (n,3,H,W); pix_to_face (n,H,W,K) view-local face ids, -1 empty;
 *          optional zbuf (n,H,W,K), bary (n,H,W,K,3), dists (n,H,W,K) (NULL to skip);
 *          counters: device int64[MVR_NUM_COUNTERS] or NULL (zeroed by the call, then counted into). */
int mvr_mesh_forward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                     int64_t total_verts, int64_t total_faces, int max_verts, int max_faces,
                     const float* R, const float* T, const float* Cc, const float* light,
                     int light_stride, const float* obj_rgb, const float* bg_rgb, float k00, float k11,
                     float z_clip, float blur_radius, int H, int W, int K, int flags, const float* out_mean_std, void* images,
                     int* pix_to_face, float* zbuf, float* bary, float* dists, int64_t* counters,
                     void* workspace, size_t workspace_bytes, void* stream);
/* backward of the above w.r.t. the cameras ([upstream] _C.rasterize_meshes_backward + autograd
 * of shading/projection): grad_images (n,3,H,W) -> gR (n,3,3), gT (n,3), gC (n,3);
 * optional grad_verts (Vtot,3) (projection + interpolated-position paths) and grad_normals
 * (Vtot,3) (gradient w.r.t. the per-vertex unit normals), both ACCUMULATED with atomics
 * (caller zero-fills).  z_clip: the forward's value.  out_mean_std / MVR_IMAGES_BF16 as in the forward: grad_images is then the cotangent of
 * the normalised (bfloat16) tensor. */
int mvr_mesh_backward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                      int64_t total_verts, int64_t total_faces, int max_verts, const float* R,
                      const float* T, const float* Cc, const float* light, int light_stride,
                      const float* obj_rgb, float k00, float k11, float z_clip, int H, int W, int K, int flags,
                      const float* out_mean_std, const int* pix_to_face, const void* grad_images, float* gR,
                      float* gT, float* gC,
                      float* grad_verts, float* grad_normals, void* workspace, size_t workspace_bytes,
                      void* stream);
/* The same for cameras that came from mvr_look_at_forward(azim, elev, dist) (renderer.py:161-166): the kernel that sums a view's
 * partial camera gradients also applies mvr_look_at_backward to them, so the chain ends in g_azim, g_elev, g_dist (n) with one
 * launch and one call less.  gR / gT / gC: optional copies of the camera gradients (NULL: not stored). */
int mvr_mesh_backward_angles(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                             int64_t total_verts, int64_t total_faces, int max_verts, const float* R, const float* T,
                             const float* C, const float* light, int light_stride, const float* obj_rgb, float k00,
                             float k11, float z_clip, int H, int W, int K, int flags, const float* out_mean_std,
                             const int* pix_to_face, const void* grad_images, const float* azim, const float* elev,
                             const float* dist, float* g_azim, float* g_elev, float* g_dist, float* gR, float* gT,
                             float* gC, float* grad_verts, float* grad_normals, void* workspace, size_t workspace_bytes,
                             void* stream);
/* mvr_mesh_backward that also returns the gradient w.r.t. the colours (texture fitting, colour attacks).  grad_rgb: with
 * per-vertex colours (MVR_RGB_PER_ELEMENT) (Vtot,3), ACCUMULATED with atomics (caller zero-fills); with one object colour (3),
 * WRITTEN by a fixed-order sum (per-warp partials, fp64 per view, fixed order over the views: bit-reproducible).  NULL: exactly
 * mvr_mesh_backward.  The camera gradients are the same, bit for bit, with and without it. */
int mvr_mesh_backward_rgb(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                          int64_t total_verts, int64_t total_faces, int max_verts, const float* R,
                          const float* T, const float* Cc, const float* light, int light_stride,
                          const float* obj_rgb, float k00, float k11, float z_clip, int H, int W, int K, int flags,
                          const float* out_mean_std, const int* pix_to_face, const void* grad_images, float* gR,
                          float* gT, float* gC,
                          float* grad_verts, float* grad_normals, void* workspace, size_t workspace_bytes,
                          void* stream, float* grad_rgb);

/* -- hard depth ([upstream] HardDepthShader: the nearest fragment's zbuf, zfar where no face covers the pixel) -------------- */
/* The depth of the nearest fragment -- the (z, face) winner of the hard rasterizer of mvr_mesh_forward with K = 1, bit for bit its
 * zbuf[..., 0] (near-plane clipping included) -- without shading: depth (n,1,H,W) fp32 = that z, depth_background where no face
 * covers the pixel; pix_to_face (n,H,W) view-local face ids, -1 empty; counters as in mvr_mesh_forward (or NULL).  flags:
 * MVR_PERSPECTIVE_CORRECT, MVR_CULL_BACKFACES and the workspace hints; MVR_IMAGES_BF16 / MVR_CLIP_BARYCENTRIC are rejected (-11).
 * The workspace is mvr_mesh_workspace_bytes(B, M, H, W, 1, ...). */
int mvr_mesh_depth_forward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                           int64_t total_verts, int64_t total_faces, int max_verts, int max_faces,
                           const float* R, const float* T, float k00, float k11, float z_clip, float depth_background,
                           int H, int W, int flags, float* depth, int* pix_to_face, int64_t* counters,
                           void* workspace, size_t workspace_bytes, void* stream);
/* its backward: grad_depth (n,1,H,W) -> gR (n,3,3), gT (n,3), WRITTEN (fixed-order sums: bit-reproducible, and the same with or
 * without grad_verts); grad_verts (Vtot,3) or NULL, ACCUMULATED with atomics (caller zero-fills).  Background pixels and
 * silhouette edges carry no gradient.  z_clip and flags: those of the forward. */
int mvr_mesh_depth_backward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                            int64_t total_verts, int64_t total_faces, int max_verts, const float* R, const float* T,
                            float k00, float k11, float z_clip, int H, int W, int flags, const int* pix_to_face,
                            const float* grad_depth, float* gR, float* gT, float* grad_verts, void* workspace,
                            size_t workspace_bytes, void* stream);

/* -- soft shading of K fragments per pixel (SURVEY 8f N3; renderer.py:4-6 SoftPhongShader / SoftSilhouetteShader) -------- */
/* mode 0: [upstream] blending.softmax_rgb_blend over per-fragment Phong colours (SoftPhongShader; sigma, gamma = BlendParams,
 * znear / zfar = the camera's 1 / 100); mode 1: blending.sigmoid_alpha_blend (SoftSilhouetteShader: RGB = 1, alpha = 1 -
 * prod(1 - sigmoid(-dists / sigma))).  Input: the fragments mvr_mesh_forward wrote with K = faces_per_pixel and
 * blur_radius > 0 (pix_to_face, zbuf, bary, dists: (n,H,W,K[,3])); output rgba (n,4,H,W) fp32.  sigma >= FLT_MIN: a
 * subnormal sigma, where 1 / sigma overflows, is refused with -7 as sigma <= 0 is; gamma > 0, zfar > znear. */
int mvr_mesh_soft_blend_forward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                int64_t total_verts, int64_t total_faces, const float* Cc, const float* light,
                                int light_stride, const float* obj_rgb, const float* bg_rgb, int H, int W, int K, int flags,
                                int mode, float sigma, float gamma, float znear, float zfar, const int* pix_to_face,
                                const float* zbuf, const float* bary, const float* dists, float* rgba, void* stream);
/* backward of rasterizer (incl. grad_zbuf, grad_dists, clipped barycentrics: [upstream] RasterizeMeshesBackward) + blend +
 * Phong + projection: grad_rgba (n,4,H,W) -> gR, gT, gC (deterministic: fixed-order sums);
 * optional grad_verts (Vtot,3) (projection + interpolated-position paths) and grad_normals (Vtot,3) (gradient w.r.t. the
 * per-vertex unit normals, to be chained with mvr_mesh_normals_backward), both ACCUMULATED with atomics (caller zero-fills;
 * the summation order is not fixed).  NULL for both: camera gradients only.  Mode 1 (silhouette) produces no normal gradient:
 * grad_normals stays untouched.  Fragments are recomputed from pix_to_face;
 * z_clip and blur_radius must be those of the mvr_mesh_forward call that produced it: a fragment of a face crossing the
 * near plane z_clip is recomputed on the clipped sub-triangle the forward kept, and the chain runs through the clipping
 * ([upstream] clip.py) to the vertices of the original face.  -1 entries of a pixel's K-list are skipped, as
 * mvr_mesh_soft_blend_forward does.  sigma, gamma, znear, zfar: checked as by mvr_mesh_soft_blend_forward (a subnormal
 * sigma is refused). */
int mvr_mesh_soft_backward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                           int64_t total_verts, int64_t total_faces, int max_verts, const float* R, const float* T,
                           const float* Cc, const float* light, int light_stride, const float* obj_rgb,
                           const float* bg_rgb, float k00, float k11, float z_clip, float blur_radius, int H, int W, int K,
                           int flags, int mode, float sigma, float gamma, float znear, float zfar, const int* pix_to_face,
                           const float* grad_rgba, float* gR, float* gT, float* gC, float* grad_verts, float* grad_normals,
                           void* workspace, size_t workspace_bytes, void* stream);
/* mvr_mesh_soft_backward that also returns the colour gradient, grad_rgb as in mvr_mesh_backward_rgb.  Mode 1 (silhouette)
 * does not depend on the colours: a (3) grad_rgb is written with zeros, a (Vtot,3) one stays untouched. */
int mvr_mesh_soft_backward_rgb(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                               int64_t total_verts, int64_t total_faces, int max_verts, const float* R, const float* T,
                               const float* Cc, const float* light, int light_stride, const float* obj_rgb,
                               const float* bg_rgb, float k00, float k11, float z_clip, float blur_radius, int H, int W, int K,
                               int flags, int mode, float sigma, float gamma, float znear, float zfar, const int* pix_to_face,
                               const float* grad_rgba, float* gR, float* gT, float* gC, float* grad_verts, float* grad_normals,
                               void* workspace, size_t workspace_bytes, void* stream, float* grad_rgb);
/* -- soft depth ([upstream] SoftDepthShader) ------------------------------------------------------------------------------ */
/* The K fragments mvr_mesh_forward wrote with K = faces_per_pixel and blur_radius > 0 (pix_to_face, zbuf, dists: (n,H,W,K)),
 * blended into depth (n,1,H,W) fp32: over the valid entries of a pixel in list order, p_k = sigmoid(-dists_k / sigma),
 * c_k = sum_{j <= k} p_j, m_k = min(c_k, 1); depth = sum_k (m_k - m_prev) zbuf_k + (1 - m_last) depth_background.  A pixel with
 * no fragment holds depth_background (any finite value).  sigma >= FLT_MIN (BlendParams.sigma; a subnormal sigma is refused,
 * as by the other soft entry points); gamma does not enter. */
int mvr_mesh_soft_depth_forward(int B, int M, int H, int W, int K, float sigma, float depth_background, const int* pix_to_face,
                                const float* zbuf, const float* dists, float* depth, void* stream);
/* its backward through the rasterizer (grad_zbuf, grad_dists, clipped barycentrics, near-plane clipping, as
 * mvr_mesh_soft_backward): grad_depth (n,1,H,W) -> gR (n,3,3), gT (n,3), WRITTEN (fixed-order sums: bit-reproducible, and the
 * same with or without grad_verts); grad_verts (Vtot,3) or NULL, ACCUMULATED with atomics (caller zero-fills).  The depth does
 * not depend on the camera centres or the colours.  z_clip, blur_radius, K, flags and sigma: those of the forward;
 * MVR_IMAGES_BF16 is rejected (-11).  The workspace is mvr_mesh_workspace_bytes(B, M, H, W, K, ...). */
int mvr_mesh_soft_depth_backward(const void* geometry, const int* vert_off, const int* face_off, int B, int M,
                                 int64_t total_verts, int64_t total_faces, int max_verts, const float* R, const float* T,
                                 float k00, float k11, float z_clip, float blur_radius, int H, int W, int K, int flags,
                                 float sigma, float depth_background, const int* pix_to_face, const float* grad_depth,
                                 float* gR, float* gT, float* grad_verts, void* workspace, size_t workspace_bytes, void* stream);

/* -- point clouds --------------------------------------------------------------------------- */
/* scratch for one forward or backward call (forward: pixel table + per-view projected points, tile lists, or for K not
 * in {1,2,4,8} a K-slot key plane; backward: per-tile partial sums) */
size_t mvr_points_workspace_bytes(int B, int Np, int M, int H, int W, int K, double radius);
/* number of uint32 words of the optional hit mask: (n, H, ceil(W/32)), bit x%32 of word x/32 = pixel (y, x) is
 * covered by at least one point */
size_t mvr_points_hit_mask_words(int B, int M, int H, int W);
/* PointsRenderer(PointsRasterizer, compositor)(Pointclouds.extend(M).scale_(1/dist))
 * (renderer.py:119-150; [upstream] _C.rasterize_points + accum_weightedsumnorm /
 * accum_alphacomposite + background).  points (B,Np,3); rgb (3) or (B*Np,3) [MVR_RGB_PER_ELEMENT];
 * inv_dist (n) = 1/dist, the scale of renderer.py:142 -- or dist itself with MVR_SCALE_IS_DIST (the kernels then take
 * the IEEE reciprocal torch's `1.0 / dist` takes, and the backward returns d/d dist in g_inv_dist); radius in NDC; K = points_per_pixel; out_mean_std / MVR_IMAGES_BF16 as in mvr_mesh_forward.
 * outputs: images (n,3,H,W); idx (n,H,W,K) cloud-local point ids (-1 empty); optional zbuf,
 * dists2 (n,H,W,K); optional hit_mask (mvr_points_hit_mask_words words), which lets the backward pass skip
 * the ~90 % background pixels without reading idx.
 * For K = 2 and K = 4, idx must be aligned to 4*K bytes (a pixel's ids are stored as one vector): a misaligned idx, e.g. a
 * slice of a larger int32 buffer, is rejected with status -10 before any launch.  mvr_points_backward takes any idx. */
int mvr_points_forward(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                       const float* T, const float* inv_dist, double radius, const float* bg_rgb,
                       int H, int W, int K, int flags, const float* out_mean_std, void* images, int* idx,
                       float* zbuf, float* dists2, uint32_t* hit_mask, void* workspace, size_t workspace_bytes,
                       void* stream);
/* backward ([upstream] accum_*_backward + _C.rasterize_points_backward + autograd of the
 * projection): grad_images -> gR (n,3,3), gT (n,3), g_inv_dist (n); optional grad_points
 * (B,Np,3) and grad_rgb ((3) or (B*Np,3)) ACCUMULATED with atomics (caller zero-fills).
 * hit_mask: the forward's mask or NULL (then idx[..., 0] >= 0 is read for every pixel). */
int mvr_points_backward(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                        const float* T, const float* inv_dist, double radius, int H, int W, int K,
                        int flags, const float* out_mean_std, const int* idx, const uint32_t* hit_mask,
                        const void* grad_images, float* gR, float* gT, float* g_inv_dist, float* grad_points, float* grad_rgb,
                        void* workspace, size_t workspace_bytes, void* stream);
/* The same for a caller whose cameras came from mvr_look_at_forward(azim, elev, dist) and whose clouds are scaled by 1 / dist
 * (MVR_SCALE_IS_DIST, the scale array = dist: renderer.py:122-123,142): the last kernel also applies the camera backward
 * (mvr_look_at_backward) and the scale term, so the chain ends in g_azim, g_elev, g_dist (n) with one launch and one call less
 * (SURVEY 8f N4).  gR / gT: optional copies of the camera gradients (NULL: not stored). */
int mvr_points_backward_angles(const float* points, const float* rgb, int B, int Np, int M, const float* R,
                               const float* T, const float* azim, const float* elev, const float* dist, double radius,
                               int H, int W, int K, int flags, const float* out_mean_std, const int* idx,
                               const uint32_t* hit_mask, const void* grad_images, float* g_azim, float* g_elev,
                               float* g_dist, float* gR, float* gT, float* grad_points, float* grad_rgb, void* workspace,
                               size_t workspace_bytes, void* stream);
/* Hard depth of a point cloud: the nearest point's view-space z (the (z, index) winner of mvr_points_forward, bit for bit its
 * zbuf[..., 0]) -- independent of K and of the compositor --, depth_background where no point covers the pixel.  Outputs:
 * depth (n,1,H,W) fp32, idx (n,H,W) (-1 empty), hit_mask (required: the backward reads it).  flags: MVR_SCALE_IS_DIST only;
 * MVR_IMAGES_BF16 / MVR_IDX_SPARSE are rejected (-11).  The workspace is mvr_points_workspace_bytes(B, Np, M, H, W, 1, radius). */
int mvr_points_depth_forward(const float* points, int B, int Np, int M, const float* R, const float* T, const float* inv_dist,
                             double radius, float depth_background, int H, int W, int flags, float* depth, int* idx,
                             uint32_t* hit_mask, void* workspace, size_t workspace_bytes, void* stream);
/* its backward: grad_depth (n,1,H,W) -> gR (n,3,3) (only its third column is non-zero), gT (n,3) (only z), g_inv_dist (n) (d/d dist
 * with MVR_SCALE_IS_DIST), WRITTEN (fixed-order sums); grad_points (B,Np,3) or NULL, ACCUMULATED with atomics (caller zero-fills). */
int mvr_points_depth_backward(const float* points, int B, int Np, int M, const float* R, const float* T, const float* inv_dist,
                              double radius, int H, int W, int flags, const int* idx, const uint32_t* hit_mask,
                              const float* grad_depth, float* gR, float* gT, float* g_inv_dist, float* grad_points,
                              void* workspace, size_t workspace_bytes, void* stream);
/* Splat depth of a point cloud ([upstream] SoftDepthShader's blend with the splat weight in place of the sigmoid): over the K =
 * points_per_pixel nearest points of a pixel, in the (z, index) order of mvr_points_forward's idx at the same K, nearest first:
 * alpha_k = 1 - d2_k / r^2 (d2: squared NDC distance of the point's projection to the pixel centre; r^2 the double radius * radius
 * rounded to fp32, the compositors' weight radius; not clamped), c_k = sum_{j <= k} alpha_j, m_k = min(c_k, 1);
 * depth = sum_k (m_k - m_prev) z_k + (1 - m_last) depth_background, z_k the point's view-space z (the rasterizer's zbuf), the sum
 * stopping after the first entry with c_k > 1.  A pixel with no point holds depth_background (any finite value, else -7).
 * Outputs: depth (n,1,H,W) fp32, idx (n,H,W,K) (-1 empty; aligned to 4*K bytes for K = 2, 4, else -10), hit_mask (required: the
 * backward reads it).  flags: MVR_SCALE_IS_DIST only; MVR_IMAGES_BF16, MVR_IDX_SPARSE, MVR_COMPOSITE_ALPHA and MVR_RGB_PER_ELEMENT
 * are rejected (-11).  The workspace is mvr_points_workspace_bytes(B, Np, M, H, W, K, radius) (smaller: -8).  Every check is made
 * before any launch. */
int mvr_points_splat_depth_forward(const float* points, int B, int Np, int M, const float* R, const float* T,
                                   const float* inv_dist, double radius, float depth_background, int H, int W, int K,
                                   int flags, float* depth, int* idx, uint32_t* hit_mask,
                                   void* workspace, size_t workspace_bytes, void* stream);
/* its backward, with g = grad_depth of the pixel: d/d z_k = g (m_k - m_prev); Z_stop = z of the first entry with c > 1, else
 * depth_background; d/d alpha_j = g (z_j - Z_stop) for the entries with c_j <= 1, 0 past them; d alpha / d d2 = -1 / r^2.
 * -> gR (n,3,3), gT (n,3), g_inv_dist (n) (d/d dist with MVR_SCALE_IS_DIST), WRITTEN (fixed-order sums: bit-reproducible, and the
 * same with or without grad_points); grad_points (B,Np,3) or NULL, ACCUMULATED with atomics (caller zero-fills).  Arguments as the
 * forward's, whose idx and hit_mask it reads. */
int mvr_points_splat_depth_backward(const float* points, int B, int Np, int M, const float* R, const float* T,
                                    const float* inv_dist, double radius, float depth_background, int H, int W, int K,
                                    int flags, const int* idx, const uint32_t* hit_mask, const float* grad_depth,
                                    float* gR, float* gT, float* g_inv_dist, float* grad_points,
                                    void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MVR_B200_H */
