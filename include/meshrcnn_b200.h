/* meshrcnn_b200 -- C ABI of the B200-native (sm_100a) Mesh R-CNN voxel-to-mesh refinement hot path.
 *
 * The reference (alondj/Mesh_R-CNN_Computer_Vision_project) has no FFI layer: its boundary is the Python module
 * API of meshRCNN/layers.py, meshRCNN/loss_functions.py and utils/mesh_sampling.py.  The Python package
 * `meshrcnn_b200` mirrors that API and calls the entry points below through ctypes from
 * torch.autograd.Function.forward/backward (see INTEGRATION.md for the binding a maintainer adds).
 *
 * Conventions
 *   - every pointer is a raw *device* pointer unless the name ends in _host; PyTorch (the caller) owns and
 *     allocates all inputs, outputs and workspaces -- the library never allocates, frees or caches memory and
 *     keeps no mutable global state;
 *   - `stream` is a cudaStream_t (the caller's current stream); no entry point synchronises;
 *   - return value 0 = success; otherwise an MRB_ERR_* code, with a message from mrb_last_error()
 *     (thread-local);
 *   - indices at the reference API are int64; "32" suffixed buffers are the int32 CSR copies used internally;
 *   - all floating-point buffers are fp32 unless stated otherwise.
 */
#ifndef MESHRCNN_B200_H
#define MESHRCNN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MRB_VERSION 100

int mrb_version(void);
const char* mrb_last_error(void);
int mrb_device_info(int* sm_major, int* sm_minor, int* num_sms);
/* FP32 FMA issue-rate microbenchmark (the measured peak of the FP32-issue-bound k-NN kernels, SURVEY.md 8d): launches
 * `blocks` CTAs of 256 threads running `iters` x 128 dependent-chain FMAs each and returns the flop count of the launch
 * (2 per FMA), or -1 on error; the caller times it with CUDA events.  out: 1 float of device scratch. */
long long mrb_fma_peak(float* out, int iters, int blocks, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Cubify  -- replaces Cubify.forward, reference meshRCNN/layers.py:403-484.
 *
 * Two phases because output sizes are data dependent and the module API returns Python lists
 * (layers.py:445,448,484):
 *   1. mrb_cubify_count  : threshold (strict >, fp32; from_logits != 0: the grid holds the voxel head's logits and
 *        sigmoid(logit) > threshold is tested, SURVEY 8 f-1), exposed-face flags, per-block counts, scans.
 *        meta (int64, 4 + 4*B entries): [0]=total vertices, [1]=total faces, [2]=directed edges E, [3]=0,
 *        then v_count[B], f_count[B], v_offset[B], f_offset[B].
 *   2. (caller copies meta to the host -- the only synchronisation -- and allocates the outputs)
 *   3. mrb_cubify_emit   : vertices (b,z,y,x order, coordinates (z, x, -y), layers.py:447,465-467),
 *        faces (b,dir,z,y,x order, 2 per quad, per-mesh local ids, layers.py:441-443,481-483),
 *        adjacency adj[2][E] sorted by (row, col) (layers.py:469-478) + its CSR form rowptr/col32.
 *        vert_mesh[v] = mesh id of vertex v; vert_aux = 8 bytes per vertex of scratch.
 * workspace: mrb_cubify_workspace_bytes(B,Z,Y,X) bytes, shared by both phases (contents must be preserved).
 * An all-empty batch yields meta[1] == 0; the Python layer raises ValueError("empty grid") like layers.py:434-435.
 */
long long mrb_cubify_workspace_bytes(int B, int Z, int Y, int X);
int mrb_cubify_count(const float* probs, int B, int Z, int Y, int X, float threshold, int from_logits, void* workspace,
                     long long* meta, void* stream);
int mrb_cubify_emit(int B, int Z, int Y, int X, void* workspace, const long long* meta, long long SV, long long SF,
                    long long E, float* verts, long long* faces, long long* adj, int32_t* rowptr, int32_t* col32,
                    int32_t* vert_mesh, void* vert_aux, void* stream);
/* The same two phases with a choice of quad placement; mrb_cubify_count / mrb_cubify_emit are these with topology 0.
 *   topology 0 (reference): the reference's corner table, bit-exact -- dirs 2/3 place the quad on the side away from the
 *     empty neighbour and c0..c3 are in lattice order, so the two triangles overlap with opposite winding.
 *   topology 1 (watertight): each quad on the side of the empty neighbour, corners cyclic from its lowest lattice corner,
 *     both triangles wound outward ((c1-c0) x (c2-c0) toward the empty neighbour): a closed surface per mesh whose fp64
 *     signed volume equals its voxel count.  Same face flags, orders, coordinates, counts of faces and workspace size.
 * Any other topology is rejected before a launch.  Precondition: the emit gets the topology the count got (the count's
 * lattice masks in the workspace, hence its vertex and edge counts, depend on it). */
int mrb_cubify_count_topo(const float* probs, int B, int Z, int Y, int X, float threshold, int from_logits, int topology,
                          void* workspace, long long* meta, void* stream);
int mrb_cubify_emit_topo(int B, int Z, int Y, int X, void* workspace, const long long* meta, long long SV, long long SF,
                         long long E, float* verts, long long* faces, long long* adj, int32_t* rowptr, int32_t* col32,
                         int32_t* vert_mesh, void* vert_aux, int topology, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Voxel-head tail (SURVEY 8 f-1) -- replaces nn.Sigmoid at the end of VoxelBranch (meshRCNN/layers.py:487-506) + voxel_loss
 * (meshRCNN/loss_functions.py:10-14) as one pass over the logits: loss_out[0] = mean BCE(sigmoid(x), target) with torch's
 * clamp of the log terms at -100 (from_logits != 0; probs_out, optional, receives the probabilities) or
 * mean BCE(x, target) on probabilities (from_logits == 0).  acc: 1 double of scratch.  Backward: gx = *g / n * dBCE/dx.
 */
int mrb_voxel_bce_fwd(const float* x, const float* target, long long n, int from_logits, float* probs_out, double* acc,
                      float* loss_out, void* stream);
int mrb_voxel_bce_bwd(const float* x, const float* target, long long n, int from_logits, const float* g, float* gx,
                      void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Graph utilities.
 * mrb_coo_to_csr: 2 x E int64 COO (any order) -> CSR rowptr[n+1] / col[E] (int32); transpose != 0 builds the CSR
 *   of the transposed matrix.  Row-sorted input keeps its edge order (deterministic); otherwise edges of a row
 *   are placed with an atomic cursor.  workspace: 2*(n+1)+2 int32.
 * mrb_csr_gather_fwd: out[i,:] = act(self[i,:] + sum_{j in row i} nbr[col[j],:]); `self` may be NULL; relu != 0
 *   applies max(.,0).  Replaces aggregate_neighbours (reference meshRCNN/utils.py:52-57) and, with self/relu,
 *   the add + ReLU of GraphConv.forward (meshRCNN/layers.py:63-68).  The backward of the aggregation is the same
 *   call on the transposed CSR.
 * mrb_relu_mask: gz = gout * (act > 0)  (backward of the ReLU at layers.py:68).
 * mrb_segment_ids: ids[i] = s such that offsets[s] <= i < offsets[s+1]  (vertex -> mesh map from v_index).
 */
int mrb_coo_to_csr(const long long* adj, long long E, int n, int transpose, int32_t* rowptr, int32_t* col,
                   int32_t* workspace, void* stream);
int mrb_csr_gather_fwd(const int32_t* rowptr, const int32_t* col, int n, const float* self, int ld_self,
                       const float* nbr, int ld_nbr, int D, int relu, float* out, int ld_out, void* stream);
int mrb_relu_mask(const float* gout, int ld_g, const float* act, int ld_a, int n, int D, float* gz, int ld_z,
                  void* stream);
int mrb_segment_ids(const int32_t* offsets, int nseg, int n, int32_t* ids, void* stream);
/* Fused backward of GraphConv's add + ReLU + aggregation (layers.py:63-68): gy[:, 0:D] = gz, gy[:, D:2D] = A^T gz with
 * gz = gout * (act > 0) formed on the fly (gout may be a strided view: ld_g >= D). */
int mrb_graphconv_bwd_gather(const int32_t* rowptr_t, const int32_t* col_t, int n, const float* gout, int ld_g,
                             const float* act, int ld_a, int D, float* gy, void* stream);
/* Column concatenation of up to three row-major matrices (torch.cat(dim=1) of the stage inputs, reference
 * meshRCNN/layers.py:160-165,241-252,321-334) into rows of pitch ld_out >= w0 + w1 + w2 floats; the pad columns are
 * zero-filled.  A pitch that is a multiple of 4 keeps every row 16-byte aligned for the tcgen05 projection's producers. */
int mrb_concat_cols(const float* s0, int w0, int ld0, const float* s1, int w1, int ld1, const float* s2, int w2, int ld2,
                    int n, float* out, int ld_out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Dense contraction  C = op(A) * op(B) + beta * C  (row-major fp32, exact fp32 accumulate on the CUDA cores).
 * Replaces torch.mm / nn.Linear at reference meshRCNN/layers.py:54,57,93,155,230,255,335 and their autograd.
 */
int mrb_sgemm(int transA, int transB, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
              float beta, float* C, int ldc, void* stream);

/* Tensor-core path (tcgen05.mma kind::tf32, accumulators in TMEM, 3xTF32 split => fp32-level accuracy) for the
 * activation x weight products  C[M x N] = A[M x K] * B[K x N]  with M = number of vertices.
 *   mrb_gemm_tc_pack  builds the weight image once per call: logical element B(k, n) = src[k*stride_k + n*stride_n],
 *                     optionally taken from a second source beyond `split_at` along n (split_axis = 1) or k
 *                     (split_axis = 2) -- this is how [W0 | W1] (GraphConv forward, layers.py:54,57) and its transpose
 *                     (backward) are formed without a concatenation.  image: mrb_gemm_tc_image_bytes(K, N) bytes, 16 B aligned.
 *   mrb_gemm_tc       A fp32 row-major (lda >= K), C fp32 row-major (ldc >= N).
 */
long long mrb_gemm_tc_image_bytes(int K, int N);
int mrb_gemm_tc_pack(const float* src0, const float* src1, long long stride_k, long long stride_n, int split_axis,
                     int split_at, int K, int N, void* image, void* stream);
/* Both weight images of one GraphConv (w0, w1: K x D row-major) in a single launch: image_fwd = operand of
 * x @ [W0 | W1] (mrb_gemm_tc_image_bytes(K, 2D) bytes), image_bwd = operand of [gz | A^T gz] @ [W0 | W1]^T
 * (mrb_gemm_tc_image_bytes(2D, K) bytes). */
int mrb_gemm_tc_pack_graphconv(const float* w0, const float* w1, int K, int D, void* image_fwd, void* image_bwd,
                               void* stream);
/* The same for n (weight block, dimension) sets in ONE launch: entry i packs the forward image of [w0[i] | w1[i]] (K[i] x
 * 2 D[i], row stride D[i]) into image_fwd[i] and, unless image_bwd[i] is NULL, the input-gradient image into image_bwd[i].
 * The arrays live in host memory (all dense GraphConv blocks of a forward pass: 11 launches become one). */
int mrb_gemm_tc_pack_graphconv_batch(int n, const void* const* w0, const void* const* w1, const int* K, const int* D,
                                     void* const* image_fwd, void* const* image_bwd, void* stream);
int mrb_gemm_tc(const float* A, int lda, int M, int K, const void* image, int N, float* C, int ldc, void* stream);
/* Weight gradients on the same tensor-core path: C[Kin x N] += X^T (V x Kin) * G (V x N), reduced over the V vertices
 * (split over CTAs, fp32 vector reductions into C -- the caller zero-fills C).  Columns [0, n_split) go to C0 and
 * [n_split, N) to C1 (both Kin x * with leading dimension ldc), so that dW0 and dW1 of a GraphConv come out of one
 * pass over x and [gz | A^T gz].  N, n_split multiples of 32; C rows 16-byte aligned. */
int mrb_gemm_tc_wgrad(const float* X, int ldx, const float* G, int ldg, int V, int Kin, int N, float* C0, float* C1,
                      int n_split, int ldc, void* stream);

/* mrb_gemm_tc with an optional C += A * B (accumulate != 0): a product with a column concatenation [x_a | x_b] is
 * evaluated as two calls on the parts, the second one accumulating. */
int mrb_gemm_tc_acc(const float* A, int lda, int M, int K, const void* image, int N, float* C, int ldc, int accumulate,
                    void* stream);
/* mrb_gemm_tc_wgrad with the <= 4 "tail" feature columns (the 3 vertex-position columns of a stage input) taken from a
 * separate matrix Xtail (V x n_tail, pitch ld_tail) and written to separate rows:  T0[m, 0:n_split) / T1[m, 0:N-n_split)
 * += sum_v Xtail[v, m] * G[v, :]  -- so that dW of [pos | x] or [x | pos | ...] needs no concatenated input. */
int mrb_gemm_tc_wgrad_split(const float* X, int ldx, const float* G, int ldg, int V, int Kin, int N, float* C0, float* C1,
                            int n_split, int ldc, const float* Xtail, int ld_tail, int n_tail, float* T0, float* T1,
                            void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Split-input GraphConv (csrc/graphconv2.cu) -- GraphConv.forward (reference meshRCNN/layers.py:47-68) applied to the
 * column concatenations the stages build (layers.py:160-165,241-252,321-334) WITHOUT forming them:
 *   z_i = y0_i + p_i Wp0 + T0[tex_i] + sum_{j in N(i)} (y1_j + T1[tex_j]) + (sum_{j in N(i)} p_j) Wp1 ;  out = relu(z) (+ residual)
 *   y [n x 2D] = x_main [W0_x | W1_x] (mrb_gemm_tc on the dense columns), p = vertex positions with the 3 x D row blocks
 *   wp0 / wp1 of W0 / W1, T [R x 2D] = texel rows [W0_a | W1_a] (VertexAlign fused as a row gather: tex_i = texel row of
 *   vertex i or -1, from mrb_vert_align_texrows).  Any of the three terms may be absent (NULL).
 *   mask (optional): ReLU mask as bits, n x ceil(D/32) words -- all the backward needs of this layer's output.
 * mrb_gc_gather_bwd: gy[i] = [gz_i | sum_{j in N^T(i)} gz_j], gz = gout * mask;  optional gpos[i] = gy_i [Wp0 | Wp1]^T
 *   (n x 3, overwritten) and gT[tex_i] += gy_i (gT: tex_rows x 2D, zero-filled by the call).
 * mrb_head_fwd / _bwd: new_pos = pos + tanh(x Wx^T + pos Wp^T) with Wx = W[:, x_col:x_col+Kx], Wp = W[:, p_col:p_col+3]
 *   of nn.Linear's 3 x Kin weight (p_col < 0: no position columns) -- layers.py:255-259,335-339; delta = the tanh output
 *   (saved for the backward); bwd: gpre = g (1 - delta^2) (n x 3, for dW), gx = gpre Wx, gpos = g + gpre Wp.
 */
int mrb_vert_align_texrows(const float* pos, const int32_t* vert_mesh, const int32_t* mesh_info, int SV, int map_size,
                           int32_t* texrow, void* stream);
int mrb_gc_gather_fwd(const int32_t* rowptr, const int32_t* col, int n, int D, const float* y, int ld_y, const float* pos,
                      const float* wp0, const float* wp1, const int32_t* texrow, const float* T, int relu, uint32_t* mask,
                      const float* residual, int ld_res, float* out, int ld_out, void* stream);
int mrb_gc_gather_bwd(const int32_t* rowptr_t, const int32_t* col_t, int n, int D, const float* gout, int ld_g,
                      const uint32_t* mask, float* gy, const float* wp0, const float* wp1, float* gpos, const int32_t* texrow,
                      float* gT, long long tex_rows, void* stream);
int mrb_head_fwd(const float* x, int ld_x, int Kx, const float* pos, const float* W, int ld_w, int x_col, int p_col, int n,
                 float* new_pos, float* delta, void* stream);
int mrb_head_bwd(const float* g, const float* delta, const float* W, int ld_w, int x_col, int p_col, int n, int Kx,
                 float* gpre, float* gx, int ld_gx, float* gpos, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * VertexAlign -- replaces VertexAlign.forward / single_projection / project, reference meshRCNN/layers.py:521-613,
 * with the reference's exact (non-bilinear) semantics: out[v,c] = fmap[img,c,x1,y1] * [x2>x1 && y2>y1], as a gather of
 * channels-last texel rows.
 *   pos        SV x 3;  vert_mesh[v] = mesh of vertex v;  mesh_info[mesh] = {image index, image H, image W}.  Every image
 *              index must be < n_img: the caller validates it, the kernels do not clamp it.
 *   mrb_feature_map_to_rows   NCHW map (dtype 0 = fp32, 1 = bf16) -> channels-last fp32 rows (n_img*HW x C)
 *   mrb_rows_to_feature_map   channels-last fp32 rows (pitch ld_rows) -> NCHW fp32 (gradient of a map)
 *   mrb_vert_align_proj_fwd   T: packed texel rows, map m occupying rows [n_img * sum_{m'<m} HW_m', ...) in (image, x1, y1)
 *                             order, D columns; map_size_host: n_maps (<= 8) map sizes Hm == Wm, a HOST array (read during
 *                             the call);  out[v, 0:D] = sum_m mask * T[row_m(v)], out rows of pitch ld_out (pass a
 *                             column-offset pointer to fill a column block)
 *   mrb_vert_align_proj_bwd   gT (same shape as T, overwritten): gT[row_m(v)] += mask * gout[v]  (fp32 reductions)
 * The VertexAlign module calls the gather with one map, T = the map's rows and D = C.  Fused with the bias-free linear layer
 * that follows it in the ShapeNet stages (reference meshRCNN/layers.py:115,151-155 and :192,230), T_m = rows(f_m) @ W_m^T
 * are the per-texel projections (computed once per step with mrb_gemm_tc):  linear(align(f))[v] = sum_m mask_{v,m} *
 * T_m[img(v)*HW_m + texel_m(v)].  float4 path when D % 4 == 0 and T / gT / out rows are 16-byte aligned, scalar otherwise;
 * the forward of one such map (D <= 4096) moves whole rows with TMA bulk copies.
 * Vertex positions receive no gradient (as in the reference, where the integer cast at layers.py:592 cuts the graph). */
int mrb_feature_map_to_rows(const void* fmap, int dtype, int n_img, int C, int HW, float* rows, void* stream);
int mrb_rows_to_feature_map(const float* rows, int ld_rows, int n_img, int C, int HW, float* gfmap, void* stream);
int mrb_vert_align_proj_fwd(const float* T, int D, int n_maps, const int* map_size_host, int n_img, const float* pos,
                            const int32_t* vert_mesh, const int32_t* mesh_info, int SV, float* out, int ld_out, void* stream);
int mrb_vert_align_proj_bwd(const float* gout, int ld_g, int D, int n_maps, const int* map_size_host, int n_img,
                            const float* pos, const int32_t* vert_mesh, const int32_t* mesh_info, int SV, float* gT,
                            void* stream);

/* Bilinear VertexAlign (opt-in mode; csrc/vert_align_bilinear.cu), differentiable in the vertex positions.  One square S x S
 * map given as channels-last fp32 rows: texel (i, j) of image img is rows[((img * S + i) * S + j) * ld_rows + 0 .. D-1] (the
 * output of mrb_feature_map_to_rows, or per-texel projections T of it).  Projection as mrb_vert_align_proj_fwd up to and including
 * the clamps to the image (x = w / sx indexes the H axis, y = h / sy the W axis), then x, y clamped to [0, S-1] and
 *   out[v] = (1-fx)(1-fy) f[x0,y0] + (1-fx) fy f[x0,y0+1] + fx (1-fy) f[x0+1,y0] + fx fy f[x0+1,y0+1]
 * with x0 = clamp(floor(x), 0, S-2), fx = x - x0 (y0, fy alike); S == 1 gives f[0,0].  This is grid_sample(align_corners=True,
 * padding_mode="border") at (x, y).
 *   mrb_vert_align_bilinear_fwd  out[v, 0:D] = sample (accumulate == 0) or += sample (accumulate != 0); out rows of pitch
 *                                ld_out (pass a column-offset pointer to fill a column block)
 *   mrb_vert_align_bilinear_bwd  grows (may be NULL; zero-filled by the caller, pitch ld_grows) += w_corner * gout[v] for the
 *                                four corners (fp32 reductions); gpos (may be NULL, SV x 3) = (accumulate_gpos == 0) or +=
 *                                (!= 0) the position gradient, written by the one warp that owns the vertex (no atomics:
 *                                deterministic, and calls for several maps issued in sequence on one stream may accumulate).
 *                                Clamps pass the gradient inside their closed interval; at a texel knot the derivative is the
 *                                one-sided one of the cell the floor rule picks; where the projection or its derivative is not
 *                                finite (p2 == 0, NaN positions) the sample is the clamped one and the gradient is exactly 0.
 * Every mesh_info image index must be < n_img (the caller validates; the kernels clamp it as well).  SV == 0 returns 0
 * without a launch; D, S, n_img >= 1 and pitches >= D are required.  float4 path when D % 4 == 0 and all rows 16-byte aligned. */
int mrb_vert_align_bilinear_fwd(const float* rows, int ld_rows, int D, int S, int n_img, const float* pos,
                                const int32_t* vert_mesh, const int32_t* mesh_info, int SV, int accumulate, float* out,
                                int ld_out, void* stream);
int mrb_vert_align_bilinear_bwd(const float* gout, int ld_g, const float* rows, int ld_rows, int D, int S, int n_img,
                                const float* pos, const int32_t* vert_mesh, const int32_t* mesh_info, int SV, float* grows,
                                int ld_grows, float* gpos, int accumulate_gpos, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Surface sampling -- replaces utils/mesh_sampling.py:6-57 (sample, surface_areas), utils/process.py:7-20
 * (normalize_mesh) and the per-mesh loop of batched_mesh_sampling (meshRCNN/loss_functions.py:80-89).
 * Packed batch: verts SV x 3, faces SF x 3 int64 per-mesh local ids, v_off / f_off int32 offsets (B+1 entries).
 *   mrb_face_areas        areas[f] = |AB x AC| / 2
 *   mrb_face_area_cdf     + inclusive per-mesh CDF in fp64
 *   mrb_sample_points_fwd n points per mesh: face by inverse CDF of u (or injected face_idx, local ids), barycentric
 *                         weights (1-sqrt(xi1), (1-xi2)sqrt(xi1), xi2 sqrt(xi1)); u/xi2/xi1 NULL => Philox(seed).
 *                         Outputs: raw points, global face id, weights (saved for backward), normalised cloud and
 *                         per-cloud stats (8 doubles: mean[3], factor, argmax row or -1).
 *   mrb_sample_points_bwd gcloud -> gverts (accumulated with atomics; caller zero-fills); scratch: 4 * B doubles
 */
int mrb_face_areas(const float* verts, const long long* faces, const int32_t* v_off, const int32_t* f_off, int B,
                   int max_faces, float* areas, void* stream);
int mrb_face_area_cdf(const float* verts, const long long* faces, const int32_t* v_off, const int32_t* f_off, int B,
                      int max_faces, float* areas, double* cdf, void* stream);
int mrb_sample_points_fwd(const float* verts, const long long* faces, const int32_t* v_off, const int32_t* f_off,
                          const double* cdf, int B, int n, const float* u, const long long* face_idx, const float* xi2,
                          const float* xi1, unsigned long long seed, float* raw, int32_t* fidx_out, float* w_out,
                          float* cloud, double* stats, void* stream);
int mrb_normalize_cloud_fwd(const float* raw, int B, int n, float* cloud, double* stats, void* stream);
int mrb_sample_points_bwd(const float* gcloud, const float* cloud, const double* stats, const int32_t* fidx,
                          const float* w, const long long* faces, const int32_t* v_off, int B, int n, float* gverts,
                          double* scratch /* 4 * B doubles */, void* stream);
/* the same with gverts rows of ld_gverts floats: 3, or 4 (xyz + one unused lane, 16-byte aligned: one vector reduction per
 * face corner instead of three scalar atomics) */
int mrb_sample_points_bwd_ld(const float* gcloud, const float* cloud, const double* stats, const int32_t* fidx,
                             const float* w, const long long* faces, const int32_t* v_off, int B, int n, float* gverts,
                             int ld_gverts, double* scratch /* 4 * B doubles */, void* stream);
/* Eval-side sampling (no backward): the points of mrb_sample_points_fwd for the same randomness (same face choice, weights
 * and Philox counter), multiplied by scale[b] (scale may be NULL: unscaled, bitwise the `raw` output) and NOT normalised;
 * normals = unit normal (B-A)x(C-A)/|.| of each point's face (zero vector for a degenerate face); fidx_out = global face id.
 * points, normals: B x n x 3. */
int mrb_sample_surface_fwd(const float* verts, const long long* faces, const int32_t* v_off, const int32_t* f_off,
                           const double* cdf, int B, int n, const float* u, const long long* face_idx, const float* xi2,
                           const float* xi1, unsigned long long seed, const float* scale, float* points, float* normals,
                           int32_t* fidx_out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Mesh evaluation metrics (the Mesh R-CNN paper's protocol; reported by eval_utils.compare_meshes).
 *   mrb_mesh_gt_scale  scale[b] = target / longest side of the bounding box of vertices [v_off[b], v_off[b+1]) (exact fp32
 *                      min / max; zero extent gives inf)
 *   mrb_mesh_metrics   from the k = 0 outputs of mrb_knn_fwd (d_p, i_p: B x P; d_q, i_q: B x Q) and the unit normals
 *                      n_p (B x P x 3), n_q (B x Q x 3): out[b][3 + 3T] = Chamfer-L2 (mean d_p + mean d_q), NC, AbsNC
 *                      (0.5 * (mean n.m + mean m.n) over the nearest neighbours, without / with |.|), then for each of the
 *                      T <= 8 thresholds tau_host[t] (a HOST array, read during the call): Precision, Recall (100 x share of
 *                      points with fp32 sqrt(d) < tau) and F1 = 2PR / (P + R + 1e-8).  fp64 sums in a fixed order.
 */
int mrb_mesh_gt_scale(const float* verts, const int32_t* v_off, int B, float target, float* scale, void* stream);
int mrb_mesh_metrics(const float* d_p, const int32_t* i_p, const float* d_q, const int32_t* i_q, const float* n_p,
                     const float* n_q, int B, int P, int Q, const float* tau_host, int T, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Chamfer / k-NN -- replaces batched_point2point_distance (cross branch), batched_chamfer_distance and the topk of
 * compute_normals, reference meshRCNN/loss_functions.py:93-102,141,207-220.  No B x P x Q matrix is formed.
 *   mrb_knn_fwd     both directions in one call: for each point of a (B x P x 3) the squared distance + index of the
 *                   nearest point of b (B x Q x 3) and, if k > 0 (k <= 16), the k nearest indices sorted by
 *                   (distance, index) -- outputs *_a -- and the same for each point of b against a -- outputs *_b
 *                   (either output set may be NULL).  Exact (direct (p-q)^2 distances).  Clouds of <= 65535 points are
 *                   counting-sorted into a uniform cell grid and every query scans a growing cell box until its k-th
 *                   best distance is proven final; larger clouds use the shared-memory tiled scan (x-sorted, far tiles
 *                   pruned).  Both return identical results.  workspace: mrb_knn_workspace_bytes(B,P,Q).
 *   mrb_knn_fwd_algo  same, with the search strategy forced: 0 automatic, 1 tiled scan, 2 cell grid.
 *   mrb_sum_scaled  out[0] = scale * sum(x[0..n))   (fp64 accumulation; acc = 1 double of scratch)
 *   mrb_chamfer_bwd gradient of  *g_a * scale * sum_i |a_i - b_idx_a[i]|^2 + *g_b * scale * sum_j |a_idx_b[j] - b_j|^2
 *                   accumulated into ga / gb (either may be NULL).
 */
long long mrb_knn_workspace_bytes(int B, int P, int Q);
int mrb_knn_fwd(const float* a, const float* b, int B, int P, int Q, int k, float* min_d_a, int32_t* min_i_a,
                int32_t* knn_a, float* min_d_b, int32_t* min_i_b, int32_t* knn_b, void* workspace, void* stream);
int mrb_knn_fwd_algo(const float* a, const float* b, int B, int P, int Q, int k, float* min_d_a, int32_t* min_i_a,
                     int32_t* knn_a, float* min_d_b, int32_t* min_i_b, int32_t* knn_b, void* workspace, int algo,
                     void* stream);
int mrb_sum_scaled(const float* x, long long n, double scale, double* acc, float* out, void* stream);
int mrb_chamfer_bwd(const float* a, const float* b, int B, int P, int Q, const int32_t* idx_a, const int32_t* idx_b,
                    const float* g_a, const float* g_b, float scale, float* ga, float* gb, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Normals + normal / edge losses -- replaces compute_normals, batched_normal_distance and total_edge_length,
 * reference meshRCNN/loss_functions.py:107-170,175-189 (incl. the S.cpu() -> symeig -> .to(device) round trip).
 *   mrb_normals_fwd     normal[b,p] = row 0 of the (ascending, canonically signed) eigenvector matrix of the 3x3
 *                       scatter matrix of pt[b, knn[b,p,:]]
 *   mrb_normals_bwd     gn -> gpt (atomic accumulate into B x P x 3); rows with gn = 0 are skipped.  Degenerate spectra: the
 *                       derivative of an eigenvector divides by the gap to each other eigenvalue, and a pair of eigenvalues
 *                       closer than 1e-14 * (|w0| + |w1| + |w2|) contributes nothing instead.  So a row whose three eigenvalues
 *                       coincide (k = 1, all k neighbours the same point, an isotropic neighbourhood) has an exactly zero
 *                       gradient, and a row with one coinciding pair (k = 2, a square axis-aligned planar patch) keeps only the
 *                       terms of the other pairs; both stay finite.  The forward normal of such a row is unit length, but
 *                       within the degenerate eigenspace its direction is the eigensolver's choice, not a defined quantity.
 *   mrb_normals_fwd_eig also writes the eigen-decomposition: eig = 12 planes of B * P doubles (w0 w1 w2 | V row-major)
 *   mrb_normals_bwd_ld  the same into rows of ld_gpt floats: 3, or 4 (xyz + one unused lane, 16-byte aligned) -- the padded
 *                       layout turns the 3 scalar atomics per neighbour into one 16-byte vector reduction; eig (may be
 *                       NULL) = the planes mrb_normals_fwd_eig wrote for the same pt / knn: the Jacobi sweeps are skipped
 *   mrb_normal_loss_fwd out2[0] = sum_i |na_i . nb_idx_a[i]|, out2[1] = sum_j |nb_j . na_idx_b[j]|
 *   mrb_edge_loss_fwd   out[0] = mean over the E directed edges of |v_r - v_c|^2
 */
int mrb_normals_fwd(const float* pt, const int32_t* knn, int B, int P, int k, float* normals_out, void* stream);
int mrb_normals_bwd(const float* pt, const int32_t* knn, int B, int P, int k, const float* gn, float* gpt, void* stream);
int mrb_normals_fwd_eig(const float* pt, const int32_t* knn, int B, int P, int k, float* normals_out, double* eig,
                        void* stream);
int mrb_normals_bwd_ld(const float* pt, const int32_t* knn, int B, int P, int k, const float* gn, float* gpt, int ld_gpt,
                       const double* eig, void* stream);
int mrb_normal_loss_fwd(const float* na, const float* nb, int B, int P, int Q, const int32_t* idx_a, const int32_t* idx_b,
                        double* acc2, float* out2, void* stream);
int mrb_normal_loss_bwd(const float* na, const float* nb, int B, int P, int Q, const int32_t* idx_a, const int32_t* idx_b,
                        const float* g0, const float* g1, float* gna, float* gnb, void* stream);
/* Scaled totals (what mesh_loss returns, loss_functions.py:66,72): out1[0] = scale * (sum_i |na.nb| + sum_j |nb.na|) and its
 * backward with the single upstream gradient *g -- the add / negate / divide chain of the reference folded into the kernels. */
int mrb_normal_loss_total_fwd(const float* na, const float* nb, int B, int P, int Q, const int32_t* idx_a, const int32_t* idx_b,
                              double scale, double* acc2, float* out1, void* stream);
int mrb_normal_loss_total_bwd(const float* na, const float* nb, int B, int P, int Q, const int32_t* idx_a, const int32_t* idx_b,
                              const float* g, float scale, float* gna, float* gnb, void* stream);
/* Scalar glue of the loss (sums over the refinement stages, the weighted total of utils/train_utils.py:208-225):
 * out[0] = sum_i w[i] * *xs[i]   and   out[i] = *g * w[i]   (n <= 16; xs_host: HOST array of n device pointers,
 * w_host: HOST array of n weights -- both are read during the call). */
int mrb_scalar_combine(const void* xs_host, const float* w_host, int n, float* out, void* stream);
int mrb_scalar_scatter(const float* g, const float* w_host, int n, float* out, void* stream);
int mrb_edge_loss_fwd(const float* pos, const long long* adj, long long E, double* acc, float* out, void* stream);
int mrb_edge_loss_bwd(const float* pos, const long long* adj, long long E, const float* g, float* gpos, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MESHRCNN_B200_H */
