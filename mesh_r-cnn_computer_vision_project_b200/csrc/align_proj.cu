// VertexAlign as a gather of channels-last texel rows: the per-texel projections of the ShapeNet bottleneck, and the feature
// rows of the plain VertexAlign module.
//
// In the ShapeNet refinement stages VertexAlign (reference meshRCNN/layers.py:509-613) feeds a bias-free bottleneck
// `linear(3840 -> 128)` (layers.py:115,151-155 residual head; :192,230 plain head).  VertexAlign is a masked row gather
// (out[v, c] = fmap[img, c, x1, y1] * [x2 > x1 and y2 > y1], see valign.cuh), and a gather commutes with a linear map:
//
//     linear(align(f))[v, :] = sum_m  mask_{v,m} * ( f_m[img(v), :, texel_m(v)] . W_m^T )
//                            = sum_m  mask_{v,m} * T_m[img(v) * HW_m + texel_m(v), :]        T_m = rows(f_m) @ W_m^T
//
// with W_m the column slice of the weight that belongs to map m.  So the n_img * sum_m HW_m texels (1 655 per image for
// the four ResNet50 maps of a 137 x 137 input) are projected ONCE per step on the tensor cores (gemm_tc.cu), and every
// vertex gathers and sums <= 4 rows of D = 128 floats.  The SV x 3840 matrix (3.4 GB at BASELINE configs[2]) is never
// formed and the three big GEMMs over it (forward, input gradient, weight gradient) shrink 4x - 40x.
//
// Kernels here:
//   k_map_to_rows / k_rows_to_map   NCHW (fp32 | bf16) <-> channels-last fp32 rows (the A operand of the texel GEMM)
//   k_proj_gather_fwd               out[v, :] = sum_m mask * T[row_m(v), :]                (one warp per vertex)
//   k_fwd_bulk                      the same for one map and D % 4 == 0, by TMA bulk copies of whole rows
//   k_proj_gather_bwd               gT[row_m(v), :] += mask * gout[v, :]                   (red.global.add.v4.f32)
// The plain VertexAlign module is the same gather with one map, T = the map's own rows and D = C, written into the map's
// column block of the SV x sum(C_m) output (functional._VertAlign); odd C and column offsets take the scalar kernels.
#include <cuda_bf16.h>

#include "common.cuh"
#include "valign.cuh"
#include "../../include/meshrcnn_b200.h"

namespace mrb {
namespace valign {

constexpr int MAX_MAPS = 8;

struct MapSet {
    int n_maps;
    int size[MAX_MAPS];             // Hm == Wm of map m
    long long row_base[MAX_MAPS];   // first row of map m in the packed texel matrix: n_img * sum_{m' < m} HW_m'
};

__device__ __forceinline__ float load_as_float(const float* p) { return __ldg(p); }
__device__ __forceinline__ float load_as_float(const __nv_bfloat16* p) { return __bfloat162float(*p); }

// NCHW -> channels-last fp32 rows: per image a C x HW matrix is transposed to HW x C through a 32 x 33 shared tile.
template <typename T>
__global__ void __launch_bounds__(256) k_map_to_rows(const T* __restrict__ src, float* __restrict__ dst, int C, int HW) {
    __shared__ float t[32][33];
    const int img = blockIdx.z;
    const T* s = src + (size_t)img * C * HW;
    float* d = dst + (size_t)img * C * HW;
    const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, pix = p0 + tx;
        t[r][tx] = (c < C && pix < HW) ? load_as_float(s + (size_t)c * HW + pix) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int pix = p0 + r, c = c0 + tx;
        if (pix < HW && c < C) d[(size_t)pix * C + c] = t[tx][r];
    }
}

// channels-last fp32 rows -> NCHW fp32 (gradient of the maps)
__global__ void __launch_bounds__(256) k_rows_to_map(const float* __restrict__ src, int ld_src, float* __restrict__ dst, int C,
                                                     int HW) {
    __shared__ float t[32][33];
    const int img = blockIdx.z;
    const float* s = src + (size_t)img * HW * ld_src;
    float* d = dst + (size_t)img * C * HW;
    const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int pix = p0 + r, c = c0 + tx;
        t[r][tx] = (c < C && pix < HW) ? s[(size_t)pix * ld_src + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int c = c0 + r, pix = p0 + tx;
        if (pix < HW && c < C) d[(size_t)c * HW + pix] = t[tx][r];
    }
}

// texel row of vertex v in map m of the packed texel matrix, or -1 when the vertex is masked in that map
__device__ __forceinline__ long long texel_row(const MapSet& ms, int m, const float* __restrict__ pos,
                                               const int32_t* __restrict__ vert_mesh, const int32_t* __restrict__ mesh_info,
                                               int v) {
    const int sz = ms.size[m];
    const Texel t = project(pos, vert_mesh, mesh_info, v, sz, sz);
    return t.valid ? ms.row_base[m] + (long long)t.img * sz * sz + t.xy : -1;
}

// out[v, :D] = sum_m mask_{v,m} T[row_m(v), :D].  One warp per vertex: lane m < n_maps projects into map m, the rows are
// broadcast, and the <= 8 row loads of a vertex are independent (issued before the adds).  VEC: every lane owns 4 of each
// 128 columns (D % 4 == 0, T rows and out rows 16-byte aligned); otherwise one column of each 32.
template <bool VEC>
__global__ void __launch_bounds__(256) k_proj_gather_fwd(const float* __restrict__ T, int D, const __grid_constant__ MapSet ms,
                                                         const float* __restrict__ pos, const int32_t* __restrict__ vert_mesh,
                                                         const int32_t* __restrict__ mesh_info, int SV,
                                                         float* __restrict__ out, int ld_out) {
    const int v = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (v >= SV) return;
    long long mine = -1;
    if (lane_id() < ms.n_maps) mine = texel_row(ms, lane_id(), pos, vert_mesh, mesh_info, v);
    long long rows[MAX_MAPS];
#pragma unroll
    for (int m = 0; m < MAX_MAPS; ++m) rows[m] = __shfl_sync(0xffffffffu, mine, m);
    if (VEC) {
        for (int d = lane_id() * 4; d < D; d += 128) {
            float4 x[MAX_MAPS];
#pragma unroll
            for (int m = 0; m < MAX_MAPS; ++m) {
                x[m] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (m < ms.n_maps && rows[m] >= 0) x[m] = __ldg(reinterpret_cast<const float4*>(T + (size_t)rows[m] * D + d));
            }
            float4 acc = x[0];
#pragma unroll
            for (int m = 1; m < MAX_MAPS; ++m) { acc.x += x[m].x; acc.y += x[m].y; acc.z += x[m].z; acc.w += x[m].w; }
            *reinterpret_cast<float4*>(out + (size_t)v * ld_out + d) = acc;
        }
    } else {
        for (int d = lane_id(); d < D; d += 32) {
            float x[MAX_MAPS];
#pragma unroll
            for (int m = 0; m < MAX_MAPS; ++m) x[m] = (m < ms.n_maps && rows[m] >= 0) ? __ldg(T + (size_t)rows[m] * D + d) : 0.f;
            float acc = x[0];
#pragma unroll
            for (int m = 1; m < MAX_MAPS; ++m) acc += x[m];
            out[(size_t)v * ld_out + d] = acc;
        }
    }
}

// gT[row_m(v), :] += gout[v, :] for every unmasked (vertex, map); fp32 reductions, vector ones when VEC (D % 4 == 0, gT
// 16-byte aligned) -- the texel rows are shared by the vertices that project to the same texel.  Fully masked vertices
// return before touching gout.
template <bool VEC>
__global__ void __launch_bounds__(256) k_proj_gather_bwd(const float* __restrict__ gout, int ld_g, int D, const __grid_constant__ MapSet ms,
                                                         const float* __restrict__ pos, const int32_t* __restrict__ vert_mesh,
                                                         const int32_t* __restrict__ mesh_info, int SV, float* __restrict__ gT) {
    const int v = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (v >= SV) return;
    long long mine = -1;
    if (lane_id() < ms.n_maps) mine = texel_row(ms, lane_id(), pos, vert_mesh, mesh_info, v);
    if (__ballot_sync(0xffffffffu, mine >= 0) == 0) return;
    long long rows[MAX_MAPS];
#pragma unroll
    for (int m = 0; m < MAX_MAPS; ++m) rows[m] = __shfl_sync(0xffffffffu, mine, m);
    if (VEC) {
        const bool vec = ((ld_g & 3) == 0) && ((reinterpret_cast<uintptr_t>(gout) & 15) == 0);
        for (int d = lane_id() * 4; d < D; d += 128) {
            float4 g;
            const float* gp = gout + (size_t)v * ld_g + d;
            if (vec) g = __ldg(reinterpret_cast<const float4*>(gp));
            else g = make_float4(__ldg(gp), __ldg(gp + 1), __ldg(gp + 2), __ldg(gp + 3));
#pragma unroll
            for (int m = 0; m < MAX_MAPS; ++m)
                if (m < ms.n_maps && rows[m] >= 0)
                    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(gT + (size_t)rows[m] * D + d), "f"(g.x),
                                 "f"(g.y), "f"(g.z), "f"(g.w)
                                 : "memory");
        }
    } else {
        for (int d = lane_id(); d < D; d += 32) {
            const float g = __ldg(gout + (size_t)v * ld_g + d);
#pragma unroll
            for (int m = 0; m < MAX_MAPS; ++m)
                if (m < ms.n_maps && rows[m] >= 0) atomicAdd(gT + (size_t)rows[m] * D + d, g);
        }
    }
}

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// The one-map gather with D % 4 == 0 done by the TMA engine (measured faster than k_proj_gather_fwd<true> for the module's
// 256..2048-channel maps): grid-stride over vertex batches; warp = `slots` vertices per batch, lane = vertex.  Every lane
// issues a bulk copy (cp.async.bulk) of its texel row global -> shared, waits on the warp's mbarrier, and issues the bulk
// store shared -> global of the output row (masked vertices store a row of zeros).  No feature value passes through a
// register, loads and stores are full 128-byte lines, and 16-32 rows per warp are in flight.
constexpr int VA_WARPS = 4;
constexpr int VA_WARP_BYTES = 16384;

__global__ void __launch_bounds__(VA_WARPS * 32) k_fwd_bulk(const float* __restrict__ fmap_cl, int C, int Hm, int Wm,
                                                           const float* __restrict__ pos, const int32_t* __restrict__ vert_mesh,
                                                           const int32_t* __restrict__ mesh_info, int SV,
                                                           float* __restrict__ out, int ld_out, int slots) {
    extern __shared__ __align__(128) unsigned char va_smem[];
    __shared__ __align__(8) unsigned long long bars[VA_WARPS];
    const int row_bytes = C * 4;
    unsigned char* zero_row = va_smem;                                         // row_bytes of zeros (shared by the CTA)
    unsigned char* my_slots = va_smem + ((row_bytes + 127) & ~127) + warp_id() * VA_WARP_BYTES;
    for (int i = threadIdx.x; i < C; i += blockDim.x) reinterpret_cast<float*>(zero_row)[i] = 0.f;
    const uint32_t bar = smem_addr(&bars[warp_id()]);
    if (lane_id() == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");                // zero row + barrier visible to the async proxy
    __syncthreads();

    const size_t plane = (size_t)Hm * Wm;
    uint32_t phase = 0;
    const int batches = (SV + slots - 1) / slots;
    for (int b = blockIdx.x * VA_WARPS + warp_id(); b < batches; b += gridDim.x * VA_WARPS) {
        const int v = b * slots + lane_id();
        const bool mine = lane_id() < slots && v < SV;
        Texel t;
        t.valid = 0;
        if (mine) t = project(pos, vert_mesh, mesh_info, v, Hm, Wm);
        const unsigned valid_mask = __ballot_sync(0xffffffffu, mine && t.valid);
        const uint32_t slot = smem_addr(my_slots + lane_id() * row_bytes);
        if (valid_mask) {
            if (lane_id() == 0)
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar),
                             "r"((uint32_t)(__popc(valid_mask) * row_bytes))
                             : "memory");
            __syncwarp();
            if (mine && t.valid) {
                const float* src = fmap_cl + ((size_t)t.img * plane + t.xy) * C;
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(slot),
                             "l"(src), "r"((uint32_t)row_bytes), "r"(bar)
                             : "memory");
            }
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "VA_WAIT:\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                "@p bra.uni VA_DONE;\n\t"
                "bra.uni VA_WAIT;\n\t"
                "VA_DONE:\n\t}" ::"r"(bar), "r"(phase) : "memory");
            phase ^= 1;
        }
        if (mine) {
            float* dst = out + (size_t)v * ld_out;
            const uint32_t srcs = t.valid ? slot : smem_addr(zero_row);
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(srcs),
                         "r"((uint32_t)row_bytes)
                         : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");        // slots may be overwritten by the next batch
        __syncwarp();
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

static int make_mapset(MapSet& ms, int n_maps, const int* map_size_host, int n_img, const char* what) {
    MRB_REQUIRE(n_maps >= 1 && n_maps <= MAX_MAPS && map_size_host, "%s: 1..%d feature maps", what, MAX_MAPS);
    ms.n_maps = n_maps;
    long long base = 0;
    for (int m = 0; m < MAX_MAPS; ++m) {
        ms.size[m] = m < n_maps ? map_size_host[m] : 1;
        ms.row_base[m] = base;
        if (m < n_maps) {
            MRB_REQUIRE(map_size_host[m] > 0, "%s: bad map size", what);
            base += (long long)n_img * map_size_host[m] * map_size_host[m];
        }
    }
    return MRB_OK;
}

}  // namespace valign
}  // namespace mrb

using namespace mrb;
using namespace mrb::valign;

extern "C" int mrb_feature_map_to_rows(const void* fmap, int dtype, int n_img, int C, int HW, float* rows, void* stream_) {
    MRB_REQUIRE(fmap && rows && n_img >= 0 && C > 0 && HW > 0, "feature_map_to_rows: bad arguments");
    MRB_REQUIRE(dtype == 0 || dtype == 1, "feature_map_to_rows: dtype must be 0 (fp32) or 1 (bf16)");
    MRB_REQUIRE(n_img <= 65535, "feature_map_to_rows: too many images");
    if (n_img == 0) return MRB_OK;
    const dim3 grid(ceil_div(HW, 32), ceil_div(C, 32), n_img);
    cudaStream_t s = (cudaStream_t)stream_;
    if (dtype == 0) k_map_to_rows<float><<<grid, 256, 0, s>>>((const float*)fmap, rows, C, HW);
    else k_map_to_rows<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)fmap, rows, C, HW);
    return check_launch("feature_map_to_rows");
}

extern "C" int mrb_rows_to_feature_map(const float* rows, int ld_rows, int n_img, int C, int HW, float* gfmap, void* stream_) {
    MRB_REQUIRE(rows && gfmap && n_img >= 0 && C > 0 && HW > 0 && ld_rows >= C, "rows_to_feature_map: bad arguments");
    MRB_REQUIRE(n_img <= 65535, "rows_to_feature_map: too many images");
    if (n_img == 0) return MRB_OK;
    k_rows_to_map<<<dim3(ceil_div(HW, 32), ceil_div(C, 32), n_img), 256, 0, (cudaStream_t)stream_>>>(rows, ld_rows, gfmap, C, HW);
    return check_launch("rows_to_feature_map");
}

extern "C" int mrb_vert_align_proj_fwd(const float* T, int D, int n_maps, const int* map_size_host, int n_img,
                                       const float* pos, const int32_t* vert_mesh, const int32_t* mesh_info, int SV,
                                       float* out, int ld_out, void* stream_) {
    MRB_REQUIRE(T && pos && vert_mesh && mesh_info && out, "vert_align_proj_fwd: null pointer");
    MRB_REQUIRE(D > 0 && ld_out >= D, "vert_align_proj_fwd: D > 0 and ld_out >= D required");
    MapSet ms;
    if (int rc = make_mapset(ms, n_maps, map_size_host, n_img, "vert_align_proj_fwd")) return rc;
    if (SV == 0) return MRB_OK;
    const bool vec = D % 4 == 0 && ld_out % 4 == 0 && ((uintptr_t)T & 15) == 0 && ((uintptr_t)out & 15) == 0;
    const dim3 grid(ceil_div(SV, 8));
    cudaStream_t s = (cudaStream_t)stream_;
    if (vec && n_maps == 1 && D * 4 <= VA_WARP_BYTES) {
        const int row_bytes = D * 4;
        const int slots = min(32, VA_WARP_BYTES / row_bytes);
        const size_t smem = ((row_bytes + 127) & ~127) + (size_t)VA_WARPS * VA_WARP_BYTES;
        static SmemOptIn optin;
        if (int rc = ensure_dynamic_smem(k_fwd_bulk, 16384 + VA_WARPS * VA_WARP_BYTES, optin, "vert_align_proj_fwd")) return rc;
        const int batches = ceil_div(SV, slots);
        const int bulk_grid = min(ceil_div(batches, VA_WARPS), 2 * kNumSMs);
        k_fwd_bulk<<<bulk_grid, VA_WARPS * 32, smem, s>>>(T, D, ms.size[0], ms.size[0], pos, vert_mesh, mesh_info, SV, out, ld_out,
                                                          slots);
    } else if (vec) {
        k_proj_gather_fwd<true><<<grid, 256, 0, s>>>(T, D, ms, pos, vert_mesh, mesh_info, SV, out, ld_out);
    } else {
        k_proj_gather_fwd<false><<<grid, 256, 0, s>>>(T, D, ms, pos, vert_mesh, mesh_info, SV, out, ld_out);
    }
    return check_launch("vert_align_proj_fwd");
}

extern "C" int mrb_vert_align_proj_bwd(const float* gout, int ld_g, int D, int n_maps, const int* map_size_host, int n_img,
                                       const float* pos, const int32_t* vert_mesh, const int32_t* mesh_info, int SV, float* gT,
                                       void* stream_) {
    MRB_REQUIRE(gout && pos && vert_mesh && mesh_info && gT, "vert_align_proj_bwd: null pointer");
    MRB_REQUIRE(D > 0 && ld_g >= D, "vert_align_proj_bwd: D > 0 and ld_g >= D required");
    MapSet ms;
    if (int rc = make_mapset(ms, n_maps, map_size_host, n_img, "vert_align_proj_bwd")) return rc;
    cudaStream_t s = (cudaStream_t)stream_;
    long long total_rows = 0;
    for (int m = 0; m < n_maps; ++m) total_rows += (long long)n_img * map_size_host[m] * map_size_host[m];
    cudaError_t e = cudaMemsetAsync(gT, 0, sizeof(float) * (size_t)total_rows * D, s);     // gT is overwritten, not accumulated
    if (e != cudaSuccess) {
        set_error("vert_align_proj_bwd: memset: %s", cudaGetErrorString(e));
        return MRB_ERR_CUDA;
    }
    if (SV == 0) return MRB_OK;
    if (D % 4 == 0 && ((uintptr_t)gT & 15) == 0)
        k_proj_gather_bwd<true><<<ceil_div(SV, 8), 256, 0, s>>>(gout, ld_g, D, ms, pos, vert_mesh, mesh_info, SV, gT);
    else
        k_proj_gather_bwd<false><<<ceil_div(SV, 8), 256, 0, s>>>(gout, ld_g, D, ms, pos, vert_mesh, mesh_info, SV, gT);
    return check_launch("vert_align_proj_bwd");
}
