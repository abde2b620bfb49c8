// Bilinear VertexAlign over channels-last fp32 rows, with gradients to the rows and to the vertex positions (opt-in mode;
// the reference-mode kernels in vert_align.cu / align_proj.cu / graphconv2.cu are separate and unchanged).
//
// For vertex v of mesh m, image img = mesh_info[m] and one square S x S map whose texel (i, j) of image img is the D-wide
// row rows[(img * S + i) * S + j]:
//   1. projection: h, w exactly as valign::project (explicitly rounded fp32 ops, clamps to [0, H-1] / [0, W-1]), then
//      x = w / sx, y = h / sy with the same divisors.  x indexes the H axis of the map and y the W axis (reference axis
//      assignment, layers.py:587-590).  x and y are then clamped to [0, S-1]: x = w / sx reaches S - S/W > S - 1 on the
//      last texel column, and the clamp keeps the sample an interpolation there (grid_sample's border padding).
//   2. sampling: S == 1 gives f[0, 0].  Otherwise x0 = clamp(floor(x), 0, S-2), fx = x - x0 in [0, 1] (y0, fy alike) and
//        out = (1-fx)(1-fy) f[x0,y0] + (1-fx) fy f[x0,y0+1] + fx (1-fy) f[x0+1,y0] + fx fy f[x0+1,y0+1]
//      = grid_sample(align_corners=True, padding_mode="border") at (x, y).  Exact at integer (x, y), last row and column
//      included.
//   3. gradients: rows get the weighted scatter of the upstream gradient g.  Positions get the chain rule through the
//      weights, x = w / sx, y = h / sy, the clamps and the projection.  Every clamp passes the gradient where its argument
//      is inside the closed interval (like torch.clamp).  At a texel knot the derivative is the one-sided derivative of the
//      cell the floor rule picks.  If h, w or their derivatives are not finite (p2 == 0, a NaN position), the sample is
//      the clamped one and the position gradient is exactly 0.
//
// One warp per vertex: the projection and d(x, y)/dp are computed once per warp; lanes cover the D columns in float4 when
// D % 4 == 0 and every row base is 16-byte aligned, in scalars otherwise.  The backward scatters into grows with vector
// reductions and reduces the position gradient over the warp, so the warp that owns the vertex writes it without atomics
// (deterministic; several maps of one vertex, issued in sequence on one stream, may accumulate into it).
//
// Fault safety: every float is clamped (fminf / fmaxf map NaN to the bound) before its conversion to int, the integer
// corner and image indices are clamped again, and every row offset is computed in size_t.
#include "common.cuh"
#include "../../include/meshrcnn_b200.h"

namespace mrb {
namespace vabil {

struct Sample {
    size_t r00, r01, r10, r11;    // corner rows f[x0,y0], f[x0,y0+1], f[x0+1,y0], f[x0+1,y0+1]
    float fx, fy;
    float jx0, jx2;                // d x / d p0, d x / d p2   (x does not depend on p1)
    float jy1, jy2;                // d y / d p1, d y / d p2   (y does not depend on p0)
};

__device__ __forceinline__ bool finite(float a) { return fabsf(a) <= 3.402823466e38f; }   // false for inf and NaN

__device__ __forceinline__ Sample locate(const float* __restrict__ pos, const int32_t* __restrict__ vert_mesh,
                                         const int32_t* __restrict__ mesh_info, int v, int S, int n_img) {
    const int mesh = vert_mesh[v];
    const int img = min(max(mesh_info[3 * mesh + 0], 0), n_img - 1);
    const int Hi = mesh_info[3 * mesh + 1], Wi = mesh_info[3 * mesh + 2];
    const float H = (float)Hi, W = (float)Wi;
    const float p0 = pos[3 * (size_t)v + 0], p1 = pos[3 * (size_t)v + 1], p2 = pos[3 * (size_t)v + 2];
    // projection: the fp32 ops of valign::project (reference layers.py:557-562, 577-578)
    const float hr = __fadd_rn(__fmul_rn(248.f, __fdiv_rn(p1, p2)), 111.5f);
    const float wr = __fadd_rn(__fmul_rn(248.f, __fdiv_rn(p0, -p2)), 111.5f);
    const float h = fminf(fmaxf(hr, 0.f), H - 1.f);
    const float w = fminf(fmaxf(wr, 0.f), W - 1.f);
    const float sx = (float)((double)Wi / (double)S);
    const float sy = (float)((double)Hi / (double)S);
    const float xr = __fdiv_rn(w, sx), yr = __fdiv_rn(h, sy);
    const float top = (float)(S - 1);
    const float x = fminf(fmaxf(xr, 0.f), top), y = fminf(fmaxf(yr, 0.f), top);

    Sample s;
    int x0 = 0, y0 = 0;
    s.fx = s.fy = 0.f;
    if (S > 1) {
        const float x0f = fminf(fmaxf(floorf(x), 0.f), (float)(S - 2));
        const float y0f = fminf(fmaxf(floorf(y), 0.f), (float)(S - 2));
        s.fx = x - x0f;
        s.fy = y - y0f;
        x0 = min(max((int)x0f, 0), S - 2);
        y0 = min(max((int)y0f, 0), S - 2);
    }
    const int x1 = min(x0 + 1, S - 1), y1 = min(y0 + 1, S - 1);
    const size_t base = (size_t)img * S;
    s.r00 = (base + x0) * S + y0;
    s.r01 = (base + x0) * S + y1;
    s.r10 = (base + x1) * S + y0;
    s.r11 = (base + x1) * S + y1;

    // d(x, y)/dp: zero where a clamp is active, and everywhere when the projection is not finite
    const float inv_p2 = __fdiv_rn(1.f, p2);
    const float cx = (S > 1 && wr >= 0.f && wr <= W - 1.f && xr >= 0.f && xr <= top) ? __fdiv_rn(1.f, sx) : 0.f;
    const float cy = (S > 1 && hr >= 0.f && hr <= H - 1.f && yr >= 0.f && yr <= top) ? __fdiv_rn(1.f, sy) : 0.f;
    s.jx0 = cx * (-248.f * inv_p2);                  // w = 248 p0 / (-p2) + 111.5
    s.jx2 = cx * (248.f * (p0 * inv_p2) * inv_p2);
    s.jy1 = cy * (248.f * inv_p2);                   // h = 248 p1 / p2 + 111.5
    s.jy2 = cy * (-248.f * (p1 * inv_p2) * inv_p2);
    if (!(finite(hr) && finite(wr) && finite(s.jx0) && finite(s.jx2) && finite(s.jy1) && finite(s.jy2)))
        s.jx0 = s.jx2 = s.jy1 = s.jy2 = 0.f;
    return s;
}

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ float lerp2(float a00, float a01, float a10, float a11, float w00, float w01, float w10, float w11) {
    return fmaf(w11, a11, fmaf(w10, a10, fmaf(w01, a01, w00 * a00)));
}

template <bool VEC>
__global__ void __launch_bounds__(256) k_bil_fwd(const float* __restrict__ rows, int ld_rows, int D, int S, int n_img,
                                                 const float* __restrict__ pos, const int32_t* __restrict__ vert_mesh,
                                                 const int32_t* __restrict__ mesh_info, int SV, int accumulate,
                                                 float* __restrict__ out, int ld_out) {
    const int v = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (v >= SV) return;
    const Sample s = locate(pos, vert_mesh, mesh_info, v, S, n_img);
    const float w00 = (1.f - s.fx) * (1.f - s.fy), w01 = (1.f - s.fx) * s.fy, w10 = s.fx * (1.f - s.fy), w11 = s.fx * s.fy;
    const float* f00 = rows + s.r00 * ld_rows;
    const float* f01 = rows + s.r01 * ld_rows;
    const float* f10 = rows + s.r10 * ld_rows;
    const float* f11 = rows + s.r11 * ld_rows;
    float* dst = out + (size_t)v * ld_out;
    if (VEC) {
        for (int c = 4 * lane_id(); c < D; c += 128) {
            const float4 a = ld4(f00 + c), b = ld4(f01 + c), e = ld4(f10 + c), f = ld4(f11 + c);
            float4 r;
            r.x = lerp2(a.x, b.x, e.x, f.x, w00, w01, w10, w11);
            r.y = lerp2(a.y, b.y, e.y, f.y, w00, w01, w10, w11);
            r.z = lerp2(a.z, b.z, e.z, f.z, w00, w01, w10, w11);
            r.w = lerp2(a.w, b.w, e.w, f.w, w00, w01, w10, w11);
            float4* o = reinterpret_cast<float4*>(dst + c);
            if (accumulate) {
                const float4 p = *o;
                r.x += p.x; r.y += p.y; r.z += p.z; r.w += p.w;
            }
            *o = r;
        }
    } else {
        for (int c = lane_id(); c < D; c += 32) {
            const float r = lerp2(__ldg(f00 + c), __ldg(f01 + c), __ldg(f10 + c), __ldg(f11 + c), w00, w01, w10, w11);
            dst[c] = accumulate ? dst[c] + r : r;
        }
    }
}

__device__ __forceinline__ void red4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// d out / d fx = (1-fy)(f10 - f00) + fy (f11 - f01);  d out / d fy = (1-fx)(f01 - f00) + fx (f11 - f10)
__device__ __forceinline__ void dterms(float g, float a00, float a01, float a10, float a11, float fx, float fy, float& gx,
                                       float& gy) {
    gx = fmaf(g, fmaf(fy, a11 - a01, (1.f - fy) * (a10 - a00)), gx);
    gy = fmaf(g, fmaf(fx, a11 - a10, (1.f - fx) * (a01 - a00)), gy);
}

template <bool VEC>
__global__ void __launch_bounds__(256) k_bil_bwd(const float* __restrict__ gout, int ld_g, const float* __restrict__ rows,
                                                 int ld_rows, int D, int S, int n_img, const float* __restrict__ pos,
                                                 const int32_t* __restrict__ vert_mesh, const int32_t* __restrict__ mesh_info,
                                                 int SV, float* __restrict__ grows, int ld_grows, float* __restrict__ gpos,
                                                 int accumulate_gpos) {
    const int v = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (v >= SV) return;
    const Sample s = locate(pos, vert_mesh, mesh_info, v, S, n_img);
    const float w00 = (1.f - s.fx) * (1.f - s.fy), w01 = (1.f - s.fx) * s.fy, w10 = s.fx * (1.f - s.fy), w11 = s.fx * s.fy;
    const float* g = gout + (size_t)v * ld_g;
    const bool want_pos = gpos != nullptr;
    float gx = 0.f, gy = 0.f;
    if (VEC) {
        for (int c = 4 * lane_id(); c < D; c += 128) {
            const float4 gg = ld4(g + c);
            if (grows) {
                red4(grows + s.r00 * ld_grows + c, w00 * gg.x, w00 * gg.y, w00 * gg.z, w00 * gg.w);
                red4(grows + s.r01 * ld_grows + c, w01 * gg.x, w01 * gg.y, w01 * gg.z, w01 * gg.w);
                red4(grows + s.r10 * ld_grows + c, w10 * gg.x, w10 * gg.y, w10 * gg.z, w10 * gg.w);
                red4(grows + s.r11 * ld_grows + c, w11 * gg.x, w11 * gg.y, w11 * gg.z, w11 * gg.w);
            }
            if (want_pos) {
                const float4 a = ld4(rows + s.r00 * ld_rows + c), b = ld4(rows + s.r01 * ld_rows + c);
                const float4 e = ld4(rows + s.r10 * ld_rows + c), f = ld4(rows + s.r11 * ld_rows + c);
                dterms(gg.x, a.x, b.x, e.x, f.x, s.fx, s.fy, gx, gy);
                dterms(gg.y, a.y, b.y, e.y, f.y, s.fx, s.fy, gx, gy);
                dterms(gg.z, a.z, b.z, e.z, f.z, s.fx, s.fy, gx, gy);
                dterms(gg.w, a.w, b.w, e.w, f.w, s.fx, s.fy, gx, gy);
            }
        }
    } else {
        for (int c = lane_id(); c < D; c += 32) {
            const float gg = g[c];
            if (grows) {
                atomicAdd(grows + s.r00 * ld_grows + c, w00 * gg);
                atomicAdd(grows + s.r01 * ld_grows + c, w01 * gg);
                atomicAdd(grows + s.r10 * ld_grows + c, w10 * gg);
                atomicAdd(grows + s.r11 * ld_grows + c, w11 * gg);
            }
            if (want_pos)
                dterms(gg, __ldg(rows + s.r00 * ld_rows + c), __ldg(rows + s.r01 * ld_rows + c),
                       __ldg(rows + s.r10 * ld_rows + c), __ldg(rows + s.r11 * ld_rows + c), s.fx, s.fy, gx, gy);
        }
    }
    if (!want_pos) return;
    gx = warp_sum(gx);
    gy = warp_sum(gy);
    if (lane_id() == 0) {
        // a zero Jacobian entry gives an exact 0 even when gx / gy are not finite (NaN feature rows)
        const float d0 = s.jx0 != 0.f ? gx * s.jx0 : 0.f;
        const float d1 = s.jy1 != 0.f ? gy * s.jy1 : 0.f;
        const float d2 = (s.jx2 != 0.f ? gx * s.jx2 : 0.f) + (s.jy2 != 0.f ? gy * s.jy2 : 0.f);
        float* o = gpos + 3 * (size_t)v;
        if (accumulate_gpos) {
            o[0] += d0;
            o[1] += d1;
            o[2] += d2;
        } else {
            o[0] = d0;
            o[1] = d1;
            o[2] = d2;
        }
    }
}

inline bool al16(const void* p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace vabil
}  // namespace mrb

using namespace mrb;
using namespace mrb::vabil;

extern "C" int mrb_vert_align_bilinear_fwd(const float* rows, int ld_rows, int D, int S, int n_img, const float* pos,
                                           const int32_t* vert_mesh, const int32_t* mesh_info, int SV, int accumulate,
                                           float* out, int ld_out, void* stream_) {
    MRB_REQUIRE(SV >= 0, "vert_align_bilinear_fwd: SV < 0");
    if (SV == 0) return MRB_OK;
    MRB_REQUIRE(rows && pos && vert_mesh && mesh_info && out, "vert_align_bilinear_fwd: null pointer");
    MRB_REQUIRE(D >= 1 && S >= 1 && n_img >= 1, "vert_align_bilinear_fwd: D, S and n_img must be >= 1");
    MRB_REQUIRE(ld_rows >= D && ld_out >= D, "vert_align_bilinear_fwd: row pitches must be >= D");
    const bool vec = D % 4 == 0 && ld_rows % 4 == 0 && ld_out % 4 == 0 && al16(rows) && al16(out);
    const dim3 grid(ceil_div(SV, 8));
    cudaStream_t s = (cudaStream_t)stream_;
    if (vec)
        k_bil_fwd<true><<<grid, 256, 0, s>>>(rows, ld_rows, D, S, n_img, pos, vert_mesh, mesh_info, SV, accumulate, out, ld_out);
    else
        k_bil_fwd<false><<<grid, 256, 0, s>>>(rows, ld_rows, D, S, n_img, pos, vert_mesh, mesh_info, SV, accumulate, out, ld_out);
    return check_launch("vert_align_bilinear_fwd");
}

extern "C" int mrb_vert_align_bilinear_bwd(const float* gout, int ld_g, const float* rows, int ld_rows, int D, int S,
                                           int n_img, const float* pos, const int32_t* vert_mesh, const int32_t* mesh_info,
                                           int SV, float* grows, int ld_grows, float* gpos, int accumulate_gpos,
                                           void* stream_) {
    MRB_REQUIRE(SV >= 0, "vert_align_bilinear_bwd: SV < 0");
    if (SV == 0) return MRB_OK;
    MRB_REQUIRE(gout && rows && pos && vert_mesh && mesh_info, "vert_align_bilinear_bwd: null pointer");
    MRB_REQUIRE(D >= 1 && S >= 1 && n_img >= 1, "vert_align_bilinear_bwd: D, S and n_img must be >= 1");
    MRB_REQUIRE(ld_g >= D && ld_rows >= D && (!grows || ld_grows >= D), "vert_align_bilinear_bwd: row pitches must be >= D");
    if (!grows && !gpos) return MRB_OK;
    const bool vec = D % 4 == 0 && ld_g % 4 == 0 && ld_rows % 4 == 0 && al16(gout) && al16(rows) &&
                     (!grows || (ld_grows % 4 == 0 && al16(grows)));
    const dim3 grid(ceil_div(SV, 8));
    cudaStream_t s = (cudaStream_t)stream_;
    if (vec)
        k_bil_bwd<true><<<grid, 256, 0, s>>>(gout, ld_g, rows, ld_rows, D, S, n_img, pos, vert_mesh, mesh_info, SV, grows,
                                             ld_grows, gpos, accumulate_gpos);
    else
        k_bil_bwd<false><<<grid, 256, 0, s>>>(gout, ld_g, rows, ld_rows, D, S, n_img, pos, vert_mesh, mesh_info, SV, grows,
                                              ld_grows, gpos, accumulate_gpos);
    return check_launch("vert_align_bilinear_bwd");
}
