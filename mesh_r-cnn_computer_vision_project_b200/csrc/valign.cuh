// Camera projection shared by the reference-mode VertexAlign kernels (align_proj.cu, graphconv2.cu).
#pragma once
#include "common.cuh"

namespace mrb {
namespace valign {

struct Texel {
    int img;     // image index
    int xy;      // x1 * Wm + y1
    int valid;   // mask
};

// per-mesh record: image index, image height, image width
__device__ __forceinline__ Texel project(const float* __restrict__ pos, const int32_t* __restrict__ vert_mesh,
                                         const int32_t* __restrict__ mesh_info, int v, int Hm, int Wm) {
    const int mesh = vert_mesh[v];
    const int img = mesh_info[3 * mesh + 0];
    const float H = (float)mesh_info[3 * mesh + 1], W = (float)mesh_info[3 * mesh + 2];
    const float p0 = pos[3 * (size_t)v + 0], p1 = pos[3 * (size_t)v + 1], p2 = pos[3 * (size_t)v + 2];
    // layers.py:557-558 (separate fp32 ops: div, mul, add)
    float h = __fadd_rn(__fmul_rn(248.f, __fdiv_rn(p1, p2)), 111.5f);
    float w = __fadd_rn(__fmul_rn(248.f, __fdiv_rn(p0, -p2)), 111.5f);
    // :561-562  clamp(min=0, max=H-1)
    h = fminf(fmaxf(h, 0.f), H - 1.f);
    w = fminf(fmaxf(w, 0.f), W - 1.f);
    // :577-578  divisor is a python double cast to fp32; true division
    const float sx = (float)((double)mesh_info[3 * mesh + 2] / (double)Wm);
    const float sy = (float)((double)mesh_info[3 * mesh + 1] / (double)Hm);
    const float x = __fdiv_rn(w, sx), y = __fdiv_rn(h, sy);
    const int x1 = (int)floorf(x), y1 = (int)floorf(y);
    const int x2 = min((int)ceilf(x), Wm - 1), y2 = min((int)ceilf(y), Hm - 1);   // :583-584
    Texel t;
    t.img = img;
    // x (from w, scaled by size_x = last dim) indexes the H axis; y indexes the W axis (:587)
    t.xy = x1 * Wm + y1;
    t.valid = (x2 > x1) && (y2 > y1) && x1 >= 0 && y1 >= 0 && x1 < Hm && y1 < Wm;
    return t;
}

}  // namespace valign
}  // namespace mrb
