// Per-mesh evaluation metrics (the Mesh R-CNN paper's protocol): the GT-10 scale of a packed vertex buffer, and Chamfer-L2,
// normal consistency and precision / recall / F1 at distance thresholds from the nearest-neighbour outputs of mrb_knn_fwd.
// Every sum is accumulated in fp64 in a fixed order (per-thread strided loop, xor-shuffle tree, warps in index order), so
// repeated calls give bitwise-equal results.
#include <cooperative_groups.h>

#include "common.cuh"
#include "../../include/meshrcnn_b200.h"

namespace mrb {
namespace metrics {

constexpr int SCALE_THREADS = 256;
constexpr int MET_THREADS = 512;
constexpr int MAX_TAU = 8;

// scale[b] = target / (longest side of the bounding box of vertices [v_off[b], v_off[b+1])), one CTA per mesh.  fp32 min / max
// are exact and order-free; a mesh of zero extent gets target / 0 = inf.
__global__ void __launch_bounds__(SCALE_THREADS) k_gt_scale(const float* __restrict__ verts, const int32_t* __restrict__ v_off,
                                                            float target, float* __restrict__ scale) {
    __shared__ float s_lo[3][SCALE_THREADS / 32], s_hi[3][SCALE_THREADS / 32];
    const int b = blockIdx.x;
    const int beg = v_off[b], end = v_off[b + 1];
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int v = beg + threadIdx.x; v < end; v += SCALE_THREADS) {
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const float x = verts[3 * (size_t)v + d];
            lo[d] = fminf(lo[d], x);
            hi[d] = fmaxf(hi[d], x);
        }
    }
#pragma unroll
    for (int d = 0; d < 3; ++d) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
            hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
        }
        if (lane_id() == 0) { s_lo[d][warp_id()] = lo[d]; s_hi[d][warp_id()] = hi[d]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float ext = 0.f;
        for (int d = 0; d < 3; ++d) {
            float l = s_lo[d][0], h = s_hi[d][0];
            for (int w = 1; w < SCALE_THREADS / 32; ++w) { l = fminf(l, s_lo[d][w]); h = fmaxf(h, s_hi[d][w]); }
            ext = fmaxf(ext, h - l);
        }
        scale[b] = target / ext;
    }
}

struct Taus {
    float t[MAX_TAU];   // unused entries are -inf: no distance is below them
    int n;
};

// One cluster of two CTAs per mesh: rank 0 reduces the predicted -> GT direction (d_p, i_p, own normals n_p), rank 1 the
// GT -> predicted one.  Each CTA forms sum d, sum n.m, sum |n.m| (fp64) and the hit count of every threshold (int); rank 0
// reads rank 1's partials through distributed shared memory and writes the row of the mesh.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(MET_THREADS)
k_mesh_metrics(const float* __restrict__ d_p, const int32_t* __restrict__ i_p, const float* __restrict__ d_q,
               const int32_t* __restrict__ i_q, const float* __restrict__ n_p, const float* __restrict__ n_q, int P, int Q,
               const __grid_constant__ Taus taus, float* __restrict__ out) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    constexpr int NW = MET_THREADS / 32;
    __shared__ double w_sum[3][NW];
    __shared__ int w_cnt[MAX_TAU][NW];
    __shared__ double part[3];
    __shared__ int part_cnt[MAX_TAU];
    const int dir = (int)cluster.block_rank();
    const int b = blockIdx.x >> 1;
    const int n = dir ? Q : P, m = dir ? P : Q;
    const float* d = (dir ? d_q : d_p) + (size_t)b * n;
    const int32_t* nn = (dir ? i_q : i_p) + (size_t)b * n;
    const float* own = (dir ? n_q : n_p) + 3 * (size_t)b * n;
    const float* other = (dir ? n_p : n_q) + 3 * (size_t)b * m;
    double s_d = 0.0, s_dot = 0.0, s_abs = 0.0;
    int cnt[MAX_TAU];
#pragma unroll
    for (int t = 0; t < MAX_TAU; ++t) cnt[t] = 0;
    for (int i = threadIdx.x; i < n; i += MET_THREADS) {
        const float di = d[i];
        const size_t j = (size_t)nn[i];
        const double dot = (double)own[3 * i] * other[3 * j] + (double)own[3 * i + 1] * other[3 * j + 1] +
                           (double)own[3 * i + 2] * other[3 * j + 2];
        s_d += (double)di;
        s_dot += dot;
        s_abs += fabs(dot);
        const float r = sqrtf(di);                       // IEEE fp32 sqrt, compared with the fp32 threshold
#pragma unroll
        for (int t = 0; t < MAX_TAU; ++t) cnt[t] += r < taus.t[t] ? 1 : 0;
    }
    s_d = warp_sum(s_d);
    s_dot = warp_sum(s_dot);
    s_abs = warp_sum(s_abs);
#pragma unroll
    for (int t = 0; t < MAX_TAU; ++t) cnt[t] = warp_sum(cnt[t]);
    if (lane_id() == 0) {
        w_sum[0][warp_id()] = s_d; w_sum[1][warp_id()] = s_dot; w_sum[2][warp_id()] = s_abs;
#pragma unroll
        for (int t = 0; t < MAX_TAU; ++t) w_cnt[t][warp_id()] = cnt[t];
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double a = 0.0;
        for (int w = 0; w < NW; ++w) a += w_sum[threadIdx.x][w];
        part[threadIdx.x] = a;
    } else if (threadIdx.x < 3 + MAX_TAU) {
        int a = 0;
        for (int w = 0; w < NW; ++w) a += w_cnt[threadIdx.x - 3][w];
        part_cnt[threadIdx.x - 3] = a;
    }
    cluster.sync();
    if (dir == 0 && threadIdx.x == 0) {
        const double* rq = cluster.map_shared_rank(part, 1);
        const int* cq = cluster.map_shared_rank(part_cnt, 1);
        const double np = (double)P, nq = (double)Q;
        float* o = out + (size_t)b * (3 + 3 * taus.n);
        o[0] = (float)(part[0] / np + rq[0] / nq);
        o[1] = (float)(0.5 * (part[1] / np + rq[1] / nq));
        o[2] = (float)(0.5 * (part[2] / np + rq[2] / nq));
        for (int t = 0; t < taus.n; ++t) {
            const double prec = 100.0 * (double)part_cnt[t] / np, rec = 100.0 * (double)cq[t] / nq;
            o[3 + 3 * t] = (float)prec;
            o[4 + 3 * t] = (float)rec;
            o[5 + 3 * t] = (float)(2.0 * prec * rec / (prec + rec + 1e-8));
        }
    }
    cluster.sync();          // rank 1's shared memory must stay alive until rank 0 has read it
}

}  // namespace metrics
}  // namespace mrb

using namespace mrb;
using namespace mrb::metrics;

extern "C" int mrb_mesh_gt_scale(const float* verts, const int32_t* v_off, int B, float target, float* scale, void* stream_) {
    MRB_REQUIRE(verts && v_off && scale, "mesh_gt_scale: null pointer");
    if (B == 0) return MRB_OK;
    k_gt_scale<<<B, SCALE_THREADS, 0, (cudaStream_t)stream_>>>(verts, v_off, target, scale);
    return check_launch("mesh_gt_scale");
}

extern "C" int mrb_mesh_metrics(const float* d_p, const int32_t* i_p, const float* d_q, const int32_t* i_q, const float* n_p,
                                const float* n_q, int B, int P, int Q, const float* tau_host, int T, float* out, void* stream_) {
    MRB_REQUIRE(d_p && i_p && d_q && i_q && n_p && n_q && out, "mesh_metrics: null pointer");
    MRB_REQUIRE(T >= 0 && T <= MAX_TAU && (tau_host || T == 0), "mesh_metrics: 0..%d thresholds (got %d)", MAX_TAU, T);
    MRB_REQUIRE(B == 0 || (P > 0 && Q > 0), "mesh_metrics: every cloud needs at least one point (P = %d, Q = %d)", P, Q);
    if (B == 0) return MRB_OK;
    Taus taus;
    taus.n = T;
    for (int t = 0; t < MAX_TAU; ++t) taus.t[t] = t < T ? tau_host[t] : -INFINITY;
    k_mesh_metrics<<<2 * B, MET_THREADS, 0, (cudaStream_t)stream_>>>(d_p, i_p, d_q, i_q, n_p, n_q, P, Q, taus, out);
    return check_launch("mesh_metrics");
}
