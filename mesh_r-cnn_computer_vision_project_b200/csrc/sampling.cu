// Mesh surface sampling: triangle areas, per-mesh area CDF, area-weighted face draw + barycentric points,
// unit-ball normalisation, and the backward of all of it.
//
// Replaces utils/mesh_sampling.py:6-57 (`surface_areas`, `multinomial`, two `rand`, gather, weighted sum) and
// utils/process.py:7-20 (`normalize_mesh`, which builds an n x n matrix for its diagonal) plus the per-mesh
// Python loop at meshRCNN/loss_functions.py:86-87.  One launch handles the whole packed batch.
#include <cooperative_groups.h>

#include "common.cuh"
#include "../../include/meshrcnn_b200.h"

namespace mrb {
namespace sampling {

__device__ __forceinline__ double warp_inclusive_scan_f64(double v) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        double n = __shfl_up_sync(0xffffffffu, v, o);
        if (lane_id() >= o) v += n;
    }
    return v;
}

__device__ __forceinline__ float tri_area(const float* __restrict__ verts, long long a, long long b, long long c) {
    // |AB x AC| / 2  (mesh_sampling.py:46-56), fp32
    const float ax = verts[3 * a], ay = verts[3 * a + 1], az = verts[3 * a + 2];
    const float ux = verts[3 * b] - ax, uy = verts[3 * b + 1] - ay, uz = verts[3 * b + 2] - az;
    const float vx = verts[3 * c] - ax, vy = verts[3 * c + 1] - ay, vz = verts[3 * c + 2] - az;
    const float nx = uy * vz - uz * vy, ny = uz * vx - ux * vz, nz = ux * vy - uy * vx;
    return sqrtf(nx * nx + ny * ny + nz * nz) * 0.5f;
}

// areas of a packed batch; faces hold per-mesh local ids, v_off/f_off are the mesh offsets (B+1 entries)
__global__ void k_areas(const float* __restrict__ verts, const long long* __restrict__ faces,
                        const int32_t* __restrict__ v_off, const int32_t* __restrict__ f_off, int B,
                        float* __restrict__ areas) {
    const int b = blockIdx.y;
    const int f = f_off[b] + blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= f_off[b + 1]) return;
    const long long o = v_off[b];
    areas[f] = tri_area(verts, faces[3 * (size_t)f] + o, faces[3 * (size_t)f + 1] + o, faces[3 * (size_t)f + 2] + o);
}

// inclusive per-mesh CDF of the areas in fp64 (one block per mesh)
__global__ void __launch_bounds__(1024) k_cdf(const float* __restrict__ areas, const int32_t* __restrict__ f_off,
                                              double* __restrict__ cdf) {
    __shared__ double wsum[33];
    const int b = blockIdx.x;
    const int beg = f_off[b], end = f_off[b + 1];
    double carry = 0.0;
    for (int base = beg; base < end; base += 1024) {
        const int i = base + threadIdx.x;
        const double v = (i < end) ? (double)areas[i] : 0.0;
        double inc = warp_inclusive_scan_f64(v);
        __syncthreads();
        if (lane_id() == 31) wsum[warp_id()] = inc;
        __syncthreads();
        if (warp_id() == 0) {
            double w = wsum[lane_id()];
            double winc = warp_inclusive_scan_f64(w);
            wsum[lane_id()] = winc - w;
            if (lane_id() == 31) wsum[32] = winc;
        }
        __syncthreads();
        if (i < end) cdf[i] = carry + wsum[warp_id()] + inc;
        carry += wsum[32];
    }
}

// Philox4x32-10 counter RNG (own implementation; one call yields 4 x 32 random bits)
__device__ __forceinline__ uint4 philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }   // [0,1)

// One area-weighted surface draw: global face id, global corner vertex ids and barycentric weights of point i of mesh b
// (pi = b * n + i), from the injected draws or from Philox(i, b, seed).  Shared by k_sample and k_sample_surface, so both
// draw the same point for the same randomness.
struct SurfaceDraw {
    int f;
    long long a, b, c;
    float w0, w1, w2;
};

__device__ __forceinline__ SurfaceDraw draw_surface_point(const long long* __restrict__ faces, const int32_t* __restrict__ v_off,
                                                          const int32_t* __restrict__ f_off, const double* __restrict__ cdf,
                                                          const float* __restrict__ u_in, const long long* __restrict__ fidx_in,
                                                          const float* __restrict__ xi2_in, const float* __restrict__ xi1_in,
                                                          unsigned long long seed, int b, int i, size_t pi) {
    const int fb = f_off[b], fe = f_off[b + 1];
    float u, xi2, xi1;
    if (xi2_in) {
        xi2 = xi2_in[pi]; xi1 = xi1_in[pi]; u = u_in ? u_in[pi] : 0.f;
    } else {
        const uint4 r = philox4x32((uint32_t)i, (uint32_t)b, 0x5eedu, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
        u = u01(r.x); xi2 = u01(r.y); xi1 = u01(r.z);
    }
    SurfaceDraw s;
    if (fidx_in) {
        s.f = fb + (int)fidx_in[pi];
    } else {
        // inverse CDF: first face whose inclusive cumulative area exceeds u * total (multinomial, :16)
        const double target = (double)u * cdf[fe - 1];
        int lo = fb, hi = fe - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (cdf[mid] > target) hi = mid; else lo = mid + 1;
        }
        s.f = lo;
    }
    const long long o = v_off[b];
    s.a = faces[3 * (size_t)s.f] + o; s.b = faces[3 * (size_t)s.f + 1] + o; s.c = faces[3 * (size_t)s.f + 2] + o;
    const float r = sqrtf(xi1);                          // :21
    s.w0 = 1.0f - r; s.w1 = (1.0f - xi2) * r; s.w2 = xi2 * r;   // :23-25
    return s;
}

// coordinate d of the drawn point (the weighted sum of mesh_sampling.py:27-35)
__device__ __forceinline__ float surface_coord(const SurfaceDraw& s, const float* __restrict__ verts, int d) {
    return fmaf(s.w2, verts[3 * s.c + d], fmaf(s.w1, verts[3 * s.b + d], s.w0 * verts[3 * s.a + d]));
}

// one thread per sampled point
__global__ void __launch_bounds__(256) k_sample(const float* __restrict__ verts, const long long* __restrict__ faces,
                                                const int32_t* __restrict__ v_off, const int32_t* __restrict__ f_off,
                                                const double* __restrict__ cdf, int n,
                                                const float* __restrict__ u_in, const long long* __restrict__ fidx_in,
                                                const float* __restrict__ xi2_in, const float* __restrict__ xi1_in,
                                                unsigned long long seed, float* __restrict__ raw,
                                                int32_t* __restrict__ fidx_out, float* __restrict__ w_out) {
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t pi = (size_t)b * n + i;
    const SurfaceDraw s = draw_surface_point(faces, v_off, f_off, cdf, u_in, fidx_in, xi2_in, xi1_in, seed, b, i, pi);
#pragma unroll
    for (int d = 0; d < 3; ++d) raw[3 * pi + d] = surface_coord(s, verts, d);
    fidx_out[pi] = s.f;
    w_out[3 * pi] = s.w0; w_out[3 * pi + 1] = s.w1; w_out[3 * pi + 2] = s.w2;
}

// Eval-side sampling (no backward): the k_sample point times an optional per-mesh scale (no unit-ball normalisation), the
// unit normal (B-A)x(C-A)/|.| of its face (zero vector for a degenerate face) and the global face id.
__global__ void __launch_bounds__(256) k_sample_surface(const float* __restrict__ verts, const long long* __restrict__ faces,
                                                        const int32_t* __restrict__ v_off, const int32_t* __restrict__ f_off,
                                                        const double* __restrict__ cdf, int n,
                                                        const float* __restrict__ u_in, const long long* __restrict__ fidx_in,
                                                        const float* __restrict__ xi2_in, const float* __restrict__ xi1_in,
                                                        unsigned long long seed, const float* __restrict__ scale,
                                                        float* __restrict__ points, float* __restrict__ normals,
                                                        int32_t* __restrict__ fidx_out) {
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t pi = (size_t)b * n + i;
    const SurfaceDraw s = draw_surface_point(faces, v_off, f_off, cdf, u_in, fidx_in, xi2_in, xi1_in, seed, b, i, pi);
    const float sc = scale ? scale[b] : 1.0f;            // x * 1.0f == x: unscaled points equal k_sample's raw points
#pragma unroll
    for (int d = 0; d < 3; ++d) points[3 * pi + d] = sc * surface_coord(s, verts, d);
    const float ax = verts[3 * s.a], ay = verts[3 * s.a + 1], az = verts[3 * s.a + 2];
    const float ux = verts[3 * s.b] - ax, uy = verts[3 * s.b + 1] - ay, uz = verts[3 * s.b + 2] - az;
    const float vx = verts[3 * s.c] - ax, vy = verts[3 * s.c + 1] - ay, vz = verts[3 * s.c + 2] - az;
    const float nx = uy * vz - uz * vy, ny = uz * vx - ux * vz, nz = ux * vy - uy * vx;
    const float len = sqrtf(nx * nx + ny * ny + nz * nz);
    normals[3 * pi] = len > 0.f ? nx / len : 0.f;
    normals[3 * pi + 1] = len > 0.f ? ny / len : 0.f;
    normals[3 * pi + 2] = len > 0.f ? nz / len : 0.f;
    fidx_out[pi] = s.f;
}

struct Stats {   // per cloud, 8 doubles
    double mean[3];
    double factor;   // 1 when no rescale
    double argmax;   // index of the max-norm row (as double), -1 when no rescale
    double pad[3];
};

// normalize_mesh (process.py:11-20): centre by the mean; if max |coord| > 1 divide by the largest row norm.
// One block per cloud; fp64 accumulation.
__global__ void __launch_bounds__(1024) k_normalize(const float* __restrict__ raw, int n, float* __restrict__ out,
                                                    double* __restrict__ stats) {
    __shared__ double sd[33];
    __shared__ double s_mean[3];
    __shared__ double s_best[32];
    __shared__ int s_besti[32];
    const int b = blockIdx.x;
    const float* x = raw + (size_t)b * n * 3;
    for (int d = 0; d < 3; ++d) {
        double acc = 0.0;
        for (int i = threadIdx.x; i < n; i += blockDim.x) acc += (double)x[3 * i + d];
        acc = block_sum<double>(acc, sd);
        if (threadIdx.x == 0) s_mean[d] = acc / (double)n;
        __syncthreads();
    }
    const double m0 = s_mean[0], m1 = s_mean[1], m2 = s_mean[2];
    double amax = 0.0, best = -1.0;
    int besti = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double c0 = x[3 * i] - m0, c1 = x[3 * i + 1] - m1, c2 = x[3 * i + 2] - m2;
        amax = fmax(amax, fmax(fabs(c0), fmax(fabs(c1), fabs(c2))));
        const double r2 = c0 * c0 + c1 * c1 + c2 * c2;
        if (r2 > best) { best = r2; besti = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
    }
    __syncthreads();
    if (lane_id() == 0) { sd[warp_id()] = amax; s_best[warp_id()] = best; s_besti[warp_id()] = besti; }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int nw = blockDim.x >> 5;
        for (int w = 1; w < nw; ++w) {
            amax = fmax(amax, sd[w]);
            if (s_best[w] > best || (s_best[w] == best && s_besti[w] < besti)) { best = s_best[w]; besti = s_besti[w]; }
        }
        const bool scale = amax > 1.0;
        double* st = stats + 8 * (size_t)b;
        st[0] = m0; st[1] = m1; st[2] = m2;
        st[3] = scale ? sqrt(best) : 1.0;
        st[4] = scale ? (double)besti : -1.0;
        sd[32] = st[3];
    }
    __syncthreads();
    const double inv = 1.0 / sd[32];
    float* y = out + (size_t)b * n * 3;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        y[3 * i] = (float)((x[3 * i] - m0) * inv);
        y[3 * i + 1] = (float)((x[3 * i + 1] - m1) * inv);
        y[3 * i + 2] = (float)((x[3 * i + 2] - m2) * inv);
    }
}

// Same result with a thread-block CLUSTER of NORM_CTAS CTAs per cloud (clouds of <= NORM_CTAS * 256 * NORM_PPT points, i.e. the
// 10 000-point loss clouds): every thread keeps its points in registers (one global read instead of five strided passes by a
// single CTA), the partial sums / maxima of the CTAs are exchanged through distributed shared memory
// (cluster.map_shared_rank) between two cluster barriers and combined in rank order (deterministic).  21 us -> ~6 us per call.
constexpr int NORM_CTAS = 8, NORM_THREADS = 256, NORM_PPT = 8;

__global__ void __cluster_dims__(NORM_CTAS, 1, 1) __launch_bounds__(NORM_THREADS)
k_normalize_cluster(const float* __restrict__ raw, int n, float* __restrict__ out, double* __restrict__ stats) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double sd[33];
    __shared__ double part[8];          // [0..2] coordinate sums, [3] max |centred coord|, [4] best r^2
    __shared__ int part_i[1];           // index of the best r^2
    __shared__ double s_best[NORM_THREADS / 32];
    __shared__ int s_besti[NORM_THREADS / 32];
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.x / NORM_CTAS;
    const float* x = raw + (size_t)b * n * 3;
    const int chunk = (n + NORM_CTAS - 1) / NORM_CTAS;
    const int lo = rank * chunk, hi = min(n, lo + chunk);
    float px[NORM_PPT], py[NORM_PPT], pz[NORM_PPT];
    double a0 = 0.0, a1 = 0.0, a2 = 0.0;
#pragma unroll
    for (int u = 0; u < NORM_PPT; ++u) {
        const int i = lo + u * NORM_THREADS + threadIdx.x;
        px[u] = py[u] = pz[u] = 0.f;
        if (i < hi) { px[u] = x[3 * i]; py[u] = x[3 * i + 1]; pz[u] = x[3 * i + 2]; }
    }
#pragma unroll
    for (int u = 0; u < NORM_PPT; ++u) { a0 += (double)px[u]; a1 += (double)py[u]; a2 += (double)pz[u]; }   // absent points add 0
    a0 = block_sum<double>(a0, sd);
    a1 = block_sum<double>(a1, sd);
    a2 = block_sum<double>(a2, sd);
    if (threadIdx.x == 0) { part[0] = a0; part[1] = a1; part[2] = a2; }
    cluster.sync();
    double m0 = 0.0, m1 = 0.0, m2 = 0.0;
    for (int r = 0; r < NORM_CTAS; ++r) {
        const double* rp = cluster.map_shared_rank(part, r);
        m0 += rp[0]; m1 += rp[1]; m2 += rp[2];
    }
    m0 /= (double)n; m1 /= (double)n; m2 /= (double)n;
    double amax = 0.0, best = -1.0;
    int besti = 0;
#pragma unroll
    for (int u = 0; u < NORM_PPT; ++u) {
        const int i = lo + u * NORM_THREADS + threadIdx.x;
        if (i < hi) {
            const double c0 = px[u] - m0, c1 = py[u] - m1, c2 = pz[u] - m2;
            amax = fmax(amax, fmax(fabs(c0), fmax(fabs(c1), fabs(c2))));
            const double r2 = c0 * c0 + c1 * c1 + c2 * c2;
            if (r2 > best) { best = r2; besti = i; }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        amax = fmax(amax, __shfl_xor_sync(0xffffffffu, amax, o));
        const double ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
        if (ob > best || (ob == best && oi < besti)) { best = ob; besti = oi; }
    }
    if (lane_id() == 0) { sd[warp_id()] = amax; s_best[warp_id()] = best; s_besti[warp_id()] = besti; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < NORM_THREADS / 32; ++w) {
            amax = fmax(amax, sd[w]);
            if (s_best[w] > best || (s_best[w] == best && s_besti[w] < besti)) { best = s_best[w]; besti = s_besti[w]; }
        }
        part[3] = amax; part[4] = best; part_i[0] = besti;
    }
    cluster.sync();
    amax = 0.0; best = -1.0; besti = 0;
    for (int r = 0; r < NORM_CTAS; ++r) {
        const double* rp = cluster.map_shared_rank(part, r);
        const int ri = *cluster.map_shared_rank(part_i, r);
        amax = fmax(amax, rp[3]);
        if (rp[4] > best || (rp[4] == best && ri < besti)) { best = rp[4]; besti = ri; }
    }
    const bool scale = amax > 1.0;
    const double norm = scale ? sqrt(best) : 1.0;
    if (rank == 0 && threadIdx.x == 0) {
        double* st = stats + 8 * (size_t)b;
        st[0] = m0; st[1] = m1; st[2] = m2;
        st[3] = norm;
        st[4] = scale ? (double)besti : -1.0;
    }
    const double inv = 1.0 / norm;
    float* y = out + (size_t)b * n * 3;
#pragma unroll
    for (int u = 0; u < NORM_PPT; ++u) {
        const int i = lo + u * NORM_THREADS + threadIdx.x;
        if (i < hi) {
            y[3 * i] = (float)((px[u] - m0) * inv);
            y[3 * i + 1] = (float)((py[u] - m1) * inv);
            y[3 * i + 2] = (float)((pz[u] - m2) * inv);
        }
    }
    cluster.sync();          // remote shared memory must stay alive until every CTA of the cluster has read it
}

static void launch_normalize(const float* raw, int B, int n, float* cloud, double* stats, cudaStream_t s) {
    if (n <= NORM_CTAS * NORM_THREADS * NORM_PPT) k_normalize_cluster<<<B * NORM_CTAS, NORM_THREADS, 0, s>>>(raw, n, cloud, stats);
    else k_normalize<<<B, 1024, 0, s>>>(raw, n, cloud, stats);
}

// backward of normalise + barycentric combination, two launches over the whole batch:
//   k_sample_bwd_sums : tot[b] = (sum_i g_i, sum_i g_i . y_i)  -- 8 blocks per cloud, fp64 atomics into tot (zeroed)
//   k_sample_bwd      : one thread per sampled point scatters into gverts (atomics)
constexpr int BWD_SPLIT = 8;
__global__ void __launch_bounds__(256) k_sample_bwd_sums(const float* __restrict__ gy, const float* __restrict__ y, int n,
                                                         double* __restrict__ tot) {
    __shared__ double sd[33];
    const int b = blockIdx.y;
    const size_t base = (size_t)b * n;
    double acc[4] = {0, 0, 0, 0};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const double g0 = gy[3 * (base + i)], g1 = gy[3 * (base + i) + 1], g2 = gy[3 * (base + i) + 2];
        acc[0] += g0; acc[1] += g1; acc[2] += g2;
        acc[3] += g0 * y[3 * (base + i)] + g1 * y[3 * (base + i) + 1] + g2 * y[3 * (base + i) + 2];
    }
    for (int d = 0; d < 4; ++d) {
        const double t = block_sum<double>(acc[d], sd);
        if (threadIdx.x == 0) atomicAdd(tot + 4 * (size_t)b + d, t);
        __syncthreads();
    }
}

// PAD4: gverts rows are 4 floats wide (16-byte aligned), one red.global.add.v4.f32 per face corner instead of three atomics
template <bool PAD4>
__global__ void __launch_bounds__(256) k_sample_bwd(const float* __restrict__ gy, const float* __restrict__ y,
                                                    const double* __restrict__ stats, const double* __restrict__ tot,
                                                    const int32_t* __restrict__ fidx, const float* __restrict__ w,
                                                    const long long* __restrict__ faces, const int32_t* __restrict__ v_off, int n,
                                                    float* __restrict__ gverts) {
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t base = (size_t)b * n;
    const double f = stats[8 * (size_t)b + 3];
    const int am = (int)stats[8 * (size_t)b + 4];
    // gc_i = g_i / f  (+ for i == argmax:  -(s / f) * y_m);   gx_i = gc_i - mean_j gc_j
    double extra[3] = {0, 0, 0};
    if (am >= 0) {
        const double k = -tot[4 * (size_t)b + 3] / f;
        for (int d = 0; d < 3; ++d) extra[d] = k * (double)y[3 * (base + am) + d];
    }
    float gx[3];
    for (int d = 0; d < 3; ++d) {
        const double gmean = (tot[4 * (size_t)b + d] / f + extra[d]) / (double)n;
        double g = (double)gy[3 * (base + i) + d] / f - gmean;
        if (i == am) g += extra[d];
        gx[d] = (float)g;
    }
    const long long o = v_off[b];
    const int fi = fidx[base + i];
    for (int c = 0; c < 3; ++c) {
        const long long v = faces[3 * (size_t)fi + c] + o;
        const float wc = w[3 * (base + i) + c];
        if (PAD4) {
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(gverts + 4 * v), "f"(wc * gx[0]), "f"(wc * gx[1]),
                         "f"(wc * gx[2]), "f"(0.f)
                         : "memory");
        } else {
            atomicAdd(gverts + 3 * v, wc * gx[0]);
            atomicAdd(gverts + 3 * v + 1, wc * gx[1]);
            atomicAdd(gverts + 3 * v + 2, wc * gx[2]);
        }
    }
}

}  // namespace sampling
}  // namespace mrb

using namespace mrb;
using namespace mrb::sampling;

extern "C" int mrb_face_areas(const float* verts, const long long* faces, const int32_t* v_off, const int32_t* f_off,
                              int B, int max_faces, float* areas, void* stream_) {
    MRB_REQUIRE(verts && faces && v_off && f_off && areas, "face_areas: null pointer");
    if (B == 0 || max_faces == 0) return MRB_OK;
    k_areas<<<dim3(ceil_div(max_faces, 256), B), 256, 0, (cudaStream_t)stream_>>>(verts, faces, v_off, f_off, B, areas);
    return check_launch("face_areas");
}

extern "C" int mrb_face_area_cdf(const float* verts, const long long* faces, const int32_t* v_off, const int32_t* f_off,
                                 int B, int max_faces, float* areas, double* cdf, void* stream_) {
    MRB_REQUIRE(verts && faces && v_off && f_off && areas && cdf, "face_area_cdf: null pointer");
    if (B == 0 || max_faces == 0) return MRB_OK;
    cudaStream_t s = (cudaStream_t)stream_;
    k_areas<<<dim3(ceil_div(max_faces, 256), B), 256, 0, s>>>(verts, faces, v_off, f_off, B, areas);
    k_cdf<<<B, 1024, 0, s>>>(areas, f_off, cdf);
    return check_launch("face_area_cdf");
}

extern "C" int mrb_sample_points_fwd(const float* verts, const long long* faces, const int32_t* v_off,
                                     const int32_t* f_off, const double* cdf, int B, int n, const float* u,
                                     const long long* face_idx, const float* xi2, const float* xi1,
                                     unsigned long long seed, float* raw, int32_t* fidx_out, float* w_out,
                                     float* cloud, double* stats, void* stream_) {
    MRB_REQUIRE(verts && faces && v_off && f_off && raw && fidx_out && w_out && cloud && stats,
                "sample_points_fwd: null pointer");
    MRB_REQUIRE(cdf || face_idx, "sample_points_fwd: need a CDF or injected face indices");
    MRB_REQUIRE((xi2 == nullptr) == (xi1 == nullptr), "sample_points_fwd: xi1/xi2 must be given together");
    MRB_REQUIRE(face_idx || xi2 == nullptr || u, "sample_points_fwd: injected xi needs injected u or face_idx");
    if (B == 0 || n == 0) return MRB_OK;
    cudaStream_t s = (cudaStream_t)stream_;
    k_sample<<<dim3(ceil_div(n, 256), B), 256, 0, s>>>(verts, faces, v_off, f_off, cdf, n, u, face_idx, xi2, xi1, seed,
                                                         raw, fidx_out, w_out);
    launch_normalize(raw, B, n, cloud, stats, s);
    return check_launch("sample_points_fwd");
}

extern "C" int mrb_sample_surface_fwd(const float* verts, const long long* faces, const int32_t* v_off,
                                      const int32_t* f_off, const double* cdf, int B, int n, const float* u,
                                      const long long* face_idx, const float* xi2, const float* xi1, unsigned long long seed,
                                      const float* scale, float* points, float* normals, int32_t* fidx_out, void* stream_) {
    MRB_REQUIRE(verts && faces && v_off && f_off && points && normals && fidx_out, "sample_surface_fwd: null pointer");
    MRB_REQUIRE(cdf || face_idx, "sample_surface_fwd: need a CDF or injected face indices");
    MRB_REQUIRE((xi2 == nullptr) == (xi1 == nullptr), "sample_surface_fwd: xi1/xi2 must be given together");
    MRB_REQUIRE(face_idx || xi2 == nullptr || u, "sample_surface_fwd: injected xi needs injected u or face_idx");
    MRB_REQUIRE(B <= 65535, "sample_surface_fwd: batch too large");
    if (B == 0 || n == 0) return MRB_OK;
    k_sample_surface<<<dim3(ceil_div(n, 256), B), 256, 0, (cudaStream_t)stream_>>>(verts, faces, v_off, f_off, cdf, n, u, face_idx,
                                                                                   xi2, xi1, seed, scale, points, normals,
                                                                                   fidx_out);
    return check_launch("sample_surface_fwd");
}

extern "C" int mrb_normalize_cloud_fwd(const float* raw, int B, int n, float* cloud, double* stats, void* stream_) {
    MRB_REQUIRE(raw && cloud && stats, "normalize_cloud_fwd: null pointer");
    if (B == 0 || n == 0) return MRB_OK;
    launch_normalize(raw, B, n, cloud, stats, (cudaStream_t)stream_);
    return check_launch("normalize_cloud_fwd");
}

static int launch_sample_bwd(const float* gcloud, const float* cloud, const double* stats, const int32_t* fidx, const float* w,
                             const long long* faces, const int32_t* v_off, int B, int n, float* gverts, int ld_gverts,
                             double* scratch, void* stream_) {
    MRB_REQUIRE(gcloud && cloud && stats && fidx && w && faces && v_off && gverts && scratch, "sample_points_bwd: null pointer");
    MRB_REQUIRE(B <= 65535, "sample_points_bwd: batch too large");
    MRB_REQUIRE(ld_gverts == 3 || (ld_gverts == 4 && ((uintptr_t)gverts & 15) == 0),
                "sample_points_bwd: gradient rows must be 3 floats, or 4 floats and 16-byte aligned (got ld = %d)", ld_gverts);
    if (B == 0 || n == 0) return MRB_OK;
    cudaStream_t s = (cudaStream_t)stream_;
    cudaMemsetAsync(scratch, 0, sizeof(double) * 4 * (size_t)B, s);
    k_sample_bwd_sums<<<dim3(BWD_SPLIT, B), 256, 0, s>>>(gcloud, cloud, n, scratch);
    const dim3 grid(ceil_div(n, 256), B);
    if (ld_gverts == 4) k_sample_bwd<true><<<grid, 256, 0, s>>>(gcloud, cloud, stats, scratch, fidx, w, faces, v_off, n, gverts);
    else k_sample_bwd<false><<<grid, 256, 0, s>>>(gcloud, cloud, stats, scratch, fidx, w, faces, v_off, n, gverts);
    return check_launch("sample_points_bwd");
}

extern "C" int mrb_sample_points_bwd(const float* gcloud, const float* cloud, const double* stats, const int32_t* fidx,
                                     const float* w, const long long* faces, const int32_t* v_off, int B, int n,
                                     float* gverts, double* scratch, void* stream_) {
    return launch_sample_bwd(gcloud, cloud, stats, fidx, w, faces, v_off, B, n, gverts, 3, scratch, stream_);
}

extern "C" int mrb_sample_points_bwd_ld(const float* gcloud, const float* cloud, const double* stats, const int32_t* fidx,
                                        const float* w, const long long* faces, const int32_t* v_off, int B, int n,
                                        float* gverts, int ld_gverts, double* scratch, void* stream_) {
    return launch_sample_bwd(gcloud, cloud, stats, fidx, w, faces, v_off, B, n, gverts, ld_gverts, scratch, stream_);
}
