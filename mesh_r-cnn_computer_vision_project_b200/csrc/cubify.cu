// Cubify: voxel occupancy probabilities -> packed triangle meshes + sorted COO / CSR adjacency.
//
// Replaces Cubify.forward (reference meshRCNN/layers.py:403-484): threshold + conv3d + nonzero + 6 masked
// index ops + argsort + unique(dim=0) + a Python dict over every vertex/face key + unique(dim=1).
//
// B200 design: every output order of the reference is a scan order (SURVEY.md 8a-1):
//   faces     : (b, dir, z, y, x), two triangles per exposed quad
//   vertices  : (b, z, y, x) over the (Z+1)(Y+1)(X+1) corner lattice  (== torch.unique(dim=0) order)
//   adjacency : (row, col)  == CSR with sorted columns                (== torch.unique(dim=1) order)
// so no sort, no hash table and no dictionary are needed: flags -> block counts -> one small scan ->
// (host reads 2B+3 counters once, the API returns Python lists) -> emit.  All kernels are HBM-bound byte /
// integer work: one coalesced pass over the probabilities (4 B/voxel), a 1 B/voxel face-flag array that stays
// L2 resident, and coalesced int64 output streams (24 B/face, 16 B/directed edge, 12 B/vertex).
#include "common.cuh"
#include "../../include/meshrcnn_b200.h"

namespace mrb {
namespace cubify {

constexpr int CH = 512;  // items (voxels or lattice points) per block

// neighbour whose emptiness exposes the face, (dz,dy,dx) per direction -- layers.py:357-362
__constant__ int kNbr[6][3] = {{-1, 0, 0}, {1, 0, 0}, {0, 1, 0}, {0, -1, 0}, {0, 0, -1}, {0, 0, 1}};
// quad corners c0..c3 per direction as lattice offsets {0,1}^3 in (z,y,x) -- layers.py:370-400
// (dirs 2/3 sit on the side opposite the empty neighbour: reference quirk kept for bit-exactness)
__constant__ int kCorner[6][4][3] = {
    {{0, 0, 0}, {0, 0, 1}, {0, 1, 0}, {0, 1, 1}}, {{1, 0, 0}, {1, 0, 1}, {1, 1, 0}, {1, 1, 1}},
    {{1, 0, 0}, {1, 0, 1}, {0, 0, 0}, {0, 0, 1}}, {{0, 1, 0}, {0, 1, 1}, {1, 1, 0}, {1, 1, 1}},
    {{1, 0, 0}, {0, 0, 0}, {1, 1, 0}, {0, 1, 0}}, {{0, 0, 1}, {1, 0, 1}, {0, 1, 1}, {1, 1, 1}}};
// For a lattice point that is corner `s` (sz<<2|sy<<1|sx, 1 = +1/2 side) of a voxel with exposed face `d`:
// 27-bit mask over neighbour offsets (dz+1)*9+(dy+1)*3+(dx+1) reached through the quad's triangle edges
// c0c1, c0c2, c1c2, c2c3, c0c3 (layers.py:441-443,469-472); 0 if the quad does not touch that corner.
__constant__ uint32_t kLatMask[8][6] = {
    {0x0034000u, 0x0000000u, 0x0c04000u, 0x0000000u, 0x2400000u, 0x0000000u},
    {0x0009000u, 0x0000000u, 0x0201000u, 0x0000000u, 0x0000000u, 0x2410000u},
    {0x0004c00u, 0x0000000u, 0x0000000u, 0x0c04000u, 0x0480000u, 0x0000000u},
    {0x0001200u, 0x0000000u, 0x0000000u, 0x0201000u, 0x0000000u, 0x0480400u},
    {0x0000000u, 0x0034000u, 0x0004030u, 0x0000000u, 0x0010090u, 0x0000000u},
    {0x0000000u, 0x0009000u, 0x0001008u, 0x0000000u, 0x0000000u, 0x0000090u},
    {0x0000000u, 0x0004c00u, 0x0000000u, 0x0004030u, 0x0000412u, 0x0000000u},
    {0x0000000u, 0x0001200u, 0x0000000u, 0x0001008u, 0x0000000u, 0x0000012u}};
// The same rule for the watertight topology (opt-in): quad on the side of the empty neighbour, corners cyclic from the
// quad's lowest lattice corner with outward winding -- corner_id<kWatertight> below, oracle/cubify_watertight.py.
// The triangles (c0,c1,c2),(c0,c2,c3) have the same five edges, so only the corner positions change the mask.
__constant__ uint32_t kLatMaskWT[8][6] = {
    {0x0034000u, 0x0000000u, 0x0000000u, 0x0c04000u, 0x2410000u, 0x0000000u},
    {0x0011000u, 0x0000000u, 0x0000000u, 0x0401000u, 0x0000000u, 0x2410000u},
    {0x0004400u, 0x0000000u, 0x0c04000u, 0x0000000u, 0x0400400u, 0x0000000u},
    {0x0001600u, 0x0000000u, 0x0401000u, 0x0000000u, 0x0000000u, 0x0400400u},
    {0x0000000u, 0x0034000u, 0x0000000u, 0x0004010u, 0x0010010u, 0x0000000u},
    {0x0000000u, 0x0011000u, 0x0000000u, 0x0001018u, 0x0000000u, 0x0010010u},
    {0x0000000u, 0x0004400u, 0x0004010u, 0x0000000u, 0x0000412u, 0x0000000u},
    {0x0000000u, 0x0001600u, 0x0001018u, 0x0000000u, 0x0000000u, 0x0000412u}};

// Quad placement, a compile-time choice of the two kernels that depend on it (k_lattice_count, k_emit_faces); every other
// kernel works from the face flags and lattice masks and is shared.
enum Topology { kReference = 0, kWatertight = 1 };

template <int TOPO>
__device__ __forceinline__ uint32_t lat_mask(int s, int k) {
    if constexpr (TOPO == kWatertight) return kLatMaskWT[s][k];
    else return kLatMask[s][k];
}

struct Dims {
    int B, Z, Y, X;
    int LZ, LY, LX;
    int nvox;   // Z*Y*X
    int nlat;   // LZ*LY*LX
    int nchF;   // voxel chunks per mesh
    int nchL;   // lattice chunks per mesh
};

static Dims make_dims(int B, int Z, int Y, int X) {
    Dims d;
    d.B = B; d.Z = Z; d.Y = Y; d.X = X;
    d.LZ = Z + 1; d.LY = Y + 1; d.LX = X + 1;
    d.nvox = Z * Y * X;
    d.nlat = d.LZ * d.LY * d.LX;
    d.nchF = (d.nvox + CH - 1) / CH;
    d.nchL = (d.nlat + CH - 1) / CH;
    return d;
}

struct Workspace {
    uint8_t* ff;      // [B*nvox] 6 face-flag bits per voxel
    int32_t* rank;    // [B*nlat] vertex id per used lattice point
    uint32_t* lmask;  // [B*nlat] 27-bit neighbour mask per lattice point (0 <=> not a vertex), written by the count pass
    int32_t* segBase; // [3][B+1] first face-quad / vertex / directed edge of every mesh (+ totals): the chunk counters above
                      // are scanned per mesh (local offsets), the per-mesh bases are added by the emit kernels
    int32_t* faceOff; // [B*6*nchF + 1]
    int32_t* vertOff; // [B*nchL + 1]
    int32_t* edgeOff; // [B*nchL + 1]
};

static size_t align16(size_t x) { return (x + 15) & ~size_t(15); }

static size_t carve(const Dims& d, void* base, Workspace* ws) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off += align16(bytes);
        return base ? (void*)((char*)base + o) : (void*)nullptr;
    };
    void* p0 = take((size_t)d.B * d.nvox);
    void* p1 = take((size_t)d.B * d.nlat * 4);
    void* p2 = take(((size_t)d.B * 6 * d.nchF + 1) * 4);
    void* p3 = take(((size_t)d.B * d.nchL + 1) * 4);
    void* p4 = take(((size_t)d.B * d.nchL + 1) * 4);
    void* p5 = take((size_t)d.B * d.nlat * 4);
    void* p6 = take((size_t)3 * (d.B + 1) * 4);
    if (ws) {
        ws->segBase = (int32_t*)p6;
        ws->ff = (uint8_t*)p0; ws->rank = (int32_t*)p1; ws->faceOff = (int32_t*)p2;
        ws->vertOff = (int32_t*)p3; ws->edgeOff = (int32_t*)p4; ws->lmask = (uint32_t*)p5;
    }
    return off;
}

// ---------------------------------------------------------------------------------------------------------
// pass 1a: threshold + exposed-face flags + per-(mesh, dir, chunk) face counts
// ---------------------------------------------------------------------------------------------------------
// occupancy test: probs > th (strict, fp32 -- layers.py:405), or sigmoid(logit) > th when the grid holds the voxel head's
// logits (SURVEY 8 f-1: the sigmoid of VoxelBranch folded into Cubify; same formula as voxel.cu / torch's CUDA sigmoid)
template <bool LOGITS>
__device__ __forceinline__ bool occupied(float v, float th) {
    return (LOGITS ? 1.0f / (1.0f + expf(-v)) : v) > th;
}

template <bool LOGITS>
__global__ void __launch_bounds__(CH) k_faceflags(const float* __restrict__ probs, float th, Dims d, Workspace ws) {
    const int b = blockIdx.y, chunk = blockIdx.x;
    const int v = chunk * CH + threadIdx.x;
    unsigned f = 0;
    if (v < d.nvox) {
        const float* p = probs + (size_t)b * d.nvox;
        if (occupied<LOGITS>(__ldg(p + v), th)) {
            const int x = v % d.X, y = (v / d.X) % d.Y, z = v / (d.X * d.Y);
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                const int nz = z + kNbr[k][0], ny = y + kNbr[k][1], nx = x + kNbr[k][2];
                bool occ = false;                      // zero padding (layers.py:411)
                if (nz >= 0 && nz < d.Z && ny >= 0 && ny < d.Y && nx >= 0 && nx < d.X)
                    occ = occupied<LOGITS>(__ldg(p + ((size_t)nz * d.Y + ny) * d.X + nx), th);
                if (!occ) f |= 1u << k;
            }
        }
        ws.ff[(size_t)b * d.nvox + v] = (uint8_t)f;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        int c = __syncthreads_count((f >> k) & 1u);
        if (threadIdx.x == 0) ws.faceOff[((size_t)b * 6 + k) * d.nchF + chunk] = c;
    }
}

// neighbour mask (27 bits) of lattice point (lz,ly,lx) of mesh b; 0 <=> not a vertex.  tab[s][f] = OR of kLatMask[s][k] over
// the set bits k of the 6-bit face-flag byte f (built once per block in shared memory): one lookup per adjacent voxel
// instead of six predicated ORs.
__device__ __forceinline__ uint32_t lattice_mask(const uint8_t* __restrict__ ffb, const uint32_t (*tab)[64], const Dims& d, int lz,
                                                 int ly, int lx) {
    uint32_t m = 0;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int vz = lz - 1 + ((a >> 2) & 1), vy = ly - 1 + ((a >> 1) & 1), vx = lx - 1 + (a & 1);
        if (vz < 0 || vz >= d.Z || vy < 0 || vy >= d.Y || vx < 0 || vx >= d.X) continue;
        const unsigned f = ffb[((size_t)vz * d.Y + vy) * d.X + vx];
        m |= tab[7 - a][f];        // corner position relative to that voxel: (1-az, 1-ay, 1-ax)
    }
    return m;
}

// pass 1b: per-(mesh, lattice chunk) vertex and directed-edge counts; the masks are kept for the emit pass
template <int TOPO>
__global__ void __launch_bounds__(CH) k_lattice_count(Dims d, Workspace ws) {
    __shared__ int scratch[33];
    __shared__ uint32_t tab[8][64];
    {
        const int s8 = threadIdx.x >> 6, f = threadIdx.x & 63;      // CH == 512 == 8 * 64 table entries
        uint32_t m = 0;
#pragma unroll
        for (int k = 0; k < 6; ++k)
            if ((f >> k) & 1) m |= lat_mask<TOPO>(s8, k);
        tab[s8][f] = m;
    }
    __syncthreads();
    const int b = blockIdx.y, chunk = blockIdx.x;
    const int l = chunk * CH + threadIdx.x;
    uint32_t m = 0;
    if (l < d.nlat) {
        const int lx = l % d.LX, ly = (l / d.LX) % d.LY, lz = l / (d.LX * d.LY);
        m = lattice_mask(ws.ff + (size_t)b * d.nvox, tab, d, lz, ly, lx);
        ws.lmask[(size_t)b * d.nlat + l] = m;
    }
    const int nv = __syncthreads_count(m != 0);
    const int ne = block_sum<int>(__popc(m), scratch);
    if (threadIdx.x == 0) {
        ws.vertOff[(size_t)b * d.nchL + chunk] = nv;
        ws.edgeOff[(size_t)b * d.nchL + chunk] = ne;
    }
}

// pass 1c: exclusive scans of the three chunk-count arrays, two levels: one block per (mesh, array) scans that mesh's
// segment in place (coalesced through shared memory) and records its total; one block then scans the B totals per array
// and fills meta.  (A single-block scan of the 83k face counters of 64 x 48^3 took 65 us.)
// meta layout (int64): [0]=SV [1]=SF [2]=E [3]=unused, then v_count[B], f_count[B], v_offset[B], f_offset[B]
constexpr int SEG_THREADS = 256, SEG_PER = 8;
__global__ void __launch_bounds__(SEG_THREADS) k_scan_seg(Dims d, Workspace ws) {
    __shared__ int buf[SEG_THREADS * SEG_PER];
    __shared__ int scratch[33];
    const int b = blockIdx.x, which = blockIdx.y;
    const int len = which == 0 ? 6 * d.nchF : d.nchL;
    int32_t* arr = (which == 0 ? ws.faceOff : (which == 1 ? ws.vertOff : ws.edgeOff)) + (size_t)b * len;
    int carry = 0;
    for (int base = 0; base < len; base += SEG_THREADS * SEG_PER) {
#pragma unroll
        for (int u = 0; u < SEG_PER; ++u) {
            const int i = base + u * SEG_THREADS + threadIdx.x;
            buf[u * SEG_THREADS + threadIdx.x] = i < len ? arr[i] : 0;
        }
        __syncthreads();
        int vals[SEG_PER], sum = 0;
#pragma unroll
        for (int u = 0; u < SEG_PER; ++u) { vals[u] = buf[threadIdx.x * SEG_PER + u]; sum += vals[u]; }
        int total;
        int run = carry + block_exclusive_scan(sum, scratch, &total);
#pragma unroll
        for (int u = 0; u < SEG_PER; ++u) { buf[threadIdx.x * SEG_PER + u] = run; run += vals[u]; }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < SEG_PER; ++u) {
            const int i = base + u * SEG_THREADS + threadIdx.x;
            if (i < len) arr[i] = buf[u * SEG_THREADS + threadIdx.x];
        }
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) ws.segBase[which * (d.B + 1) + b] = carry;      // the segment total; k_scan_top turns it into a base
}

__global__ void __launch_bounds__(1024) k_scan_top(Dims d, Workspace ws, long long* __restrict__ meta) {
    __shared__ int scratch[33];
    const int which = blockIdx.x;
    int32_t* seg = ws.segBase + which * (d.B + 1);
    int carry = 0;
    for (int base = 0; base < d.B; base += 1024) {
        const int b = base + threadIdx.x;
        const int cnt = b < d.B ? seg[b] : 0;
        int total;
        const int ex = carry + block_exclusive_scan(cnt, scratch, &total);
        if (b < d.B) {
            seg[b] = ex;
            if (which == 0) { meta[4 + d.B + b] = 2LL * cnt; meta[4 + 3 * d.B + b] = 2LL * ex; }
            else if (which == 1) { meta[4 + b] = cnt; meta[4 + 2 * d.B + b] = ex; }
        }
        carry += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        seg[d.B] = carry;
        if (which == 0) meta[1] = 2LL * carry;
        else if (which == 1) meta[0] = carry;
        else { meta[2] = carry; meta[3] = 0; }
    }
}

// ---------------------------------------------------------------------------------------------------------
// pass 2a: vertices, lattice ranks, CSR row pointers
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CH) k_emit_verts(Dims d, Workspace ws, float* __restrict__ verts,
                                                   int32_t* __restrict__ rowptr, int32_t* __restrict__ vert_mesh,
                                                   uint32_t* __restrict__ vmask, int32_t* __restrict__ vlat) {
    __shared__ int scratch[33];
    const int b = blockIdx.y, chunk = blockIdx.x;
    const int l = chunk * CH + threadIdx.x;
    uint32_t m = 0;
    int lx = 0, ly = 0, lz = 0;
    if (l < d.nlat) {
        m = ws.lmask[(size_t)b * d.nlat + l];          // computed once by k_lattice_count
        if (m) { lx = l % d.LX; ly = (l / d.LX) % d.LY; lz = l / (d.LX * d.LY); }
    }
    int tot;
    const int exv = block_exclusive_scan(m != 0 ? 1 : 0, scratch, &tot);
    __syncthreads();
    const int exe = block_exclusive_scan(__popc(m), scratch, &tot);
    if (m) {
        const int vid = ws.segBase[(d.B + 1) + b] + ws.vertOff[(size_t)b * d.nchL + chunk] + exv;
        ws.rank[(size_t)b * d.nlat + l] = vid;
        // (z,y,x) half-integers rotated 90 deg about axis 0: (z, x, -y)  (layers.py:465-467, exact in fp32)
        verts[3 * (size_t)vid + 0] = (float)lz - 0.5f;
        verts[3 * (size_t)vid + 1] = (float)lx - 0.5f;
        verts[3 * (size_t)vid + 2] = -((float)ly - 0.5f);
        rowptr[vid] = ws.segBase[2 * (d.B + 1) + b] + ws.edgeOff[(size_t)b * d.nchL + chunk] + exe;
        vert_mesh[vid] = b;
        vmask[vid] = m;
        vlat[vid] = b * d.nlat + l;
    }
    if (b == d.B - 1 && chunk == d.nchL - 1 && threadIdx.x == 0) {
        const int SV = ws.segBase[(d.B + 1) + d.B];
        rowptr[SV] = ws.segBase[2 * (d.B + 1) + d.B];
    }
}

// pass 2b: adjacency.  One thread per vertex enumerates its neighbours in ascending lattice order (== ascending
// vertex id); the block's edges form one contiguous output range, so they are staged in shared memory and streamed out
// with fully coalesced int64 / int32 stores (the 16 B/edge COO + 4 B/edge CSR streams are the bulk of Cubify's traffic).
constexpr int ADJ_BLOCK = 256;
constexpr int ADJ_CAP = ADJ_BLOCK * 18;   // a lattice vertex has at most 18 neighbours (6 axis + 12 face-diagonal)

__global__ void __launch_bounds__(ADJ_BLOCK) k_emit_adj(Dims d, Workspace ws, int SV, const int32_t* __restrict__ rowptr,
                                                        const uint32_t* __restrict__ vmask, const int32_t* __restrict__ vlat,
                                                        long long* __restrict__ adj_row, long long* __restrict__ adj_col,
                                                        int32_t* __restrict__ col32) {
    __shared__ int32_t s_col[ADJ_CAP];
    __shared__ unsigned char s_row[ADJ_CAP];
    const int v0 = blockIdx.x * ADJ_BLOCK;
    const int vid = v0 + threadIdx.x;
    const int e_begin = rowptr[v0];
    const int e_end = rowptr[min(v0 + ADJ_BLOCK, SV)];
    if (vid < SV) {
        uint32_t m = vmask[vid];
        const int lat = vlat[vid];
        int e = rowptr[vid] - e_begin;
        const int sY = d.LX, sZ = d.LX * d.LY;
        while (m) {
            const int bit = __ffs(m) - 1;
            m &= m - 1;
            const int dz = bit / 9 - 1, dy = (bit / 3) % 3 - 1, dx = bit % 3 - 1;
            s_col[e] = ws.rank[lat + dz * sZ + dy * sY + dx];
            s_row[e] = (unsigned char)threadIdx.x;
            ++e;
        }
    }
    __syncthreads();
    const int n = e_end - e_begin;
    for (int e = threadIdx.x; e < n; e += ADJ_BLOCK) {
        const int c = s_col[e];
        adj_row[(size_t)e_begin + e] = v0 + s_row[e];
        adj_col[(size_t)e_begin + e] = c;
        col32[(size_t)e_begin + e] = c;
    }
}

// pass 2c: faces in (b, dir, z, y, x) order, two triangles (c0,c1,c2),(c0,c2,c3) per quad, per-mesh local ids.
// A quad is 6 int64 = 48 contiguous bytes and consecutive flagged lanes write consecutive quads, so every thread stores its
// quad straight from registers as three 16-byte vectors (a warp covers up to 1.5 KB of contiguous output).  The kernel was
// instruction bound (1 080 warp instructions per 32 voxels): now the 8 corner ranks of a voxel are loaded once (not 4 per
// quad with their own index arithmetic), the quad corners are compile-time picks among them, and the per-warp output offsets
// of all six directions come from one shared-memory prefix pass instead of a serial sum per (thread, direction).
template <int TOPO>
__device__ __forceinline__ constexpr int corner_id(int k, int j) {
    // kCorner[k][j] as cz*4 + cy*2 + cx (same table as the __constant__ one above, usable in constant expressions)
    constexpr int T[6][4] = {{0, 1, 2, 3}, {4, 5, 6, 7}, {4, 5, 0, 1}, {2, 3, 6, 7}, {4, 0, 6, 2}, {1, 5, 3, 7}};
    // watertight: d0 000 001 011 010, d1 100 110 111 101, d2 010 011 111 110, d3 000 100 101 001, d4 000 010 110 100,
    // d5 001 101 111 011 (z,y,x offsets; cyclic, (c1-c0) x (c2-c0) toward the empty neighbour)
    constexpr int W[6][4] = {{0, 1, 3, 2}, {4, 6, 7, 5}, {2, 3, 7, 6}, {0, 4, 5, 1}, {0, 2, 6, 4}, {1, 5, 7, 3}};
    return TOPO == kWatertight ? W[k][j] : T[k][j];
}

template <int TOPO>
__global__ void __launch_bounds__(CH) k_emit_faces(Dims d, Workspace ws, const long long* __restrict__ meta,
                                                   long long* __restrict__ faces) {
    constexpr int NW = CH / 32;
    __shared__ int wtot[6][NW];
    const int b = blockIdx.y, chunk = blockIdx.x;
    const int v = chunk * CH + threadIdx.x;
    const unsigned f = (v < d.nvox) ? ws.ff[(size_t)b * d.nvox + v] : 0u;
    int pre[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const unsigned bal = __ballot_sync(0xffffffffu, (f >> k) & 1u);
        pre[k] = __popc(bal & ((1u << lane_id()) - 1u));
        if (lane_id() == 0) wtot[k][warp_id()] = __popc(bal);
    }
    __syncthreads();
    if (threadIdx.x < 6 * 32) {                    // warp k: exclusive prefix of direction k's per-warp totals
        const int k = warp_id();
        const int mine = lane_id() < NW ? wtot[k][lane_id()] : 0;
        const int inc = warp_inclusive_scan(mine);
        __syncwarp();
        if (lane_id() < NW) wtot[k][lane_id()] = inc - mine;
    }
    __syncthreads();
    if (f == 0u) return;
    const int x = v % d.X, y = (v / d.X) % d.Y, z = v / (d.X * d.Y);
    const int voff = (int)meta[4 + 2 * d.B + b];
    const int32_t* rk = ws.rank + (size_t)b * d.nlat + ((size_t)z * d.LY + y) * d.LX + x;
    const int sY = d.LX, sZ = d.LX * d.LY;
    long long r[8];                                // local vertex ids of the voxel's 8 lattice corners (unused corners hold junk)
#pragma unroll
    for (int a = 0; a < 8; ++a) r[a] = (long long)(rk[((a >> 2) & 1) * sZ + ((a >> 1) & 1) * sY + (a & 1)] - voff);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        if (!((f >> k) & 1u)) continue;
        const long long q = ws.segBase[b] + ws.faceOff[((size_t)b * 6 + k) * d.nchF + chunk] + wtot[k][warp_id()] + pre[k];
        const long long c0 = r[corner_id<TOPO>(k, 0)], c1 = r[corner_id<TOPO>(k, 1)], c2 = r[corner_id<TOPO>(k, 2)],
                        c3 = r[corner_id<TOPO>(k, 3)];
        longlong2* o = reinterpret_cast<longlong2*>(faces + q * 6);          // 48-byte quads: 16-byte aligned
        o[0] = make_longlong2(c0, c1);
        o[1] = make_longlong2(c2, c0);
        o[2] = make_longlong2(c2, c3);
    }
}

}  // namespace cubify
}  // namespace mrb

using namespace mrb;
using namespace mrb::cubify;

extern "C" long long mrb_cubify_workspace_bytes(int B, int Z, int Y, int X) {
    if (B <= 0 || Z <= 0 || Y <= 0 || X <= 0) return -1;
    Dims d = make_dims(B, Z, Y, X);
    return (long long)carve(d, nullptr, nullptr);
}

extern "C" int mrb_cubify_count_topo(const float* probs, int B, int Z, int Y, int X, float threshold, int from_logits,
                                     int topology, void* workspace, long long* meta, void* stream_) {
    MRB_REQUIRE(topology == kReference || topology == kWatertight, "cubify_count: bad topology %d", topology);
    MRB_REQUIRE(probs && workspace && meta, "cubify_count: null pointer");
    MRB_REQUIRE(B > 0 && Z > 0 && Y > 0 && X > 0, "cubify_count: bad grid %dx%dx%dx%d", B, Z, Y, X);
    MRB_REQUIRE((long long)B * (Z + 1) * (Y + 1) * (X + 1) < (1LL << 31), "cubify_count: lattice too large for int32");
    MRB_REQUIRE(B <= 65535, "cubify_count: batch too large");
    cudaStream_t stream = (cudaStream_t)stream_;
    Dims d = make_dims(B, Z, Y, X);
    Workspace ws;
    carve(d, workspace, &ws);
    if (from_logits) k_faceflags<true><<<dim3(d.nchF, B), CH, 0, stream>>>(probs, threshold, d, ws);
    else k_faceflags<false><<<dim3(d.nchF, B), CH, 0, stream>>>(probs, threshold, d, ws);
    if (topology == kWatertight) k_lattice_count<kWatertight><<<dim3(d.nchL, B), CH, 0, stream>>>(d, ws);
    else k_lattice_count<kReference><<<dim3(d.nchL, B), CH, 0, stream>>>(d, ws);
    k_scan_seg<<<dim3(B, 3), SEG_THREADS, 0, stream>>>(d, ws);
    k_scan_top<<<3, 1024, 0, stream>>>(d, ws, meta);
    return check_launch("cubify_count");
}

extern "C" int mrb_cubify_count(const float* probs, int B, int Z, int Y, int X, float threshold, int from_logits,
                                void* workspace, long long* meta, void* stream_) {
    return mrb_cubify_count_topo(probs, B, Z, Y, X, threshold, from_logits, kReference, workspace, meta, stream_);
}

extern "C" int mrb_cubify_emit_topo(int B, int Z, int Y, int X, void* workspace, const long long* meta, long long SV,
                                    long long SF, long long E, float* verts, long long* faces, long long* adj,
                                    int32_t* rowptr, int32_t* col32, int32_t* vert_mesh, void* vert_aux, int topology,
                                    void* stream_) {
    MRB_REQUIRE(topology == kReference || topology == kWatertight, "cubify_emit: bad topology %d", topology);
    MRB_REQUIRE(workspace && meta && verts && faces && adj && rowptr && col32 && vert_mesh && vert_aux,
                "cubify_emit: null pointer");
    MRB_REQUIRE(SV > 0 && SF > 0 && E > 0, "cubify_emit: empty grid");
    cudaStream_t stream = (cudaStream_t)stream_;
    Dims d = make_dims(B, Z, Y, X);
    Workspace ws;
    carve(d, workspace, &ws);
    uint32_t* vmask = (uint32_t*)vert_aux;
    int32_t* vlat = (int32_t*)vert_aux + SV;
    k_emit_verts<<<dim3(d.nchL, B), CH, 0, stream>>>(d, ws, verts, rowptr, vert_mesh, vmask, vlat);
    k_emit_adj<<<ceil_div(SV, ADJ_BLOCK), ADJ_BLOCK, 0, stream>>>(d, ws, (int)SV, rowptr, vmask, vlat, adj, adj + E, col32);
    if (topology == kWatertight) k_emit_faces<kWatertight><<<dim3(d.nchF, B), CH, 0, stream>>>(d, ws, meta, faces);
    else k_emit_faces<kReference><<<dim3(d.nchF, B), CH, 0, stream>>>(d, ws, meta, faces);
    return check_launch("cubify_emit");
}

extern "C" int mrb_cubify_emit(int B, int Z, int Y, int X, void* workspace, const long long* meta, long long SV,
                               long long SF, long long E, float* verts, long long* faces, long long* adj,
                               int32_t* rowptr, int32_t* col32, int32_t* vert_mesh, void* vert_aux, void* stream_) {
    return mrb_cubify_emit_topo(B, Z, Y, X, workspace, meta, SV, SF, E, verts, faces, adj, rowptr, col32, vert_mesh,
                                vert_aux, kReference, stream_);
}
