// extract.cu -- zero-crossing cloud + normal extraction from the TSDF volume, sm_100a.
// Replaces FullScan6 / ExtractNormals of the reference (kfusion/src/cuda/tsdf_volume.cu:486-831).
//
// The reference appends points through one global atomicAdd cursor, so its output ORDER is nondeterministic (and the
// warp nodes are picked from that order, warp_field.cpp:49-51).  Here extraction is deterministic: a counting pass,
// an exclusive scan over block counts and an emit pass produce the points in ascending (z, y, x) voxel order, +x,+y,+z
// edge within a voxel -- the same order the CPU oracle uses, so the result is comparable element by element.
//
// Work decomposition: the volume is one contiguous array cut into blocks of EX_THREADS quads (1024 voxels when VX = 4), a
// quad = VX consecutive voxels = one 16-byte load.  A quad whose voxels are all unobserved (W == 0) or free space (F == 1)
// needs nothing else -- on real scenes that is >90 % of them; only surface quads fetch the +x / +y / +z neighbours (L1/L2
// hits).  Kernels: see the comment above extract_count_kernel.
#include "df_common.cuh"
#include <climits>

using namespace dfb;

namespace {

constexpr int EX_THREADS = 256;

struct ExtractParams {
    const uint32_t *data;
    int Dx, Dy, Dz;
    float3 vs;
    Aff pose;
    size_t nvox;
    int nblocks;
    const unsigned char *activity;   // optional (dfusion.h, DF_ACTIVITY_VOXELS): blocks whose stretch of the volume is inactive are skipped
};

__device__ __forceinline__ float vox_f(uint32_t v) { return half_bits_to_float((unsigned short)(v & 0xffffu)); }
__device__ __forceinline__ bool sign_change(float F, float Fn) { return (F > 0 && Fn < 0) || (F < 0 && Fn > 0); }

// centre of voxel (x, y, z) in volume coordinates
__device__ __forceinline__ float3 voxel_centre(const ExtractParams &p, int x, int y, int z)
{
    return make_float3(((float)x + 0.5f) * p.vs.x, ((float)y + 0.5f) * p.vs.y, ((float)z + 0.5f) * p.vs.z);
}

// The point on the edge from voxel centre V (value F) to its +axis neighbour (value Fn), interpolated as tsdf_volume.cu:573-627 does,
// then posed.  The one copy of the formula: the cloud's points and the mesh's vertices both come from here, so a mesh vertex on an edge
// the cloud also emits is bit-identical to the cloud's point.
__device__ __forceinline__ float3 edge_point(const ExtractParams &p, float3 V, float F, float Fn, int axis)
{
    const float d_inv = 1.f / (fabsf(F) + fabsf(Fn));
    if (axis == 0) V.x = (V.x * fabsf(Fn) + (V.x + p.vs.x) * fabsf(F)) * d_inv;
    else if (axis == 1) V.y = (V.y * fabsf(Fn) + (V.y + p.vs.y) * fabsf(F)) * d_inv;
    else V.z = (V.z * fabsf(Fn) + (V.z + p.vs.z) * fabsf(F)) * d_inv;
    return aff_mul(p.pose, V);
}

// Calls emit(point) for every zero crossing owned by this thread, in (voxel, axis) order.  tsdf_volume.cu:548-633.
// the thread's own VX voxels (one 16-byte load when VX = 4); zeros past the end of the volume
template <int VX>
__device__ __forceinline__ void load_quad(const ExtractParams &p, size_t v0, uint32_t (&own)[VX])
{
#pragma unroll
    for (int j = 0; j < VX; ++j) own[j] = 0u;
    if (v0 >= p.nvox) return;
    if (VX == 4) {
        const uint4 q = __ldg(reinterpret_cast<const uint4 *>(p.data + v0));
        own[0] = q.x; own[1 % VX] = q.y; own[2 % VX] = q.z; own[3 % VX] = q.w;
    } else {
        own[0] = __ldg(p.data + v0);
    }
}

template <int VX, typename Emit>
__device__ __forceinline__ void thread_crossings(const ExtractParams &p, size_t v0, const uint32_t (&own)[VX], Emit emit)
{
    bool any = false;
#pragma unroll
    for (int j = 0; j < VX; ++j) any |= vox_active(own[j]);
    if (!any) return;

    const size_t slice = (size_t)p.Dx * p.Dy;
    const int z = (int)(v0 / slice);
    if (z >= p.Dz - 1) return;                               // loop bound z < dims.z - 1, tsdf_volume.cu:553
    const int rem = (int)(v0 - (size_t)z * slice);
    const int y = rem / p.Dx;
    const int x0 = rem - y * p.Dx;

#pragma unroll
    for (int j = 0; j < VX; ++j) {
        if (!vox_active(own[j])) continue;
        const int x = x0 + j;
        const float F = vox_f(own[j]);
        const float3 V = voxel_centre(p, x, y, z);
        if (x + 1 < p.Dx) {
            const uint32_t nv = (j + 1 < VX) ? own[(j + 1) % VX] : __ldg(p.data + v0 + VX);
            if (vox_active(nv)) {
                const float Fn = vox_f(nv);
                if (sign_change(F, Fn)) emit(edge_point(p, V, F, Fn, 0));
            }
        }
        if (y + 1 < p.Dy) {
            const uint32_t nv = __ldg(p.data + v0 + j + p.Dx);
            if (vox_active(nv)) {
                const float Fn = vox_f(nv);
                if (sign_change(F, Fn)) emit(edge_point(p, V, F, Fn, 1));
            }
        }
        {
            const uint32_t nv = __ldg(p.data + v0 + j + slice);
            if (vox_active(nv)) {
                const float Fn = vox_f(nv);
                if (sign_change(F, Fn)) emit(edge_point(p, V, F, Fn, 2));
            }
        }
    }
}

// Count / emit.  A block = EX_THREADS * EX_QPT quads (4096 voxels when VX = 4), a thread owns quads tid, tid + 256, ...: all of
// its 16-byte loads are issued before any of them is used, and each load instruction of a warp is one contiguous 512-byte
// request.  History (profiles/): one quad per thread meant 131,072 CTAs for 512^3 -- the emit pass, whose CTAs mostly return at
// once, still took 0.17 ms: block scheduling, not memory, was the limit; one WARP per block (8 quads per lane, shuffle scans)
// removed the scheduling cost but serialised the dependent neighbour fetches of the surface quads and was 4x slower.
// With an activity map the quads of inactive stretches are not loaded at all.
constexpr int EX_QPT = 4;

__device__ __forceinline__ int block_exclusive_scan(int v, int *total)
{
    __shared__ int warp_sums[EX_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = lane < EX_THREADS / 32 ? warp_sums[lane] : 0;
#pragma unroll
        for (int o = 1; o < EX_THREADS / 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += n;
        }
        if (lane < EX_THREADS / 32) warp_sums[lane] = w;
    }
    __syncthreads();
    const int base = warp ? warp_sums[warp - 1] : 0;
    if (total) *total = warp_sums[EX_THREADS / 32 - 1];
    __syncthreads();
    return base + incl - v;
}

template <int VX>
__device__ __forceinline__ int quad_count(const ExtractParams &p, size_t v0, const uint32_t (&own)[VX])
{
    int n = 0;
    thread_crossings<VX>(p, v0, own, [&](const float3) { ++n; });
    return n;
}

template <int VX>
__device__ __forceinline__ void load_block_quads(const ExtractParams &p, size_t q0, uint32_t (&own)[EX_QPT][VX])
{
#pragma unroll
    for (int i = 0; i < EX_QPT; ++i) {
        const size_t v0 = (q0 + (size_t)(i * EX_THREADS) + threadIdx.x) * VX;
#pragma unroll
        for (int j = 0; j < VX; ++j) own[i][j] = 0u;
        if (p.activity && v0 < p.nvox && !p.activity[v0 / DF_ACTIVITY_VOXELS]) continue;    // cannot hold surface: not even loaded
        load_quad<VX>(p, v0, own[i]);
    }
}

template <int VX>
__global__ void __launch_bounds__(EX_THREADS) extract_count_kernel(const ExtractParams p, int *block_counts)
{
    DF_PDL_ENTRY();
    const size_t q0 = (size_t)blockIdx.x * EX_THREADS * EX_QPT;
    uint32_t own[EX_QPT][VX];
    load_block_quads<VX>(p, q0, own);
    int n = 0;
#pragma unroll
    for (int i = 0; i < EX_QPT; ++i) n += quad_count<VX>(p, (q0 + (size_t)(i * EX_THREADS) + threadIdx.x) * VX, own[i]);
    const int any = __syncthreads_or(n);
    if (!any) { if (threadIdx.x == 0) block_counts[blockIdx.x] = 0; return; }
    int total;
    block_exclusive_scan(n, &total);
    if (threadIdx.x == 0) block_counts[blockIdx.x] = total;
}

// two-level exclusive scan over the per-block counts: 1024 counts per "super" block (warp-shuffle scan), then one block
// over the <= 1024 super totals.  (A single-block serial-chunk scan of the 131,072 counts of a 512^3 volume took 0.26 ms.)
__global__ void __launch_bounds__(1024) extract_scan_local_kernel(const int *counts, int *offsets, int n, int *super_tot)
{
    DF_PDL_ENTRY();
    __shared__ int wsum[32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int i = blockIdx.x * 1024 + t;
    const int c = i < n ? counts[i] : 0;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += v; }
        wsum[lane] = w;
    }
    __syncthreads();
    const int base = warp ? wsum[warp - 1] : 0;
    if (i < n) offsets[i] = base + incl - c;
    if (t == 1023) super_tot[blockIdx.x] = wsum[31];
}

__global__ void __launch_bounds__(1024) extract_scan_super_kernel(const int *super_tot, int nsuper, int *super_off, int capacity, int *count_out)
{
    DF_PDL_ENTRY();
    __shared__ int wsum[32];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int c = t < nsuper ? super_tot[t] : 0;
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += v; }
        wsum[lane] = w;
    }
    __syncthreads();
    const int base = warp ? wsum[warp - 1] : 0;
    if (t < nsuper) super_off[t] = base + incl - c;
    if (t == 1023) *count_out = min(wsum[31], capacity);
}

template <int VX>
__global__ void __launch_bounds__(EX_THREADS) extract_emit_kernel(const ExtractParams p, const int *block_counts, const int *offsets,
                                                                  const int *super_off, float4 *out, int capacity)
{
    DF_PDL_ENTRY();
    if (block_counts[blockIdx.x] == 0) return;
    const size_t q0 = (size_t)blockIdx.x * EX_THREADS * EX_QPT;
    uint32_t own[EX_QPT][VX];
    load_block_quads<VX>(p, q0, own);
    int run = super_off[blockIdx.x >> 10] + offsets[blockIdx.x];
#pragma unroll
    for (int i = 0; i < EX_QPT; ++i) {                                // points leave in quad order i * EX_THREADS + tid
        const size_t v0 = (q0 + (size_t)(i * EX_THREADS) + threadIdx.x) * VX;
        const int c = quad_count<VX>(p, v0, own[i]);
        int total;
        int k = run + block_exclusive_scan(c, &total);
        if (c)
            thread_crossings<VX>(p, v0, own[i], [&](const float3 q) {
                if (k < capacity) out[k] = make_float4(q.x, q.y, q.z, 0.f);
                ++k;
            });
        run += total;
    }
}

ExtractParams make_params(const df_volume &vol, const df_aff3f &pose, int vx)
{
    ExtractParams p;
    p.data = vol.data;
    p.Dx = vol.dims[0]; p.Dy = vol.dims[1]; p.Dz = vol.dims[2];
    p.vs = make_float3(vol.voxel_size[0], vol.voxel_size[1], vol.voxel_size[2]);
    p.pose = make_aff(pose);
    p.nvox = (size_t)vol.dims[0] * vol.dims[1] * vol.dims[2];
    p.nblocks = (int)((p.nvox + (size_t)EX_THREADS * EX_QPT * vx - 1) / ((size_t)EX_THREADS * EX_QPT * vx));
    p.activity = nullptr;
    return p;
}

int pick_vx(const df_volume &vol) { return (vol.dims[0] % 4 == 0 && ((uintptr_t)vol.data & 15u) == 0) ? 4 : 1; }

}  // namespace

extern "C" size_t df_extract_workspace_bytes(df_volume vol)
{
    const size_t nvox = (size_t)vol.dims[0] * vol.dims[1] * vol.dims[2];
    const size_t nblocks = (nvox + EX_THREADS - 1) / EX_THREADS;          // upper bound (VX = 1)
    return (2 * nblocks + 2048 + 64) * sizeof(int);
}

extern "C" int df_extract_cloud(df_volume vol, df_aff3f pose, float *out_points, int capacity, int *count, void *workspace, void *stream)
{
    return df_extract_cloud_tracked(vol, pose, out_points, capacity, count, workspace, nullptr, stream);
}

extern "C" int df_extract_cloud_tracked(df_volume vol, df_aff3f pose, float *out_points, int capacity, int *count, void *workspace,
                                        const unsigned char *activity, void *stream)
{
    const int vx = pick_vx(vol);
    ExtractParams p = make_params(vol, pose, vx);
    p.activity = activity;
    int *block_counts = (int *)workspace;
    int *offsets = block_counts + p.nblocks;
    cudaStream_t s = (cudaStream_t)stream;
    if (vx == 4) launch_pdl(extract_count_kernel<4>, dim3(p.nblocks), dim3(EX_THREADS), 0, s, p, block_counts);
    else launch_pdl(extract_count_kernel<1>, dim3(p.nblocks), dim3(EX_THREADS), 0, s, p, block_counts);
    DF_LAUNCH_CHECK();
    const int nsuper = (p.nblocks + 1023) / 1024;
    if (nsuper > 1024) return (int)cudaErrorInvalidValue;               // > 2^20 blocks (volume > 1024^3 voxels)
    int *super_tot = offsets + p.nblocks, *super_off = super_tot + 1024;
    launch_pdl(extract_scan_local_kernel, dim3(nsuper), dim3(1024), 0, s, block_counts, offsets, p.nblocks, super_tot);
    DF_LAUNCH_CHECK();
    launch_pdl(extract_scan_super_kernel, dim3(1), dim3(1024), 0, s, super_tot, nsuper, super_off, capacity, count);
    DF_LAUNCH_CHECK();
    if (vx == 4) launch_pdl(extract_emit_kernel<4>, dim3(p.nblocks), dim3(EX_THREADS), 0, s, p, block_counts, offsets, super_off, (float4 *)out_points, capacity);
    else launch_pdl(extract_emit_kernel<1>, dim3(p.nblocks), dim3(EX_THREADS), 0, s, p, block_counts, offsets, super_off, (float4 *)out_points, capacity);
    DF_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// Mesh extraction (marching cubes; the definition is in dfusion.h above df_extract_mesh).  Same block decomposition, quad loads,
// activity skip and scans as the cloud: a counting pass writes two sets of block counts (vertices, triangles), each is scanned, then
// one pass emits the vertices (ascending edge key) and one the triangles (ascending cell, table order).  A triangle finds its vertices
// by binary search of their keys in the just-written edge_keys, inside the range of the block that owns the edge's lower endpoint.
#define DF_MC_CONST static __device__ const
#include "mc_table.h"

namespace {

__device__ __forceinline__ size_t vox_index(const ExtractParams &p, int x, int y, int z)
{
    return (size_t)x + (size_t)p.Dx * y + (size_t)p.Dx * p.Dy * z;
}

// case of the cell with min corner (x, y, z) -- bit i + 2j + 4k set iff corner (x+i, y+j, z+k) is inside (F < 0) -- or -1 if one of its
// corners is inactive.  The caller keeps x < Dx-1, y < Dy-1, z < Dz-1.
__device__ __forceinline__ int cell_case(const ExtractParams &p, int x, int y, int z)
{
    const size_t sy = (size_t)p.Dx, sz = (size_t)p.Dx * p.Dy;
    const uint32_t *b = p.data + vox_index(p, x, y, z);
    int c = 0;
    bool active = true;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const uint32_t v = __ldg(b + (i & 1) + ((i & 2) ? sy : 0) + ((i & 4) ? sz : 0));
        active &= vox_active(v);
        c |= (int)vox_negative(v) << i;
    }
    return active ? c : -1;
}

// is one of the (up to four) cells around the edge from (x, y, z) along `axis` meshed?  Its endpoints differ in the inside test, so
// every such cell has a mixed case and is meshed as soon as all its corners are active.
__device__ __forceinline__ bool edge_has_meshed_cell(const ExtractParams &p, int x, int y, int z, int axis)
{
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int cx = x - (axis == 0 ? 0 : j), cy = y - (axis == 1 ? 0 : (axis == 0 ? j : k)), cz = z - (axis == 2 ? 0 : k);
            if (cx < 0 || cy < 0 || cz < 0 || cx >= p.Dx - 1 || cy >= p.Dy - 1 || cz >= p.Dz - 1) continue;
            if (cell_case(p, cx, cy, cz) >= 0) return true;
        }
    return false;
}

// Calls emit(edge key, vertex) for every mesh vertex owned by this thread's quad (the edges leaving its voxels along +x, +y, +z), in
// ascending key order.
template <int VX, typename Emit>
__device__ __forceinline__ void thread_mesh_vertices(const ExtractParams &p, size_t v0, const uint32_t (&own)[VX], Emit emit)
{
    bool any = false;
#pragma unroll
    for (int j = 0; j < VX; ++j) any |= vox_active(own[j]);
    if (!any) return;
    const size_t slice = (size_t)p.Dx * p.Dy;
    const int z = (int)(v0 / slice);
    const int rem = (int)(v0 - (size_t)z * slice);
    const int y = rem / p.Dx;
    const int x0 = rem - y * p.Dx;
#pragma unroll
    for (int j = 0; j < VX; ++j) {
        if (!vox_active(own[j])) continue;
        const int x = x0 + j;
        const bool inside = vox_negative(own[j]);
#pragma unroll
        for (int axis = 0; axis < 3; ++axis) {
            if (axis == 0 ? x + 1 >= p.Dx : axis == 1 ? y + 1 >= p.Dy : z + 1 >= p.Dz) continue;
            const uint32_t nv = axis == 0 ? ((j + 1 < VX) ? own[(j + 1) % VX] : __ldg(p.data + v0 + VX))
                                          : __ldg(p.data + v0 + j + (axis == 1 ? (size_t)p.Dx : slice));
            if (!vox_active(nv) || vox_negative(nv) == inside) continue;
            if (!edge_has_meshed_cell(p, x, y, z, axis)) continue;
            emit(3u * (uint32_t)(v0 + j) + (uint32_t)axis, edge_point(p, voxel_centre(p, x, y, z), vox_f(own[j]), vox_f(nv), axis));
        }
    }
}

// Calls emit(voxel index, case) for every meshed cell whose min corner is one of this thread's voxels, in ascending order.
template <int VX, typename Emit>
__device__ __forceinline__ void thread_mesh_cells(const ExtractParams &p, size_t v0, const uint32_t (&own)[VX], Emit emit)
{
    bool any = false;
#pragma unroll
    for (int j = 0; j < VX; ++j) any |= vox_active(own[j]);
    if (!any) return;
    const size_t slice = (size_t)p.Dx * p.Dy;
    const int z = (int)(v0 / slice);
    if (z >= p.Dz - 1) return;
    const int rem = (int)(v0 - (size_t)z * slice);
    const int y = rem / p.Dx;
    if (y >= p.Dy - 1) return;
    const int x0 = rem - y * p.Dx;
#pragma unroll
    for (int j = 0; j < VX; ++j) {
        if (!vox_active(own[j]) || x0 + j >= p.Dx - 1) continue;
        const int c = cell_case(p, x0 + j, y, z);
        if (c > 0 && c < 255) emit(v0 + j, c);
    }
}

template <int VX>
__device__ __forceinline__ void quad_mesh_counts(const ExtractParams &p, size_t v0, const uint32_t (&own)[VX], int &nv, int &nt)
{
    thread_mesh_vertices<VX>(p, v0, own, [&](uint32_t, float3) { ++nv; });
    thread_mesh_cells<VX>(p, v0, own, [&](size_t, int c) { nt += df_mc_ntri[c]; });
}

template <int VX>
__global__ void __launch_bounds__(EX_THREADS) mesh_count_kernel(const ExtractParams p, int *vblock_counts, int *tblock_counts)
{
    DF_PDL_ENTRY();
    const size_t q0 = (size_t)blockIdx.x * EX_THREADS * EX_QPT;
    uint32_t own[EX_QPT][VX];
    load_block_quads<VX>(p, q0, own);
    int nv = 0, nt = 0;
#pragma unroll
    for (int i = 0; i < EX_QPT; ++i) quad_mesh_counts<VX>(p, (q0 + (size_t)(i * EX_THREADS) + threadIdx.x) * VX, own[i], nv, nt);
    if (!__syncthreads_or(nv | nt)) {
        if (threadIdx.x == 0) { vblock_counts[blockIdx.x] = 0; tblock_counts[blockIdx.x] = 0; }
        return;
    }
    int vtotal, ttotal;
    block_exclusive_scan(nv, &vtotal);
    block_exclusive_scan(nt, &ttotal);
    if (threadIdx.x == 0) { vblock_counts[blockIdx.x] = vtotal; tblock_counts[blockIdx.x] = ttotal; }
}

template <int VX>
__global__ void __launch_bounds__(EX_THREADS) mesh_vertex_emit_kernel(const ExtractParams p, const int *block_counts, const int *offsets,
                                                                      const int *super_off, float4 *vertices, uint32_t *keys, int vcap)
{
    DF_PDL_ENTRY();
    if (block_counts[blockIdx.x] == 0) return;
    const size_t q0 = (size_t)blockIdx.x * EX_THREADS * EX_QPT;
    uint32_t own[EX_QPT][VX];
    load_block_quads<VX>(p, q0, own);
    int run = super_off[blockIdx.x >> 10] + offsets[blockIdx.x];
#pragma unroll
    for (int i = 0; i < EX_QPT; ++i) {
        const size_t v0 = (q0 + (size_t)(i * EX_THREADS) + threadIdx.x) * VX;
        int c = 0;
        thread_mesh_vertices<VX>(p, v0, own[i], [&](uint32_t, float3) { ++c; });
        int total;
        int k = run + block_exclusive_scan(c, &total);
        if (c)
            thread_mesh_vertices<VX>(p, v0, own[i], [&](uint32_t key, float3 q) {
                if (k < vcap) { vertices[k] = make_float4(q.x, q.y, q.z, 0.f); keys[k] = key; }
                ++k;
            });
        run += total;
    }
}

// index of the vertex with edge key `key`: binary search in the range of the block that owns the key's voxel
template <int VX>
__device__ __forceinline__ int find_vertex(const uint32_t *keys, uint32_t key, const int *block_counts, const int *offsets, const int *super_off)
{
    const int blk = (int)((key / 3u) / VX / (EX_THREADS * EX_QPT));
    int lo = super_off[blk >> 10] + offsets[blk], hi = lo + block_counts[blk];
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

template <int VX>
__global__ void __launch_bounds__(EX_THREADS) mesh_triangle_emit_kernel(const ExtractParams p, const int *vblock_counts, const int *voffsets,
                                                                        const int *vsuper_off, const uint32_t *keys, const int *counts, int vcap,
                                                                        const int *block_counts, const int *offsets, const int *super_off,
                                                                        int3 *triangles, int tcap)
{
    DF_PDL_ENTRY();
    if (block_counts[blockIdx.x] == 0 || counts[0] > vcap) return;    // vertex overflow: the indices cannot be resolved
    const size_t q0 = (size_t)blockIdx.x * EX_THREADS * EX_QPT;
    uint32_t own[EX_QPT][VX];
    load_block_quads<VX>(p, q0, own);
    const uint32_t sy = (uint32_t)p.Dx, sz = (uint32_t)p.Dx * (uint32_t)p.Dy;
    int run = super_off[blockIdx.x >> 10] + offsets[blockIdx.x];
#pragma unroll
    for (int i = 0; i < EX_QPT; ++i) {
        const size_t v0 = (q0 + (size_t)(i * EX_THREADS) + threadIdx.x) * VX;
        int c = 0;
        thread_mesh_cells<VX>(p, v0, own[i], [&](size_t, int cs) { c += df_mc_ntri[cs]; });
        int total;
        int k = run + block_exclusive_scan(c, &total);
        if (c)
            thread_mesh_cells<VX>(p, v0, own[i], [&](size_t v, int cs) {
                const int n = df_mc_ntri[cs];
                for (int t = 0; t < n; ++t, ++k) {
                    if (k >= tcap) continue;
                    int idx[3];
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        const signed char *e = df_mc_edges[df_mc_tris[cs][3 * t + q]];
                        const uint32_t owner = (uint32_t)v + (uint32_t)e[0] + sy * (uint32_t)e[1] + sz * (uint32_t)e[2];
                        idx[q] = find_vertex<VX>(keys, 3u * owner + (uint32_t)e[3], vblock_counts, voffsets, vsuper_off);
                    }
                    triangles[k] = make_int3(idx[0], idx[1], idx[2]);
                }
            });
        run += total;
    }
}

}  // namespace

extern "C" size_t df_extract_mesh_workspace_bytes(df_volume vol)
{
    return 2 * df_extract_workspace_bytes(vol);          // one set of block counts / offsets / super sums for vertices, one for triangles
}

extern "C" int df_extract_mesh(df_volume vol, df_aff3f pose, const unsigned char *activity, float *vertices, uint32_t *edge_keys, int vcap,
                               int32_t *triangles, int tcap, int *counts_dev, void *workspace, void *stream)
{
    if (vcap < 0 || tcap < 0 || !counts_dev || !workspace) return (int)cudaErrorInvalidValue;
    const int vx = pick_vx(vol);
    ExtractParams p = make_params(vol, pose, vx);
    p.activity = activity;
    const int nsuper = (p.nblocks + 1023) / 1024;
    if (nsuper > 1024) return (int)cudaErrorInvalidValue;               // > 2^20 blocks (volume > 1024^3 voxels)
    int *vcounts = (int *)workspace, *voff = vcounts + p.nblocks, *vsuper_tot = voff + p.nblocks, *vsuper_off = vsuper_tot + 1024;
    int *tcounts = (int *)workspace + df_extract_workspace_bytes(vol) / sizeof(int);
    int *toff = tcounts + p.nblocks, *tsuper_tot = toff + p.nblocks, *tsuper_off = tsuper_tot + 1024;
    cudaStream_t s = (cudaStream_t)stream;
    const dim3 grid(p.nblocks), block(EX_THREADS);
    if (vx == 4) launch_pdl(mesh_count_kernel<4>, grid, block, 0, s, p, vcounts, tcounts);
    else launch_pdl(mesh_count_kernel<1>, grid, block, 0, s, p, vcounts, tcounts);
    DF_LAUNCH_CHECK();
    // the scans report the true totals (capacity INT_MAX); the emit passes clamp
    launch_pdl(extract_scan_local_kernel, dim3(nsuper), dim3(1024), 0, s, (const int *)vcounts, voff, p.nblocks, vsuper_tot);
    launch_pdl(extract_scan_super_kernel, dim3(1), dim3(1024), 0, s, (const int *)vsuper_tot, nsuper, vsuper_off, INT_MAX, counts_dev);
    launch_pdl(extract_scan_local_kernel, dim3(nsuper), dim3(1024), 0, s, (const int *)tcounts, toff, p.nblocks, tsuper_tot);
    launch_pdl(extract_scan_super_kernel, dim3(1), dim3(1024), 0, s, (const int *)tsuper_tot, nsuper, tsuper_off, INT_MAX, counts_dev + 1);
    DF_LAUNCH_CHECK();
    if (vx == 4) {
        launch_pdl(mesh_vertex_emit_kernel<4>, grid, block, 0, s, p, (const int *)vcounts, (const int *)voff, (const int *)vsuper_off,
                   (float4 *)vertices, edge_keys, vcap);
        launch_pdl(mesh_triangle_emit_kernel<4>, grid, block, 0, s, p, (const int *)vcounts, (const int *)voff, (const int *)vsuper_off,
                   (const uint32_t *)edge_keys, (const int *)counts_dev, vcap, (const int *)tcounts, (const int *)toff, (const int *)tsuper_off,
                   (int3 *)triangles, tcap);
    } else {
        launch_pdl(mesh_vertex_emit_kernel<1>, grid, block, 0, s, p, (const int *)vcounts, (const int *)voff, (const int *)vsuper_off,
                   (float4 *)vertices, edge_keys, vcap);
        launch_pdl(mesh_triangle_emit_kernel<1>, grid, block, 0, s, p, (const int *)vcounts, (const int *)voff, (const int *)vsuper_off,
                   (const uint32_t *)edge_keys, (const int *)counts_dev, vcap, (const int *)tcounts, (const int *)toff, (const int *)tsuper_off,
                   (int3 *)triangles, tcap);
    }
    DF_LAUNCH_CHECK();
    return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// extract normals: reference ExtractNormals::operator() tsdf_volume.cu:714-795 (launched with 8x redundant threads,
// :817-831); here one thread per point, count optionally read from device memory.
namespace {
struct NormalsParams {
    const uint32_t *data;
    int Dx, Dy, Dz;
    float3 vs_inv, gd;
    Aff pose;
    Mat3 Rinv;
    const float4 *points;
    int n;
    const int *count_dev;
    float4 *out;
};

__device__ __forceinline__ float en_tsdf(const NormalsParams &p, int x, int y, int z)
{ return half_bits_to_float((unsigned short)(__ldg(p.data + x + (size_t)p.Dx * y + (size_t)p.Dx * p.Dy * z) & 0xffffu)); }

__device__ __forceinline__ float en_interpolate(const NormalsParams &p, const float3 cf)
{
    const float fx = floorf(cf.x), fy = floorf(cf.y), fz = floorf(cf.z);
    if (!(fx >= 0) || !(fy >= 0) || !(fz >= 0) || !(fx < (float)(p.Dx - 1)) || !(fy < (float)(p.Dy - 1)) || !(fz < (float)(p.Dz - 1)))
        return qnan();
    const int gx = (int)fx, gy = (int)fy, gz = (int)fz;
    const float a = cf.x - (float)gx, b = cf.y - (float)gy, c = cf.z - (float)gz;
    const float v000 = en_tsdf(p, gx, gy, gz), v001 = en_tsdf(p, gx, gy, gz + 1);
    const float v010 = en_tsdf(p, gx, gy + 1, gz), v011 = en_tsdf(p, gx, gy + 1, gz + 1);
    const float v100 = en_tsdf(p, gx + 1, gy, gz), v101 = en_tsdf(p, gx + 1, gy, gz + 1);
    const float v110 = en_tsdf(p, gx + 1, gy + 1, gz), v111 = en_tsdf(p, gx + 1, gy + 1, gz + 1);
    float tsdf = 0.f;
    tsdf += v000 * (1 - a) * (1 - b) * (1 - c);
    tsdf += v001 * (1 - a) * (1 - b) * c;
    tsdf += v010 * (1 - a) * b * (1 - c);
    tsdf += v011 * (1 - a) * b * c;
    tsdf += v100 * a * (1 - b) * (1 - c);
    tsdf += v101 * a * (1 - b) * c;
    tsdf += v110 * a * b * (1 - c);
    tsdf += v111 * a * b * c;
    return tsdf;
}

__global__ void __launch_bounds__(256) extract_normals_kernel(const NormalsParams p)
{
    DF_PDL_ENTRY();
    const int n = p.count_dev ? min(*p.count_dev, p.n) : p.n;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += gridDim.x * blockDim.x) {
        const float nanv = qnan();
        float3 nrm = make_float3(nanv, nanv, nanv);
        const float4 pt = p.points[idx];
        const float3 point = mat3_mul(p.Rinv, sub3(make_float3(pt.x, pt.y, pt.z), p.pose.t));
        const int gx = __float2int_rn(point.x * p.vs_inv.x), gy = __float2int_rn(point.y * p.vs_inv.y), gz = __float2int_rn(point.z * p.vs_inv.z);
        if (gx > 1 && gy > 1 && gz > 1 && gx < p.Dx - 2 && gy < p.Dy - 2 && gz < p.Dz - 2) {
            float3 t;
            t = point; t.x += p.gd.x; const float Fx1 = en_interpolate(p, mul3(t, p.vs_inv));
            t = point; t.x -= p.gd.x; const float Fx2 = en_interpolate(p, mul3(t, p.vs_inv));
            nrm.x = (Fx1 - Fx2) / p.gd.x;
            t = point; t.y += p.gd.y; const float Fy1 = en_interpolate(p, mul3(t, p.vs_inv));
            t = point; t.y -= p.gd.y; const float Fy2 = en_interpolate(p, mul3(t, p.vs_inv));
            nrm.y = (Fy1 - Fy2) / p.gd.y;
            t = point; t.z += p.gd.z; const float Fz1 = en_interpolate(p, mul3(t, p.vs_inv));
            t = point; t.z -= p.gd.z; const float Fz2 = en_interpolate(p, mul3(t, p.vs_inv));
            nrm.z = (Fz1 - Fz2) / p.gd.z;
            nrm = normalized3(mat_mul(p.pose.r0, p.pose.r1, p.pose.r2, nrm));
        }
        p.out[idx] = make_float4(nrm.x, nrm.y, nrm.z, 0.f);
    }
}
}  // namespace

extern "C" int df_extract_normals(df_volume vol, const float *points, int n_points, const int *count_dev, df_aff3f pose,
                                  const float *Rinv_host9, float delta_factor, float *out_normals, void *stream)
{
    if (n_points <= 0) return 0;
    NormalsParams p;
    p.data = vol.data;
    p.Dx = vol.dims[0]; p.Dy = vol.dims[1]; p.Dz = vol.dims[2];
    p.vs_inv = make_float3(1.f / vol.voxel_size[0], 1.f / vol.voxel_size[1], 1.f / vol.voxel_size[2]);
    p.gd = make_float3(vol.voxel_size[0] * delta_factor, vol.voxel_size[1] * delta_factor, vol.voxel_size[2] * delta_factor);
    p.pose = make_aff(pose);
    p.Rinv = make_mat3(Rinv_host9);
    p.points = (const float4 *)points; p.n = n_points; p.count_dev = count_dev; p.out = (float4 *)out_normals;
    const int blocks = count_dev ? 148 * 8 : div_up(n_points, 256);
    launch_pdl(extract_normals_kernel, dim3(blocks), dim3(256), 0, (cudaStream_t)stream, p);
    DF_LAUNCH_CHECK();
    return 0;
}
