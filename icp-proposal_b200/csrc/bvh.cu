// bvh.cu - device LBVH construction, per-instance refit and exact nearest-primitive traversal.
//
// Replaces Scalismo's per-mesh query structures behind
//   target.operations.closestPointOnSurface   (NonRigidIcpProposal.scala:97, evaluators)
//   pointSet.findClosestPoint                  (NonRigidIcpProposal.scala:98,118)
// The static target BVH is built once on the device (Morton codes -> radix sort -> Karras 2012
// topology -> bottom-up boxes); the model-mesh BVHs keep the reference-mesh topology and are refit
// per chain and per sample. Boxes are FP32 and conservative (rounded outwards + slack), the leaf
// tests are exact FP64, so the result equals a brute-force FP64 search (ties -> lowest index).
#include <cub/device/device_radix_sort.cuh>

#include "bvh_device.cuh"
#include <algorithm>
#include <string>

#include "icp_internal.h"

namespace icp {

void bvh_refit_atomic(Bvh &b, int instances, const double *d_X, int N, const int *d_tris, cudaStream_t s);

// ---------------------------------------------------------------------------------------------------
// construction
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long expand21(unsigned long long v) {
    v &= 0x1fffffull;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}

__global__ void k_morton(int n_prims, int n, int prim_kind, const double *__restrict__ verts,
                         const int *__restrict__ tris, double lox, double loy, double loz, double sx, double sy,
                         double sz, unsigned long long *__restrict__ keys, int *__restrict__ vals) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int p = i < n_prims ? i : 0;  // a single primitive is duplicated so that the tree has a root
    double cx, cy, cz;
    if (prim_kind == 0) {
        int a = tris[3 * p], b = tris[3 * p + 1], c = tris[3 * p + 2];
        cx = (verts[3 * a] + verts[3 * b] + verts[3 * c]) * (1.0 / 3.0);
        cy = (verts[3 * a + 1] + verts[3 * b + 1] + verts[3 * c + 1]) * (1.0 / 3.0);
        cz = (verts[3 * a + 2] + verts[3 * b + 2] + verts[3 * c + 2]) * (1.0 / 3.0);
    } else {
        cx = verts[3 * p]; cy = verts[3 * p + 1]; cz = verts[3 * p + 2];
    }
    double fx = fmin(fmax((cx - lox) * sx, 0.0), 1.0), fy = fmin(fmax((cy - loy) * sy, 0.0), 1.0),
           fz = fmin(fmax((cz - loz) * sz, 0.0), 1.0);
    unsigned long long ix = (unsigned long long)(fx * 2097151.0), iy = (unsigned long long)(fy * 2097151.0),
                       iz = (unsigned long long)(fz * 2097151.0);
    keys[i] = (expand21(ix) << 2) | (expand21(iy) << 1) | expand21(iz);
    vals[i] = p;
}

__device__ __forceinline__ int lbvh_delta(const unsigned long long *keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    unsigned long long a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz(i ^ j);
    return __clzll(a ^ b);
}

__global__ void k_karras(int n, const unsigned long long *__restrict__ keys, int2 *__restrict__ children,
                         int *__restrict__ parent) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    if (i == 0) parent[0] = -1;
    int d = (lbvh_delta(keys, n, i, i + 1) - lbvh_delta(keys, n, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = lbvh_delta(keys, n, i, i - d);
    int lmax = 2;
    while (lbvh_delta(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (lbvh_delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = lbvh_delta(keys, n, i, j);
    int s = 0, t = l;
    do {
        t = (t + 1) / 2;
        if (lbvh_delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int lo = min(i, j), hi = max(i, j);
    int left, right;
    if (lo == gamma) { left = ~gamma; parent[n - 1 + gamma] = i; } else { left = gamma; parent[gamma] = i; }
    if (hi == gamma + 1) { right = ~(gamma + 1); parent[n - 1 + gamma + 1] = i; } else { right = gamma + 1; parent[gamma + 1] = i; }
    children[i] = make_int2(left, right);
}

// one thread per (instance, leaf): leaf box, then climb; the second arrival at a node merges
__global__ void k_refit(int n, int instances, int prim_kind, const int *__restrict__ prim,
                        const int2 *__restrict__ children, const int *__restrict__ parent,
                        const double *__restrict__ X, int N, const int *__restrict__ tris, float slack,
                        float4 *__restrict__ nodes, float4 *nodebox, int *counters) {
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= (long long)n * instances) return;
    int inst = (int)(g / n), slot = (int)(g % n);
    const double *Xi = X + (size_t)inst * N * 3;
    int p = prim[slot];
    double lx, ly, lz, hx, hy, hz;
    if (prim_kind == 0) {
        int a = tris[3 * p], b = tris[3 * p + 1], c = tris[3 * p + 2];
        lx = fmin(fmin(Xi[3 * a], Xi[3 * b]), Xi[3 * c]); hx = fmax(fmax(Xi[3 * a], Xi[3 * b]), Xi[3 * c]);
        ly = fmin(fmin(Xi[3 * a + 1], Xi[3 * b + 1]), Xi[3 * c + 1]); hy = fmax(fmax(Xi[3 * a + 1], Xi[3 * b + 1]), Xi[3 * c + 1]);
        lz = fmin(fmin(Xi[3 * a + 2], Xi[3 * b + 2]), Xi[3 * c + 2]); hz = fmax(fmax(Xi[3 * a + 2], Xi[3 * b + 2]), Xi[3 * c + 2]);
    } else {
        lx = hx = Xi[3 * p]; ly = hy = Xi[3 * p + 1]; lz = hz = Xi[3 * p + 2];
    }
    float4 lo = make_float4(__double2float_rd(lx) - slack, __double2float_rd(ly) - slack, __double2float_rd(lz) - slack, 0.f);
    float4 hi = make_float4(__double2float_ru(hx) + slack, __double2float_ru(hy) + slack, __double2float_ru(hz) + slack, 0.f);
    float4 *nb = nodebox + (size_t)inst * (2 * n - 1) * 2;
    float4 *nd = nodes + (size_t)inst * (n - 1) * 3;
    int *cnt = counters + (size_t)inst * (n - 1);
    __stcg(&nb[2 * (n - 1 + slot)], lo);
    __stcg(&nb[2 * (n - 1 + slot) + 1], hi);
    int node = parent[n - 1 + slot];
    while (node >= 0) {
        __threadfence();
        int old = atomicAdd(&cnt[node], 1);
        if (old == 0) return;
        __threadfence();
        int2 ch = children[node];
        int li = ch.x >= 0 ? ch.x : n - 1 + (~ch.x), ri = ch.y >= 0 ? ch.y : n - 1 + (~ch.y);
        float4 llo = __ldcg(&nb[2 * li]), lhi = __ldcg(&nb[2 * li + 1]);
        float4 rlo = __ldcg(&nb[2 * ri]), rhi = __ldcg(&nb[2 * ri + 1]);
        nd[3 * node] = make_float4(llo.x, llo.y, llo.z, lhi.x);
        nd[3 * node + 1] = make_float4(lhi.y, lhi.z, rlo.x, rlo.y);
        nd[3 * node + 2] = make_float4(rlo.z, rhi.x, rhi.y, rhi.z);
        __stcg(&nb[2 * node], make_float4(fminf(llo.x, rlo.x), fminf(llo.y, rlo.y), fminf(llo.z, rlo.z), 0.f));
        __stcg(&nb[2 * node + 1], make_float4(fmaxf(lhi.x, rhi.x), fmaxf(lhi.y, rhi.y), fmaxf(lhi.z, rhi.z), 0.f));
        node = parent[node];
    }
}

// level-synchronous refit: one CTA per instance walks the internal nodes in order of increasing height (schedule
// computed once at build time); no atomics, no counters, boxes of finished levels are read back through L2.
__global__ void __launch_bounds__(1024) k_refit_levels(int n, int prim_kind, const int *__restrict__ prim,
                                                      const int2 *__restrict__ children, const int *__restrict__ order,
                                                      const int *__restrict__ level_off, int n_levels,
                                                      const double *__restrict__ X, int N, const int *__restrict__ tris,
                                                      float slack, float4 *__restrict__ nodes, float4 *nodebox) {
    const int inst = blockIdx.x;
    const double *Xi = X + (size_t)inst * N * 3;
    float4 *nb = nodebox + (size_t)inst * (2 * n - 1) * 2;
    float4 *nd = nodes + (size_t)inst * (n - 1) * 3;
    for (int slot = threadIdx.x; slot < n; slot += blockDim.x) {
        int p = prim[slot];
        double lx, ly, lz, hx, hy, hz;
        if (prim_kind == 0) {
            int a = tris[3 * p], b = tris[3 * p + 1], c = tris[3 * p + 2];
            lx = fmin(fmin(Xi[3 * a], Xi[3 * b]), Xi[3 * c]); hx = fmax(fmax(Xi[3 * a], Xi[3 * b]), Xi[3 * c]);
            ly = fmin(fmin(Xi[3 * a + 1], Xi[3 * b + 1]), Xi[3 * c + 1]); hy = fmax(fmax(Xi[3 * a + 1], Xi[3 * b + 1]), Xi[3 * c + 1]);
            lz = fmin(fmin(Xi[3 * a + 2], Xi[3 * b + 2]), Xi[3 * c + 2]); hz = fmax(fmax(Xi[3 * a + 2], Xi[3 * b + 2]), Xi[3 * c + 2]);
        } else {
            lx = hx = Xi[3 * p]; ly = hy = Xi[3 * p + 1]; lz = hz = Xi[3 * p + 2];
        }
        __stcg(&nb[2 * (n - 1 + slot)], make_float4(__double2float_rd(lx) - slack, __double2float_rd(ly) - slack, __double2float_rd(lz) - slack, 0.f));
        __stcg(&nb[2 * (n - 1 + slot) + 1], make_float4(__double2float_ru(hx) + slack, __double2float_ru(hy) + slack, __double2float_ru(hz) + slack, 0.f));
    }
    __syncthreads();
    for (int lev = 0; lev < n_levels; lev++) {
        for (int k = level_off[lev] + threadIdx.x; k < level_off[lev + 1]; k += blockDim.x) {
            int node = order[k];
            int2 ch = children[node];
            int li = ch.x >= 0 ? ch.x : n - 1 + (~ch.x), ri = ch.y >= 0 ? ch.y : n - 1 + (~ch.y);
            float4 llo = __ldcg(&nb[2 * li]), lhi = __ldcg(&nb[2 * li + 1]);
            float4 rlo = __ldcg(&nb[2 * ri]), rhi = __ldcg(&nb[2 * ri + 1]);
            nd[3 * node] = make_float4(llo.x, llo.y, llo.z, lhi.x);
            nd[3 * node + 1] = make_float4(lhi.y, lhi.z, rlo.x, rlo.y);
            nd[3 * node + 2] = make_float4(rlo.z, rhi.x, rhi.y, rhi.z);
            __stcg(&nb[2 * node], make_float4(fminf(llo.x, rlo.x), fminf(llo.y, rlo.y), fminf(llo.z, rlo.z), 0.f));
            __stcg(&nb[2 * node + 1], make_float4(fmaxf(lhi.x, rhi.x), fmaxf(lhi.y, rhi.y), fmaxf(lhi.z, rhi.z), 0.f));
        }
        __syncthreads();
    }
}

void bvh_refit(Bvh &b, int instances, const double *d_X, int N, const int *d_tris, cudaStream_t s) {
    // ICPCUDA_REFIT = levels256 | levels1024 | atomic forces one variant (experiments; all three write the same boxes)
    static const std::string mode = getenv("ICPCUDA_REFIT") ? getenv("ICPCUDA_REFIT") : "";
    // 1024 threads per instance from 2048 primitives on: with one CTA per instance the refit is bound by the L2 round trips
    // of its own threads (measured: femur, 3240 triangles x 2368 chains 0.95 -> 0.72 ms; face-sized, 56 k triangles x 148
    // chains 2.77 -> 2.41 ms; profiles/r2_session3.md)
    const int threads = mode == "levels256" ? 256 : mode == "levels1024" ? 1024 : (b.n >= 2048 ? 1024 : 256);
    if (b.n_levels > 0 && instances >= 8 && mode != "atomic") {
        ProfScope _ps(ST_REFIT, s);
        int n = b.n;
        b.nodes.ensure((size_t)instances * (n - 1) * 3);
        b.nodebox.ensure((size_t)instances * (2 * n - 1) * 2);
        b.instances = instances;
        k_refit_levels<<<instances, threads, 0, s>>>(n, b.prim_kind, b.prim.p, b.children.p, b.order.p, b.level_off.p, b.n_levels,
                                                 d_X, N, d_tris, b.slack, b.nodes.p, b.nodebox.p);
        ICP_CUDA(cudaGetLastError());
        return;
    }
    bvh_refit_atomic(b, instances, d_X, N, d_tris, s);
}

void bvh_refit_atomic(Bvh &b, int instances, const double *d_X, int N, const int *d_tris, cudaStream_t s) {
    ProfScope _ps(ST_REFIT, s);
    int n = b.n;
    b.nodes.ensure((size_t)instances * (n - 1) * 3);
    b.nodebox.ensure((size_t)instances * (2 * n - 1) * 2);
    b.counters.ensure((size_t)instances * (n - 1));
    b.instances = instances;
    ICP_CUDA(cudaMemsetAsync(b.counters.p, 0, sizeof(int) * (size_t)instances * (n - 1), s));
    long long total = (long long)n * instances;
    int threads = 128;
    k_refit<<<(unsigned)((total + threads - 1) / threads), threads, 0, s>>>(
        n, instances, b.prim_kind, b.prim.p, b.children.p, b.parent.p, d_X, N, d_tris, b.slack, b.nodes.p,
        b.nodebox.p, b.counters.p);
    ICP_CUDA(cudaGetLastError());
}

// static structures: the three float4 of child boxes and the child links of a node in one aligned 64-byte record
__global__ void k_pack_nodes(int n_internal, const int2 *__restrict__ children, const float4 *__restrict__ nodes,
                             float4 *__restrict__ packed) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_internal) return;
    packed[4 * i] = nodes[3 * i];
    packed[4 * i + 1] = nodes[3 * i + 1];
    packed[4 * i + 2] = nodes[3 * i + 2];
    packed[4 * i + 3] = make_float4(__int_as_float(children[i].x), __int_as_float(children[i].y), 0.f, 0.f);
}

void bvh_build(Bvh &b, int prim_kind, int n_prims, const double *d_verts, const int *d_tris, double scale,
               cudaStream_t s) {
    ICP_REQUIRE(n_prims >= 1, "bvh_build: empty primitive set");
    int n = n_prims < 2 ? 2 : n_prims;
    b.n = n;
    b.prim_kind = prim_kind;
    b.slack = (float)(scale * 1e-6) + 1e-30f;
    b.children.alloc(n - 1);
    b.parent.alloc(2 * n - 1);
    b.prim.alloc(n);
    // bounding box of the vertices (host side: one-off, tiny)
    int nv_needed = 0;
    std::vector<int> htris;
    if (prim_kind == 0) {
        htris.resize((size_t)3 * n_prims);
        ICP_CUDA(cudaMemcpyAsync(htris.data(), d_tris, sizeof(int) * 3 * n_prims, cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        for (int v : htris) nv_needed = v + 1 > nv_needed ? v + 1 : nv_needed;
    } else {
        nv_needed = n_prims;
    }
    std::vector<double> hv((size_t)3 * nv_needed);
    ICP_CUDA(cudaMemcpyAsync(hv.data(), d_verts, sizeof(double) * 3 * nv_needed, cudaMemcpyDeviceToHost, s));
    ICP_CUDA(cudaStreamSynchronize(s));
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int v = 0; v < nv_needed; v++)
        for (int d = 0; d < 3; d++) {
            double x = hv[3 * v + d];
            if (x < lo[d]) lo[d] = x;
            if (x > hi[d]) hi[d] = x;
        }
    double sc[3];
    for (int d = 0; d < 3; d++) sc[d] = hi[d] > lo[d] ? 1.0 / (hi[d] - lo[d]) : 0.0;

    DevBuf<unsigned long long> keys, keys2;
    DevBuf<int> vals;
    keys.alloc(n); keys2.alloc(n); vals.alloc(n);
    int threads = 128;
    k_morton<<<(n + threads - 1) / threads, threads, 0, s>>>(n_prims, n, prim_kind, d_verts, d_tris, lo[0], lo[1], lo[2],
                                                              sc[0], sc[1], sc[2], keys.p, vals.p);
    ICP_CUDA(cudaGetLastError());
    size_t tmp_bytes = 0;
    ICP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys.p, keys2.p, vals.p, b.prim.p, n, 0, 64, s));
    DevBuf<unsigned char> tmp;
    tmp.alloc(tmp_bytes);
    ICP_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, keys.p, keys2.p, vals.p, b.prim.p, n, 0, 64, s));
    k_karras<<<(n - 1 + threads - 1) / threads, threads, 0, s>>>(n, keys2.p, b.children.p, b.parent.p);
    ICP_CUDA(cudaGetLastError());
    // bottom-up schedule for the level-synchronous refit: internal nodes sorted by height
    {
        std::vector<int2> hch(n - 1);
        ICP_CUDA(cudaMemcpyAsync(hch.data(), b.children.p, sizeof(int2) * (n - 1), cudaMemcpyDeviceToHost, s));
        ICP_CUDA(cudaStreamSynchronize(s));
        std::vector<int> height(n - 1, -1), stack;
        stack.push_back(0);
        while (!stack.empty()) {   // iterative post-order
            int v = stack.back();
            int l = hch[v].x, r = hch[v].y;
            int hl = l < 0 ? 0 : height[l], hr = r < 0 ? 0 : height[r];
            if (hl >= 0 && hr >= 0) { height[v] = 1 + (hl > hr ? hl : hr); stack.pop_back(); }
            else { if (l >= 0 && height[l] < 0) stack.push_back(l); if (r >= 0 && height[r] < 0) stack.push_back(r); }
        }
        int maxh = 0;
        for (int v = 0; v < n - 1; v++) maxh = height[v] > maxh ? height[v] : maxh;
        std::vector<int> off(maxh + 1, 0), order(n - 1);
        for (int v = 0; v < n - 1; v++) off[height[v]]++;           // heights are 1 .. maxh
        for (int h = 1, acc = 0; h <= maxh; h++) { int c = off[h]; off[h] = acc; acc += c; }
        std::vector<int> fill(off.begin(), off.end());
        for (int v = 0; v < n - 1; v++) order[fill[height[v]]++] = v;
        std::vector<int> level_off(maxh + 1);
        for (int h = 1; h <= maxh; h++) level_off[h - 1] = off[h];
        level_off[maxh] = n - 1;
        b.order.upload(order.data(), order.size(), s);
        b.level_off.upload(level_off.data(), level_off.size(), s);
        b.n_levels = maxh;
        ICP_CUDA(cudaStreamSynchronize(s));
    }
    bvh_refit_atomic(b, 1, d_verts, nv_needed, d_tris, s);
    b.packed.alloc((size_t)(n - 1) * 4);
    k_pack_nodes<<<(n - 1 + threads - 1) / threads, threads, 0, s>>>(n - 1, b.children.p, b.nodes.p, b.packed.p);
    ICP_CUDA(cudaGetLastError());
    ICP_CUDA(cudaStreamSynchronize(s));
}

constexpr int kStack = 64;
constexpr int kStackShared = 12;   // stack entries per thread kept in shared memory; deeper entries spill to local memory
constexpr int kNearestThreads = 128;
constexpr int kDone = 0x7ffffffe;

#ifdef ICP_CP_TIMING
// experiment build only (ICPCUDA_LIB_TAG=timing ICPCUDA_NVCC_EXTRA=-DICP_CP_TIMING, tools/cp_chain_major.py): k_nearest
// adds up, over all its launches since the last reset, [0] warp iterations and [1] lane iterations of the descent phase,
// [2] warp rounds and [3] lane tests of the leaf phase, [4] warps and [5] live queries. [1] / [0] is the number of lanes
// active per node visit, [3] / [2] per leaf test.
__device__ unsigned long long g_cp_count[6];
#define ICP_CPT(...) __VA_ARGS__
#else
#define ICP_CPT(...)
#endif

// Traversal in two alternating phases per warp ("while-while" with postponed leaves): every lane first descends through
// internal nodes until it holds a leaf (or has nothing left), then the warp reconverges and all lanes holding a leaf run
// the exact FP64 primitive test together. Static structures read one 64-byte packed node (child boxes + child links);
// per-chain (refitted) structures read the shared topology and their own boxes.
//
// HDMAX (Hausdorff evaluator, HausdorffDistanceEvaluator.scala:31-35: only the LARGEST of a chain's distances is used): the
// early-break scheme of directed Hausdorff distances. chain_max[c] holds the largest exact squared distance any finished
// query of chain c has produced (atomicMax on the bits of a non-negative double). A query whose current upper bound is
// already <= chain_max[c] cannot raise the maximum and stops - after its seed test in most cases; its d2 output is then an
// upper bound <= the chain's maximum, so the maximum over the outputs stays the exact Hausdorff distance. The warps of a
// launch rotate over the chains (warp w -> chain w % C, 32-query block (w / C) * blk_stride % n_blk of that chain), so the
// first wave finishes a few blocks of EVERY chain and the following waves prune against those maxima.
//
// MT (several static targets, TargetRec): query row c first reads the leaf count, packed nodes, primitive ids and leaf data
// of its own target, record mt_rec[mt_idx[c]]; the walk is the single-target one. The MT = false instantiations never read
// the two trailing arguments.
template <int PRIM, bool DYNAMIC, bool HDMAX, bool MT>
__global__ void __launch_bounds__(kNearestThreads, 7) k_nearest(int n, const int2 *__restrict__ children,
                                                 const float4 *__restrict__ nodes, const int *__restrict__ prim,
                                                 const double *__restrict__ prim_data, const double *__restrict__ X,
                                                 const int *__restrict__ tris, int N, int C, long long nq,
                                                 const double *__restrict__ q, int q_per_chain,
                                                 const double *__restrict__ Xq, const int *__restrict__ q_ids, int Nq,
                                                 const int *__restrict__ perm, int *__restrict__ seed_slot,
                                                 int *__restrict__ out_prim, int *__restrict__ out_feat,
                                                 double *__restrict__ out_cp, double *__restrict__ out_d2,
                                                 unsigned long long *__restrict__ chain_max, int n_blk, int blk_stride, int lpw,
                                                 const TargetRec *__restrict__ mt_rec, const int *__restrict__ mt_idx) {
    __shared__ int s_stack_n[kStackShared][kNearestThreads];
    __shared__ float s_stack_d[kStackShared][kNearestThreads];
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    bool live;
    int c;
    long long i;
    if (HDMAX) {
        const long long w = g >> 5;
        live = w < (long long)n_blk * C;
        c = live ? (int)(w % C) : C - 1;
        const long long b = live ? ((w / C) * blk_stride) % n_blk : 0;
        i = b * 32 + (threadIdx.x & 31);
        if (i >= nq) { live = false; i = nq - 1; }
        g = (long long)c * nq + i;
    } else {
        // lpw < 32 (small batches): only the first lpw lanes of a warp take a query. A warp runs as many rounds as its slowest
        // lane needs; with few queries in all there are SMs to spare, and eight queries per warp finish sooner than thirty-two
        if (lpw < 32) g = (g >> 5) * lpw + (threadIdx.x & 31);
        live = (lpw >= 32 || (int)(threadIdx.x & 31) < lpw) && g < nq * C;
        if (!live) g = nq * C - 1;   // idle lanes stay in the warp-synchronous loop, write nothing
        // chain-major: consecutive lanes take the same query row of consecutive chains. The same model point in different
        // chains lies a few mm apart (a quarter of a target edge), so the lanes of a warp walk nearly the same nodes to the
        // same leaves and finish together; 32 consecutive rows of one chain spread over ~40 mm of the surface. With C = 1
        // this is the row order itself.
        if (nq * C <= 0x7fffffffLL) { const int gi = (int)g; c = gi % C; i = gi / C; }
        else { c = (int)(g % C); i = g / C; }
    }
    if (perm) i = perm[i];   // spatially sorted processing order, results in caller order
    if (!HDMAX) g = (long long)c * nq + i;
    if (MT) {
        const TargetRec &r = mt_rec[__ldg(mt_idx + c)];
        n = r.n[PRIM]; nodes = r.nodes[PRIM]; prim = r.prim[PRIM]; prim_data = r.data[PRIM];
    }
    double qx, qy, qz;
    if (q_ids) {
        const double *src = Xq + ((size_t)c * Nq + q_ids[i]) * 3;
        qx = src[0]; qy = src[1]; qz = src[2];
    } else {
        const double *src = q + ((q_per_chain ? (size_t)c * nq : 0) + i) * 3;
        qx = src[0]; qy = src[1]; qz = src[2];
    }
    const float4 *nd = DYNAMIC ? nodes + (size_t)c * (n - 1) * 3 : nodes;
    const double *Xi = DYNAMIC ? X + (size_t)c * N * 3 : nullptr;
    float fx = (float)qx, fy = (float)qy, fz = (float)qz;
    Hit h;
    h.d2 = INFINITY; h.x = h.y = h.z = 0.0; h.prim = 0x7fffffff; h.feat = -1; h.slot = -1;
    float best = INFINITY;
    int stack_n[kStack - kStackShared];
    float stack_d[kStack - kStackShared];
    int sp = 0, node = 0;
    const int tid = threadIdx.x;
    if (!live || !(qx == qx && qy == qy && qz == qz)) node = kDone;  // NaN query: no traversal, NaN result
    else if (seed_slot) {
        // upper bound from the primitive that answered this query last time; ties still resolve to the lowest index
        // because subtrees are only pruned when their lower bound exceeds the best distance
        const int s0 = seed_slot[g];
        if ((unsigned)s0 < (unsigned)n) {
            leaf_test<PRIM, DYNAMIC>(s0, prim, prim_data, Xi, tris, qx, qy, qz, h);
            best = __double2float_ru(h.d2);
        }
    }
    const unsigned long long *cmax = HDMAX ? chain_max + c : nullptr;
    bool pruned = false;
    // squared distances are >= 0: their bit patterns order like the values
    if (HDMAX && node != kDone && __double_as_longlong(h.d2) <= (long long)__ldcg(cmax)) { node = kDone; pruned = true; }
    auto pop = [&]() {
        int nn = kDone;
        while (sp > 0) {
            --sp;
            float d;
            int cand;
            if (sp < kStackShared) { d = s_stack_d[sp][tid]; cand = s_stack_n[sp][tid]; }
            else { d = stack_d[sp - kStackShared]; cand = stack_n[sp - kStackShared]; }
            if (d <= best) { nn = cand; break; }
        }
        return nn;
    };
    ICP_CPT(unsigned cnt_desc = 0, cnt_leaf = 0, cnt_wdesc = 0, cnt_wleaf = 0;)
    while (true) {
        ICP_CPT(unsigned cnt_round = 0;)
        while ((unsigned)node < (unsigned)kDone) {   // internal node
            ICP_CPT(cnt_round++;)
            int2 ch;
            float4 a, b, cc;
            if (DYNAMIC) {
                ch = __ldg(&children[node]);
                a = __ldg(&nd[3 * node]); b = __ldg(&nd[3 * node + 1]); cc = __ldg(&nd[3 * node + 2]);
            } else {
                const float4 *pn = nodes + 4 * (size_t)node;
                a = __ldg(pn); b = __ldg(pn + 1); cc = __ldg(pn + 2);
                const float4 l = __ldg(pn + 3);
                ch = make_int2(__float_as_int(l.x), __float_as_int(l.y));
            }
            float dl = box_d2(a.x, a.y, a.z, a.w, b.x, b.y, fx, fy, fz);
            float dr = box_d2(b.z, b.w, cc.x, cc.y, cc.z, cc.w, fx, fy, fz);
            bool hl = dl <= best, hr = dr <= best;
            if (hl && hr) {
                int near = ch.x, far = ch.y;
                float dfar = dr;
                if (dr < dl) { near = ch.y; far = ch.x; dfar = dl; }
                if (sp < kStackShared) { s_stack_n[sp][tid] = far; s_stack_d[sp][tid] = dfar; sp++; }
                else if (sp < kStack) { stack_n[sp - kStackShared] = far; stack_d[sp - kStackShared] = dfar; sp++; }
                node = near;
            } else if (hl) node = ch.x;
            else if (hr) node = ch.y;
            else node = pop();
        }
        const bool at_leaf = node != kDone;
        ICP_CPT(cnt_desc += cnt_round; cnt_wdesc += __reduce_max_sync(0xffffffffu, cnt_round);
                cnt_leaf += at_leaf; cnt_wleaf += __any_sync(0xffffffffu, at_leaf);)
        if (!__any_sync(0xffffffffu, at_leaf)) break;
        if (at_leaf) {
            leaf_test<PRIM, DYNAMIC>(~node, prim, prim_data, Xi, tris, qx, qy, qz, h);
            best = __double2float_ru(h.d2);
            node = pop();
            if (HDMAX && node != kDone && __double_as_longlong(h.d2) <= (long long)__ldcg(cmax)) { node = kDone; pruned = true; }
        }
    }
    ICP_CPT({
        const unsigned sd = __reduce_add_sync(0xffffffffu, cnt_desc), sl = __reduce_add_sync(0xffffffffu, cnt_leaf),
                       nl = __reduce_add_sync(0xffffffffu, live ? 1u : 0u);
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&g_cp_count[0], (unsigned long long)cnt_wdesc); atomicAdd(&g_cp_count[1], (unsigned long long)sd);
            atomicAdd(&g_cp_count[2], (unsigned long long)cnt_wleaf); atomicAdd(&g_cp_count[3], (unsigned long long)sl);
            atomicAdd(&g_cp_count[4], 1ull); atomicAdd(&g_cp_count[5], (unsigned long long)nl);
        }
    })
    if (!live) return;
    if (HDMAX && !pruned && h.d2 == h.d2 && h.prim != 0x7fffffff) atomicMax(chain_max + c, (unsigned long long)__double_as_longlong(h.d2));
    if (h.prim == 0x7fffffff) { h.d2 = NAN; h.x = h.y = h.z = NAN; h.prim = -1; }
    if (seed_slot && (!HDMAX || h.slot >= 0)) seed_slot[g] = h.slot;
    if (out_prim) out_prim[g] = h.prim;
    if (out_feat) out_feat[g] = h.feat;
    if (out_cp) { out_cp[3 * g] = h.x; out_cp[3 * g + 1] = h.y; out_cp[3 * g + 2] = h.z; }
    if (out_d2) out_d2[g] = h.d2;
}

void launch_nearest(const NearestArgs &a, cudaStream_t s) {
    const bool mt = a.mt_rec != nullptr;
    if (!mt && a.wide && launch_nearest_wide(a, a.sm_count, s)) return;
    ProfScope _ps(a.prim_data ? ST_NEAREST_STATIC : ST_NEAREST_DYNAMIC, s);
    long long total = a.nq * a.C;
    if (total <= 0) return;
    const Bvh &b = *a.bvh;
    bool dynamic = a.prim_data == nullptr;
    int threads = kNearestThreads;
    unsigned blocks = (unsigned)((total + threads - 1) / threads);
    int n_blk = 0, blk_stride = 1;
    if (a.chain_max) {
        // 32-query blocks of a chain are visited with a stride coprime to their number (near the golden section), so that
        // successive waves sample the whole surface instead of sweeping it in Morton order
        n_blk = (int)((a.nq + 31) / 32);
        auto gcd = [](long long x, long long y) { while (y) { long long t = x % y; x = y; y = t; } return x; };
        blk_stride = std::max(1, (int)(n_blk * 0.618));
        while (gcd(blk_stride, n_blk) != 1) blk_stride++;
        blocks = (unsigned)(((long long)n_blk * a.C * 32 + threads - 1) / threads);
    }
    // a small batch is a chain of dependent latencies: eight queries per warp (see k_nearest) while the grid still fits one wave
    static const int lpw_small = getenv("ICPCUDA_LPW") ? atoi(getenv("ICPCUDA_LPW")) : 8;   // (experiments: 4 / 8 / 16)
    const int lpw = (!a.chain_max && total <= 16384 && lpw_small >= 1 && lpw_small < 32) ? lpw_small : 32;
    if (lpw < 32) blocks = (unsigned)((((total + lpw - 1) / lpw) * 32 + threads - 1) / threads);
#define ICP_LAUNCH_NEAREST_MT(P, D, H, M)                                                                            \
    k_nearest<P, D, H, M><<<blocks, threads, 0, s>>>(b.n, b.children.p, (D) ? b.nodes.p : b.packed.p, b.prim.p, a.prim_data, a.X, a.tris, \
                                               a.N, a.C, (long long)a.nq, a.q, a.q_per_chain, a.Xq, a.q_ids,     \
                                               a.Nq, a.perm, a.seed_slot, a.out_prim, a.out_feat, a.out_cp, a.out_d2, \
                                               a.chain_max, n_blk, blk_stride, lpw, a.mt_rec, a.mt_idx)
#define ICP_LAUNCH_NEAREST(P, D, H) ICP_LAUNCH_NEAREST_MT(P, D, H, false)
    if (mt) {
        ICP_REQUIRE(!dynamic && a.mt_idx, "launch_nearest: several targets need static structures and a target index");
        if (a.chain_max) {
            ICP_REQUIRE(b.prim_kind == 0 && !a.out_cp && !a.out_prim && !a.out_feat, "launch_nearest: chain_max is for distance-only triangle queries");
            ICP_LAUNCH_NEAREST_MT(0, false, true, true);
        } else if (b.prim_kind == 0) ICP_LAUNCH_NEAREST_MT(0, false, false, true);
        else ICP_LAUNCH_NEAREST_MT(1, false, false, true);
    } else if (a.chain_max) {
        ICP_REQUIRE(b.prim_kind == 0 && !a.out_cp && !a.out_prim && !a.out_feat, "launch_nearest: chain_max is for distance-only triangle queries");
        if (dynamic) ICP_LAUNCH_NEAREST(0, true, true); else ICP_LAUNCH_NEAREST(0, false, true);
    } else if (b.prim_kind == 0) {
        if (dynamic) ICP_LAUNCH_NEAREST(0, true, false); else ICP_LAUNCH_NEAREST(0, false, false);
    } else {
        if (dynamic) ICP_LAUNCH_NEAREST(1, true, false); else ICP_LAUNCH_NEAREST(1, false, false);
    }
#undef ICP_LAUNCH_NEAREST
#undef ICP_LAUNCH_NEAREST_MT
    ICP_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------
// nearest vertex of a small per-chain mesh, brute force: FP32 screening of all N vertices from shared memory,
// exact FP64 re-evaluation of every vertex the FP32 bound cannot exclude (result identical to an FP64 scan,
// ties -> lowest index). Replaces the vertex-BVH refit + traversal when N is a few thousand
// (currentMesh.pointSet.findClosestPoint, NonRigidIcpProposal.scala:118).
// ---------------------------------------------------------------------------------------------------
constexpr int kBruteQ = 2;  // queries per thread: one shared-memory broadcast of a vertex serves kBruteQ pairs per lane

__global__ void __launch_bounds__(128) k_nearest_vertex_brute(int N, int C, const double *__restrict__ X, long long nq,
                                                              const double *__restrict__ q, int q_per_chain, float scale,
                                                              int *__restrict__ out_prim, double *__restrict__ out_d2) {
    extern __shared__ double smd[];
    double *sx = smd;                                            // [3 N] exact coordinates
    // FP32 copy as three arrays [Np] (Np = N rounded up to even, padded with a vertex at infinity): a 64-bit load
    // yields the same coordinate of two consecutive vertices, the operand shape of the packed f32x2 arithmetic
    const int Np = (N + 1) & ~1;
    float *svx = reinterpret_cast<float *>(smd + 3 * (size_t)Np), *svy = svx + Np, *svz = svy + Np;
    const int c = blockIdx.y;
    const double *Xc = X + (size_t)c * N * 3;
    // tile load with 8 independent loads in flight per thread (a load -> store loop pays one L2 round trip per element)
    for (int e0 = threadIdx.x; e0 < 3 * N; e0 += 8 * blockDim.x) {
        double tmp[8];
#pragma unroll
        for (int u = 0; u < 8; u++) { int e = e0 + u * blockDim.x; tmp[u] = e < 3 * N ? __ldg(Xc + e) : 0.0; }
#pragma unroll
        for (int u = 0; u < 8; u++) { int e = e0 + u * blockDim.x; if (e < 3 * N) sx[e] = tmp[u]; }
    }
    __syncthreads();
    for (int v = threadIdx.x; v < Np; v += blockDim.x) {
        const bool real = v < N;
        svx[v] = real ? (float)sx[3 * v] : 1e30f; svy[v] = real ? (float)sx[3 * v + 1] : 1e30f; svz[v] = real ? (float)sx[3 * v + 2] : 1e30f;
    }
    __syncthreads();
    const long long i0 = (long long)blockIdx.x * blockDim.x * kBruteQ + threadIdx.x;
    double qx[kBruteQ], qy[kBruteQ], qz[kBruteQ];
    float fx[kBruteQ], fy[kBruteQ], fz[kBruteQ], best[kBruteQ], second[kBruteQ];
    int bid[kBruteQ];
#pragma unroll
    for (int t = 0; t < kBruteQ; t++) {
        long long i = i0 + (long long)t * blockDim.x;
        const double *src = q + ((q_per_chain ? (size_t)c * nq : 0) + (i < nq ? i : 0)) * 3;
        qx[t] = src[0]; qy[t] = src[1]; qz[t] = src[2];
        fx[t] = (float)qx[t]; fy[t] = (float)qy[t]; fz[t] = (float)qz[t];
        best[t] = INFINITY; second[t] = INFINITY; bid[t] = -1;
    }
    // single FP32 pass: minimum, runner-up and argmin; two vertices per step with packed f32x2 arithmetic (sm_100:
    // FADD2 / FMUL2 / FFMA2 - half the instructions of the distance evaluation). The rounding of each lane is that of
    // the scalar sequence d2f = fma(dx, dx, fma(dy, dy, dz * dz)), which the exact-rescan branch below repeats.
    float2 nqx[kBruteQ], nqy[kBruteQ], nqz[kBruteQ];
#pragma unroll
    for (int t = 0; t < kBruteQ; t++) { nqx[t] = make_float2(-fx[t], -fx[t]); nqy[t] = make_float2(-fy[t], -fy[t]); nqz[t] = make_float2(-fz[t], -fz[t]); }
#pragma unroll 4
    for (int v = 0; v < Np; v += 2) {
        const float2 px = *reinterpret_cast<const float2 *>(svx + v), py = *reinterpret_cast<const float2 *>(svy + v),
                     pz = *reinterpret_cast<const float2 *>(svz + v);
#pragma unroll
        for (int t = 0; t < kBruteQ; t++) {
            const float2 dx = __fadd2_rn(px, nqx[t]), dy = __fadd2_rn(py, nqy[t]), dz = __fadd2_rn(pz, nqz[t]);
            const float2 d2 = __ffma2_rn(dx, dx, __ffma2_rn(dy, dy, __fmul2_rn(dz, dz)));
            {
                const bool better = d2.x < best[t];
                second[t] = fminf(second[t], better ? best[t] : d2.x);
                bid[t] = better ? v : bid[t];
                best[t] = better ? d2.x : best[t];
            }
            {
                const bool better = d2.y < best[t];
                second[t] = fminf(second[t], better ? best[t] : d2.y);
                bid[t] = better ? v + 1 : bid[t];
                best[t] = better ? d2.y : best[t];
            }
        }
    }
#pragma unroll
    for (int t = 0; t < kBruteQ; t++) {
        long long i = i0 + (long long)t * blockDim.x;
        if (i >= nq) continue;
        // |d2f - d2| <= 2 sqrt(3) d delta + 3 delta^2 + 4 eps d2, delta = error of one FP32 coordinate difference.
        // If the runner-up lies beyond twice that bound the FP32 argmin is the exact FP64 argmin.
        const float S = fmaxf(fmaxf(fabsf(fx[t]), fabsf(fy[t])), fmaxf(fabsf(fz[t]), scale));
        const float delta = S * 2.4e-7f;  // 2^-22 S
        const float thresh = best[t] + 8.f * sqrtf(best[t]) * delta + 8.f * delta * delta + 1e-6f * best[t];
        int id = bid[t];
        double d2best = INFINITY;
        if (!(second[t] > thresh) || id < 0) {
            // rare: near-tie (or NaN query) -> exact FP64 scan of every vertex the FP32 bound cannot exclude
            id = -1;
            for (int v = 0; v < N; v++) {
                float dx = svx[v] - fx[t], dy = svy[v] - fy[t], dz = svz[v] - fz[t];
                float d2f = fmaf(dx, dx, fmaf(dy, dy, dz * dz));
                if (d2f <= thresh) {
                    double ex = qx[t] - sx[3 * v], ey = qy[t] - sx[3 * v + 1], ez = qz[t] - sx[3 * v + 2];
                    double d2 = ex * ex + ey * ey + ez * ez;
                    if (d2 < d2best || (d2 == d2best && v < id)) { d2best = d2; id = v; }
                }
            }
        } else {
            double ex = qx[t] - sx[3 * id], ey = qy[t] - sx[3 * id + 1], ez = qz[t] - sx[3 * id + 2];
            d2best = ex * ex + ey * ey + ez * ez;
        }
        size_t g = (size_t)c * nq + i;
        if (id < 0) d2best = NAN;
        if (out_prim) out_prim[g] = id;
        if (out_d2) out_d2[g] = d2best;
    }
}

// ---------------------------------------------------------------------------------------------------
// nearest vertex of a per-chain mesh through a vertex BVH whose boxes never leave the SM: one CTA per chain refits the
// reference-topology LBVH bottom-up into shared memory (level-synchronous, one __syncthreads per level instead of an
// L2 round trip) and walks it for the chain's queries, seeded with the previous answer of each query. Same boxes, same
// traversal order and tie rule as bvh_refit + k_nearest<points, dynamic>, so the results are identical; it replaces a
// 184 MB write + read of per-chain node boxes (C = 2368) by 39 KB of shared memory per CTA.
// ---------------------------------------------------------------------------------------------------
// lpw: queries per warp (32; 8 with 1024 threads per chain for small batches, where the SM has nothing else to do: the refit
// gets four times the threads and a warp waits for the slowest of eight walks instead of thirty-two)
__global__ void __launch_bounds__(1024) k_nearest_vertex_tree(int n, const int *__restrict__ prim, const int2 *__restrict__ children,
                                                              const int *__restrict__ order, const int *__restrict__ level_off,
                                                              int n_levels, const double *__restrict__ X, int N, float slack,
                                                              long long nq, const double *__restrict__ q, int q_per_chain,
                                                              int *__restrict__ seed_slot, int *__restrict__ out_prim,
                                                              double *__restrict__ out_d2, int lpw) {
    extern __shared__ float sbox[];                                // [n - 1][6] boxes of the internal nodes (lo, hi)
    const int c = blockIdx.x;
    const double *sx = X + (size_t)c * N * 3;                      // the chain's vertices stay in global memory (L1 / L2): each
                                                                   // is read once by the refit and ~5 times by the leaf tests,
                                                                   // and without them five CTAs share an SM instead of two
    // box of child `ch` of an internal node: an internal node's box from shared memory, a leaf's from its vertex
    auto child_box = [&](int ch, float (&b)[6]) {
        if (ch >= 0) {
#pragma unroll
            for (int k = 0; k < 6; k++) b[k] = sbox[6 * ch + k];
        } else {
            const double *v = sx + 3 * __ldg(&prim[~ch]);
            const double vx = __ldg(v), vy = __ldg(v + 1), vz = __ldg(v + 2);
            b[0] = __double2float_rd(vx) - slack; b[1] = __double2float_rd(vy) - slack; b[2] = __double2float_rd(vz) - slack;
            b[3] = __double2float_ru(vx) + slack; b[4] = __double2float_ru(vy) + slack; b[5] = __double2float_ru(vz) + slack;
        }
    };
    for (int lev = 0; lev < n_levels; lev++) {
        const int k1 = __ldg(&level_off[lev + 1]);
        for (int k = __ldg(&level_off[lev]) + threadIdx.x; k < k1; k += blockDim.x) {
            const int node = __ldg(&order[k]);
            const int2 ch = __ldg(&children[node]);
            float l[6], r[6];
            child_box(ch.x, l);
            child_box(ch.y, r);
#pragma unroll
            for (int d = 0; d < 3; d++) { sbox[6 * node + d] = fminf(l[d], r[d]); sbox[6 * node + 3 + d] = fmaxf(l[3 + d], r[3 + d]); }
        }
        __syncthreads();
    }
    const int q_lane = threadIdx.x & 31, q_warps = blockDim.x >> 5;
    for (long long i = (long long)(threadIdx.x >> 5) * lpw + q_lane; q_lane < lpw && i < nq; i += (long long)q_warps * lpw) {
        const long long g = (long long)c * nq + i;
        const double *src = q + ((q_per_chain ? (size_t)c * nq : 0) + i) * 3;
        const double qx = src[0], qy = src[1], qz = src[2];
        const float fx = (float)qx, fy = (float)qy, fz = (float)qz;
        double bd2 = INFINITY;
        int bprim = 0x7fffffff, bslot = -1;
        float best = INFINITY;
        auto leaf = [&](int slot) {
            const int p = __ldg(&prim[slot]);
            const double dx = qx - __ldg(sx + 3 * p), dy = qy - __ldg(sx + 3 * p + 1), dz = qz - __ldg(sx + 3 * p + 2);
            const double d2 = dx * dx + dy * dy + dz * dz;
            if (d2 < bd2 || (d2 == bd2 && p < bprim)) { bd2 = d2; bprim = p; bslot = slot; }
            best = __double2float_ru(bd2);
        };
        int stack_n[kStack];
        float stack_d[kStack];
        int sp = 0, node = 0;
        if (!(qx == qx && qy == qy && qz == qz)) node = 0x7ffffffe;  // NaN query: no traversal, NaN result
        else if (seed_slot) {
            const int s0 = seed_slot[g];
            if ((unsigned)s0 < (unsigned)n) leaf(s0);
        }
        while (node != 0x7ffffffe) {   // node is always internal here
            const int2 ch = __ldg(&children[node]);
            // a leaf child is a point: its exact distance costs what its box test would, so it is tested on the spot and
            // never pushed; only internal children get a box test
            float dl = INFINITY, dr = INFINITY;
            if (ch.x < 0) leaf(~ch.x);
            if (ch.y < 0) leaf(~ch.y);
            if (ch.x >= 0) {
                const float *b = sbox + 6 * ch.x;
                dl = box_d2(b[0], b[1], b[2], b[3], b[4], b[5], fx, fy, fz);
            }
            if (ch.y >= 0) {
                const float *b = sbox + 6 * ch.y;
                dr = box_d2(b[0], b[1], b[2], b[3], b[4], b[5], fx, fy, fz);
            }
            const bool hl = ch.x >= 0 && dl <= best, hr = ch.y >= 0 && dr <= best;
            if (hl && hr) {
                int near = ch.x, far = ch.y;
                float dfar = dr;
                if (dr < dl) { near = ch.y; far = ch.x; dfar = dl; }
                if (sp < kStack) { stack_n[sp] = far; stack_d[sp] = dfar; sp++; }
                node = near;
                continue;
            } else if (hl) { node = ch.x; continue; }
            else if (hr) { node = ch.y; continue; }
            node = 0x7ffffffe;
            while (sp > 0) {
                --sp;
                if (stack_d[sp] <= best) { node = stack_n[sp]; break; }
            }
        }
        if (bprim == 0x7fffffff) { bd2 = NAN; bprim = -1; }
        if (seed_slot) seed_slot[g] = bslot;
        if (out_prim) out_prim[g] = bprim;
        if (out_d2) out_d2[g] = bd2;
    }
}

bool nearest_vertex_tree_fits(const Bvh &b, int N) {
    return b.prim_kind == 1 && b.n_levels > 0 && b.n == N && sizeof(float) * 6 * (size_t)(b.n - 1) <= 110 * 1024;
}
bool nearest_vertex_brute_fits(int N) {
    return sizeof(double) * 3 * (size_t)((N + 1) & ~1) + sizeof(float) * 3 * (size_t)((N + 1) & ~1) <= 100 * 1024;
}

// false (nothing launched) when the tree does not fit shared memory or has no level schedule
bool launch_nearest_vertex_tree(const Bvh &b, int N, int C, const double *d_X, int64_t nq, const double *d_q, int q_per_chain,
                                int *d_seed, int *d_prim, double *d_d2, cudaStream_t s) {
    size_t smem = sizeof(float) * 6 * (size_t)(b.n - 1);
    if (!nearest_vertex_tree_fits(b, N) || C <= 0 || nq <= 0) return false;
    ProfScope _ps(ST_NEAREST_DYNAMIC, s);
    ICP_CUDA(cudaFuncSetAttribute(k_nearest_vertex_tree, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    static const int lpw_small = getenv("ICPCUDA_LPW") ? atoi(getenv("ICPCUDA_LPW")) : 8;   // (experiments: 4 / 8 / 16)
    const bool small = C <= 64 && lpw_small >= 1 && lpw_small < 32;   // the SMs are mostly idle: 1024 threads per chain, eight queries per warp
    k_nearest_vertex_tree<<<C, small ? 1024 : 256, smem, s>>>(b.n, b.prim.p, b.children.p, b.order.p, b.level_off.p, b.n_levels, d_X, N,
                                                              b.slack, (long long)nq, d_q, q_per_chain, d_seed, d_prim, d_d2, small ? lpw_small : 32);
    ICP_CUDA(cudaGetLastError());
    return true;
}

bool launch_nearest_vertex_brute(int N, int C, const double *d_X, int64_t nq, const double *d_q, int q_per_chain, double scale,
                                 int *d_prim, double *d_d2, cudaStream_t s) {
    size_t smem = sizeof(double) * 3 * (size_t)((N + 1) & ~1) + sizeof(float) * 3 * (size_t)((N + 1) & ~1);
    if (!nearest_vertex_brute_fits(N) || C <= 0 || nq <= 0) return false;
    ProfScope _ps(ST_NEAREST_DYNAMIC, s);
    if (smem > 48 * 1024) ICP_CUDA(cudaFuncSetAttribute(k_nearest_vertex_brute, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((unsigned)((nq + 128 * kBruteQ - 1) / (128 * kBruteQ)), C);
    k_nearest_vertex_brute<<<grid, 128, smem, s>>>(N, C, d_X, (long long)nq, d_q, q_per_chain, (float)scale, d_prim, d_d2);
    ICP_CUDA(cudaGetLastError());
    return true;
}

// ---------------------------------------------------------------------------------------------------
// large batches of free query points: process them in Morton order so that the 32 queries of a warp walk
// the same part of the tree (2x on random near-surface queries), write results in the caller's order
// ---------------------------------------------------------------------------------------------------
__global__ void k_query_morton(long long nq, const double *__restrict__ q, double lox, double loy, double loz, double sx,
                               double sy, double sz, unsigned int *__restrict__ keys, int *__restrict__ vals) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq) return;
    double fx = fmin(fmax((q[3 * i] - lox) * sx, 0.0), 1.0), fy = fmin(fmax((q[3 * i + 1] - loy) * sy, 0.0), 1.0),
           fz = fmin(fmax((q[3 * i + 2] - loz) * sz, 0.0), 1.0);
    if (!(fx == fx)) fx = 0.0;
    if (!(fy == fy)) fy = 0.0;
    if (!(fz == fz)) fz = 0.0;
    unsigned long long ix = (unsigned long long)(fx * 1023.0), iy = (unsigned long long)(fy * 1023.0), iz = (unsigned long long)(fz * 1023.0);
    // 8 bits per axis: three 8-bit radix passes
    keys[i] = (unsigned int)(((expand21(ix) << 2) | (expand21(iy) << 1) | expand21(iz)) >> 6);
    vals[i] = (int)i;
}

void launch_nearest_sorted(NearestArgs a, QuerySort &qs, const double lo[3], const double hi[3], cudaStream_t s) {
    const long long nq = a.nq;
    if (a.C != 1 || a.q == nullptr || nq < 16384 || nq > 0x7fffffffLL) { launch_nearest(a, s); return; }
    ProfScope _ps(ST_NEAREST_STATIC, s);
    qs.keys.ensure(nq); qs.keys2.ensure(nq); qs.vals.ensure(nq); qs.perm.ensure(nq);
    double sc[3], l2[3];
    for (int d = 0; d < 3; d++) {  // twice the structure's box: far-field queries still get distinct codes
        double c = 0.5 * (lo[d] + hi[d]), h = hi[d] - lo[d];
        l2[d] = c - h;
        sc[d] = h > 0 ? 1.0 / (2.0 * h) : 0.0;
    }
    k_query_morton<<<(unsigned)((nq + 255) / 256), 256, 0, s>>>(nq, a.q, l2[0], l2[1], l2[2], sc[0], sc[1], sc[2], qs.keys.p, qs.vals.p);
    ICP_CUDA(cudaGetLastError());
    size_t tmp_bytes = 0;
    ICP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, qs.keys.p, qs.keys2.p, qs.vals.p, qs.perm.p, (int)nq, 0, 24, s));
    qs.tmp.ensure(tmp_bytes);
    ICP_CUDA(cub::DeviceRadixSort::SortPairs(qs.tmp.p, tmp_bytes, qs.keys.p, qs.keys2.p, qs.vals.p, qs.perm.p, (int)nq, 0, 24, s));
    a.perm = qs.perm.p;
    launch_nearest(a, s);
}

// flags[i] = table[prim[i]] (0 when prim < 0); with rec, row i / per reads the table of its own target
__global__ void k_lookup_flags(long long n, const int *__restrict__ prim, const uint8_t *__restrict__ table, int table_n,
                               uint8_t *__restrict__ flags, const TargetRec *__restrict__ rec, const int *__restrict__ tidx,
                               long long per) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (rec) {
        const TargetRec &r = rec[tidx[i / per]];
        table = r.boundary; table_n = r.Nt;
    }
    int p = prim[i];
    flags[i] = (p >= 0 && p < table_n) ? table[p] : 0;
}

void launch_lookup_flags(int64_t n, const int *d_prim, const uint8_t *d_table, int table_n, uint8_t *d_flags,
                         cudaStream_t s, const TargetRec *rec, const int *tidx, int64_t per) {
    if (n <= 0) return;
    k_lookup_flags<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(n, d_prim, d_table, table_n, d_flags, rec, tidx, per);
    ICP_CUDA(cudaGetLastError());
}

}  // namespace icp

#ifdef ICP_CP_TIMING
// copies the six k_nearest counters to out (host memory); reset != 0 then clears them
extern "C" int32_t icp_debug_cp_counters(unsigned long long *out, int32_t reset) {
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess && out) e = cudaMemcpyFromSymbol(out, icp::g_cp_count, sizeof(icp::g_cp_count));
    if (e == cudaSuccess && reset) {
        const unsigned long long zero[6] = {0, 0, 0, 0, 0, 0};
        e = cudaMemcpyToSymbol(icp::g_cp_count, zero, sizeof(zero));
    }
    return (int32_t)e;
}
#endif
