// Near-duplicate groups (ffr_self_groups; DESIGN.md section 4, "Near-duplicate groups"): the connected components of the self-mode
// match graph, labelled by their smallest row.  The edges are the match list's pairs (run_pairs, unchanged); these three kernels run
// a lock-free union-find over them in place in the caller's labels:
//
//   G1 groups_init_kernel      labels[i] = i, *group_count = 0
//   G2 groups_hook_kernel      grid-stride over the accepted edges (their number read on the device): both roots with path
//                              halving, then the larger root is hooked under the smaller one with atomicCAS(parent, itself,
//                              smaller), retried from the winner's root when another edge got there first (ECL-CC's hook)
//   G3 groups_finalise_kernel  labels[i] = root of i (a read-only walk; each thread writes its own row only), rows with
//                              labels[i] == i counted warp-aggregated into *group_count
//
// Invariant: labels[v] <= v for every v, with equality exactly at the roots.  Init starts there, a hook only ever writes a smaller
// root into a root's own slot, and path halving only replaces a parent by one of its ancestors.  Every parent chain therefore
// strictly decreases, so a tree's root is its smallest row -- the label of the whole component once every edge has been hooked.
#include "ffr_common.cuh"

namespace ffr {

namespace {

constexpr int kThreads = 256;

// Root of v with path halving: each visited node is re-pointed at its grandparent.  A concurrent hook or halving only ever lowers
// a parent to one of its ancestors, so a stale read is still an ancestor and the walk still ends at the current root.
__device__ __forceinline__ int32_t find_root(int32_t* parent, int32_t v) {
    volatile int32_t* p = parent;
    int32_t par = p[v];
    while (par != v) {
        const int32_t next = p[par];
        if (next != par) p[v] = next;
        v = par;
        par = next;
    }
    return v;
}

// Root of v without writing: the final pass writes each row's own slot only, with its root.  (Halving there could re-point a
// slot another thread has just set to the root back at a stale, non-root ancestor.)
__device__ __forceinline__ int32_t walk_root(const int32_t* parent, int32_t v) {
    const volatile int32_t* p = parent;
    int32_t next;
    while ((next = p[v]) != v) v = next;
    return v;
}

__global__ void __launch_bounds__(kThreads)
groups_init_kernel(int32_t* __restrict__ labels, int64_t n, int64_t* __restrict__ group_count) {
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kThreads;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; i < n; i += stride)
        labels[i] = static_cast<int32_t>(i);
    if (blockIdx.x == 0 && threadIdx.x == 0) *group_count = 0;
}

// filled: the number of edge slots the pairs kernels wrote (it may exceed cap: only [0, cap) exist)
__global__ void __launch_bounds__(kThreads)
groups_hook_kernel(const int32_t* __restrict__ edge_a, const int32_t* __restrict__ edge_b, int64_t cap,
                   const unsigned long long* __restrict__ filled, int32_t* labels) {
    const unsigned long long f = *filled;
    const int64_t n_edges = f < static_cast<unsigned long long>(cap) ? static_cast<int64_t>(f) : cap;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kThreads;
    for (int64_t e = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; e < n_edges; e += stride) {
        int32_t a = find_root(labels, __ldg(edge_a + e));
        int32_t b = find_root(labels, __ldg(edge_b + e));
        while (a != b) {
            const int32_t hi = a > b ? a : b, lo = a > b ? b : a;
            const int32_t old = atomicCAS(labels + hi, hi, lo);
            if (old == hi) break;                              // hooked
            // hi was hooked under `old` meanwhile: continue from its new root
            a = find_root(labels, old);
            b = find_root(labels, lo);
        }
    }
}

__global__ void __launch_bounds__(kThreads)
groups_finalise_kernel(int32_t* labels, int64_t n, int64_t* __restrict__ group_count) {
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kThreads;
    const int lane = threadIdx.x & 31;
    // every lane of a warp runs the same number of iterations (the bound is rounded up to whole warps) for the ballot
    const int64_t n_up = (n + 31) / 32 * 32;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * kThreads + threadIdx.x; i < n_up; i += stride) {
        bool rep = false;
        if (i < n) {
            const int32_t r = walk_root(labels, static_cast<int32_t>(i));
            if (r != i) labels[i] = r;
            rep = r == i;
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, rep);
        if (lane == 0 && bal != 0u) atomicAdd(reinterpret_cast<unsigned long long*>(group_count), static_cast<unsigned long long>(__popc(bal)));
    }
}

unsigned grid_for(int64_t items) {
    const int64_t cap = static_cast<int64_t>(num_sms()) * 8;
    const int64_t g = (items + kThreads - 1) / kThreads;
    return static_cast<unsigned>(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace

int launch_groups_init(int32_t* labels, int64_t n, int64_t* group_count, cudaStream_t s) {
    groups_init_kernel<<<grid_for(n), kThreads, 0, s>>>(labels, n, group_count);
    FFR_LAUNCH_CHECK("groups_init");
    return FFR_OK;
}

int launch_groups_union(const int32_t* edge_a, const int32_t* edge_b, int64_t cap, const unsigned long long* filled, int32_t* labels,
                        int64_t n, int64_t* group_count, cudaStream_t s) {
    if (cap > 0) {            // (the edge count is on the device: the grid covers the capacity, the loop the count)
        groups_hook_kernel<<<grid_for(cap), kThreads, 0, s>>>(edge_a, edge_b, cap, filled, labels);
        FFR_LAUNCH_CHECK("groups_hook");
    }
    groups_finalise_kernel<<<grid_for(n), kThreads, 0, s>>>(labels, n, group_count);
    FFR_LAUNCH_CHECK("groups_finalise");
    return FFR_OK;
}

}  // namespace ffr
