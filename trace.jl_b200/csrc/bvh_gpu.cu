// bvh_gpu.cu — opt-in LBVH build on the GPU (trace_bvh_build_gpu, include/trace_cuda.h).
//
// A Karras (2012) binary radix tree over 63-bit Morton codes of the primitive centroids, emitted in the same flattened
// preorder node format as the host builders (first child = parent + 1), so every kernel walks it unchanged.  The tree
// is fully specified by its inputs (tests/test_gpu_lbvh.py restates it in numpy and compares bit for bit):
//   centroid   c = 0.5 bmin + 0.5 bmax (the host builders' formula), float32, unfused (-fmad=false);
//   quantised  q = min(2^21 - 1, floor((c - lo) * s)) with s = 2^21 / (hi - lo) per axis (0 for a flat axis), lo / hi
//              the exact centroid box;
//   key        x at bit 3k+2, y at 3k+1, z at 3k; sorted stably, so the order is lexicographic on (key, index);
//   split      at the highest bit where the range's first and last key differ (left child: that bit 0, axis 2 - h % 3),
//              or, for a range of equal keys, at the highest differing bit of the two positions (axis 0);
//   leaf       a range of <= max_node_primitives primitives (its whole subtree collapses into one node).
// Node boxes use Julia's min / max (-0.0 < +0.0): with NaN refused the union is exact and independent of the order in
// which the bottom-up threads arrive, so the output is deterministic.
#include <algorithm>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

#include "context.hpp"
#include "traverse.cuh"

// bvh_build.cpp: an uninitialised host handle with room for the given arrays (nullptr when out of memory)
trace_bvh* bvh_alloc(int64_t n_nodes, int64_t n_prims, trace_bvh_node** nodes, uint32_t** order);

namespace {

// Node ids: internal nodes 0 .. n-2 (Karras numbering), leaf k (sorted position k) is n-1+k.  The root is id 0 in both
// cases (n == 1: the single leaf).
struct Status {
    uint32_t cmin[3], cmax[3];      // centroid box as order-preserving keys (ord_key)
    uint32_t nan;                   // a centroid is NaN
    uint32_t root_size, root_depth; // emitted nodes, levels (root = 1)
    uint32_t bad;                   // mesh builds: a NaN normal (bit 0), a material index out of range (bit 1)
};

// float <-> uint32 in Julia's total order on non-NaN floats (-0.0 sorts below +0.0), so atomicMin / atomicMax pick it
__device__ __forceinline__ uint32_t ord_key(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_float(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}
__device__ __forceinline__ float centroid(const float* pb, int64_t i, int k) {
    return __fadd_rn(__fmul_rn(0.5f, pb[6 * i + k]), __fmul_rn(0.5f, pb[6 * i + 3 + k]));
}

// 21 bits -> every third bit of 63
__device__ __forceinline__ uint64_t spread3(uint64_t x) {
    x &= 0x1FFFFFull;
    x = (x | x << 32) & 0x1F00000000FFFFull;
    x = (x | x << 16) & 0x1F0000FF0000FFull;
    x = (x | x << 8) & 0x100F00F00F00F00Full;
    x = (x | x << 4) & 0x10C30C30C30C30C3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

// 1. exact centroid box (Julia order) and the NaN flag
__global__ void lbvh_centroid_box(const float* __restrict__ pb, int64_t n, Status* st) {
    uint32_t lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
    bool nan = false;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        for (int k = 0; k < 3; ++k) {
            const float c = centroid(pb, i, k);
            if (c != c) { nan = true; continue; }
            const uint32_t q = ord_key(c);
            lo[k] = min(lo[k], q);
            hi[k] = max(hi[k], q);
        }
    }
    for (int k = 0; k < 3; ++k) {
        lo[k] = __reduce_min_sync(0xFFFFFFFFu, lo[k]);
        hi[k] = __reduce_max_sync(0xFFFFFFFFu, hi[k]);
    }
    nan = __any_sync(0xFFFFFFFFu, nan);
    if ((threadIdx.x & 31) == 0) {
        for (int k = 0; k < 3; ++k) { atomicMin(&st->cmin[k], lo[k]); atomicMax(&st->cmax[k], hi[k]); }
        if (nan) atomicOr(&st->nan, 1u);
    }
}

// 2. Morton keys and the identity permutation (the sort's values)
__global__ void lbvh_keys(const float* __restrict__ pb, int64_t n, const Status* __restrict__ st, uint64_t* __restrict__ keys,
                          uint32_t* __restrict__ ids) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t key = 0;
    for (int k = 0; k < 3; ++k) {
        const float lo = ord_float(st->cmin[k]), hi = ord_float(st->cmax[k]);
        const float ext = __fsub_rn(hi, lo);
        const float s = ext > 0.0f ? __fdiv_rn(2097152.0f, ext) : 0.0f;
        const float v = __fmul_rn(__fsub_rn(centroid(pb, i, k), lo), s);
        // v >= 0 (c >= lo); a NaN (0 * inf on a denormal-thin axis) is position 0
        const uint32_t q = v >= 2097151.0f ? 2097151u : (v > 0.0f ? (uint32_t)floorf(v) : 0u);
        key |= spread3(q) << (2 - k);
    }
    keys[i] = key;
    ids[i] = (uint32_t)i;
}

// common prefix length of the strings (key, position) at sorted positions i and j; -1 outside [0, n)
__device__ __forceinline__ int delta(const uint64_t* __restrict__ K, int64_t n, int64_t i, int64_t j) {
    if (j < 0 || j >= n) return -1;
    const uint64_t a = K[i], b = K[j];
    if (a != b) return __clzll((long long)(a ^ b));
    return 64 + __clz((int)((uint32_t)i ^ (uint32_t)j));
}

// 3. hierarchy: internal node i finds its range and split (Karras 2012, Fig. 4)
__global__ void lbvh_hierarchy(const uint64_t* __restrict__ K, int64_t n, uint32_t* __restrict__ child,
                               int32_t* __restrict__ parent, uint32_t* __restrict__ first, uint32_t* __restrict__ count,
                               uint8_t* __restrict__ axis) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const int d = delta(K, n, i, i + 1) - delta(K, n, i, i - 1) > 0 ? 1 : -1;
    const int dmin = delta(K, n, i, i - d);
    int64_t lmax = 2;
    while (delta(K, n, i, i + lmax * d) > dmin) lmax *= 2;
    int64_t l = 0;
    for (int64_t t = lmax / 2; t >= 1; t /= 2)
        if (delta(K, n, i, i + (l + t) * d) > dmin) l += t;
    const int64_t j = i + l * d;
    const int dnode = delta(K, n, i, j);
    int64_t s = 0;
    for (int64_t div = 2;; div *= 2) {
        const int64_t t = (l + div - 1) / div;
        if (delta(K, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    const int64_t gamma = i + s * d + (d < 0 ? -1 : 0);
    const int64_t lo = d > 0 ? i : j, hi = d > 0 ? j : i;
    const uint32_t left = (uint32_t)(lo == gamma ? (n - 1) + gamma : gamma);
    const uint32_t right = (uint32_t)(hi == gamma + 1 ? (n - 1) + gamma + 1 : gamma + 1);
    child[2 * i] = left;
    child[2 * i + 1] = right;
    parent[left] = (int32_t)i;
    parent[right] = (int32_t)i;
    first[i] = (uint32_t)lo;
    count[i] = (uint32_t)(hi - lo + 1);
    const uint64_t x = K[lo] ^ K[hi];
    axis[i] = x ? (uint8_t)(2 - (63 - __clzll((long long)x)) % 3) : 0;
}

// 4. bottom-up: boxes, emitted subtree sizes and depths; one thread per leaf climbs while it is the second to arrive
__global__ void lbvh_bottom_up(const float* __restrict__ pb, const uint32_t* __restrict__ sorted_ids, int64_t n, int m,
                               const uint32_t* __restrict__ child, const int32_t* __restrict__ parent,
                               const uint32_t* __restrict__ count, uint32_t* arrive, float* box, uint32_t* size,
                               uint32_t* depth, Status* st) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    int64_t v = (n - 1) + k;
    const int64_t p0 = sorted_ids[k];
    for (int c = 0; c < 6; ++c) box[6 * v + c] = pb[6 * p0 + c];
    size[v] = 1;
    depth[v] = 1;
    for (;;) {
        const int32_t p = parent[v];
        if (p < 0) break;
        __threadfence();
        if (atomicAdd(&arrive[p], 1u) == 0) return;           // the sibling's thread continues
        __threadfence();
        const uint32_t l = child[2 * p], r = child[2 * p + 1];
        for (int c = 0; c < 3; ++c) {
            box[6 * (int64_t)p + c] = jl_min(__ldcg(&box[6 * (int64_t)l + c]), __ldcg(&box[6 * (int64_t)r + c]));
            box[6 * (int64_t)p + 3 + c] = jl_max(__ldcg(&box[6 * (int64_t)l + 3 + c]), __ldcg(&box[6 * (int64_t)r + 3 + c]));
        }
        const bool leaf = count[p] <= (uint32_t)m;
        size[p] = leaf ? 1u : 1u + __ldcg(&size[l]) + __ldcg(&size[r]);
        depth[p] = leaf ? 1u : 1u + max(__ldcg(&depth[l]), __ldcg(&depth[r]));
        v = p;
    }
    st->root_size = size[0];                                 // v == 0: the last thread to arrive at the root
    st->root_depth = depth[0];
}

// 5. emit: every emitted node finds its preorder slot by climbing to the root (left child = parent + 1, right child =
// parent + 1 + size(left); depth <= TR_STACK_SIZE is checked before this runs) and writes its record, interior offsets
// shifted by node_shift and leaf offsets by prim_shift (an attached mesh's place in the composed scene; else 0)
__global__ void lbvh_emit(int64_t n, int m, const uint32_t* __restrict__ child, const int32_t* __restrict__ parent,
                          const uint32_t* __restrict__ first, const uint32_t* __restrict__ count,
                          const uint8_t* __restrict__ axis, const float* __restrict__ box, const uint32_t* __restrict__ size,
                          uint32_t node_shift, uint32_t prim_shift, trace_bvh_node* __restrict__ out) {
    const int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (v >= 2 * n - 1) return;
    const bool internal = v < n - 1;
    const int32_t pv = parent[v];
    if (pv >= 0 && count[pv] <= (uint32_t)m) return;         // inside a collapsed subtree
    uint32_t pre = 0;
    for (int64_t c = v; c != 0;) {
        const int32_t p = parent[c];
        const uint32_t l = child[2 * p];
        pre += c == l ? 1u : 1u + size[l];
        c = p;
    }
    trace_bvh_node nd;
    for (int c = 0; c < 3; ++c) { nd.bmin[c] = box[6 * v + c]; nd.bmax[c] = box[6 * v + 3 + c]; }
    const uint32_t cnt = internal ? count[v] : 1u;
    if (cnt <= (uint32_t)m) {
        nd.offset = prim_shift + (internal ? first[v] : (uint32_t)(v - (n - 1)));
        nd.meta = TRACE_NODE_LEAF | cnt;
    } else {
        nd.offset = node_shift + pre + 1u + size[child[2 * v]];
        nd.meta = (uint32_t)axis[v] << 30;
    }
    out[pre] = nd;
}

// The build's device buffers, carved out of one allocation: carve() with base == 0 sizes it, then again on the real one.
// `pb` (the primitive bounds) and the node array are carved only when asked for.
struct Buffers {
    float* pb = nullptr; Status* st;
    uint64_t *keys, *keys_sorted; uint32_t *ids, *ids_sorted;                  // sort in / out
    uint32_t *child, *first, *count; int32_t* parent; uint8_t* axis;           // hierarchy (parent: every node)
    uint32_t* arrive; float* box; uint32_t *size, *depth;                      // bottom-up, every node
    trace_bvh_node* nodes = nullptr; void* sort_tmp;
    Carve k;
    char* base = nullptr;
    template <class T> T* take(int64_t count) { return reinterpret_cast<T*>(base + k.take((size_t)count * sizeof(T))); }
    void carve(int64_t n, size_t sort_bytes, bool with_pb, bool with_nodes) {
        const int64_t nn = 2 * n - 1;
        k = Carve();
        if (with_pb) pb = take<float>(6 * n);
        st = take<Status>(1);
        keys = take<uint64_t>(n); keys_sorted = take<uint64_t>(n); ids = take<uint32_t>(n); ids_sorted = take<uint32_t>(n);
        child = take<uint32_t>(2 * (n - 1)); first = take<uint32_t>(n - 1); count = take<uint32_t>(n - 1);
        parent = take<int32_t>(nn); axis = take<uint8_t>(n - 1);
        arrive = take<uint32_t>(n - 1); box = take<float>(6 * nn); size = take<uint32_t>(nn); depth = take<uint32_t>(nn);
        if (with_nodes) nodes = take<trace_bvh_node>(nn);
        sort_tmp = take<char>((int64_t)sort_bytes);
    }
    // one allocation for everything; freed by the destructor
    int alloc(int64_t n, size_t sort_bytes, bool with_pb, bool with_nodes) {
        carve(n, sort_bytes, with_pb, with_nodes);
        if (cudaMalloc(&base, k.used) != cudaSuccess) { cudaGetLastError(); base = nullptr; return LBVH_CUDA; }
        owned = true;
        carve(n, sort_bytes, with_pb, with_nodes);
        return 0;
    }
    // the caller's allocation of at least lbvh_scratch_bytes(n) bytes (with pb, without nodes); kept by the caller
    void borrow(void* scratch, int64_t n, size_t sort_bytes) {
        base = static_cast<char*>(scratch);
        carve(n, sort_bytes, true, false);
    }
    bool owned = false;
    ~Buffers() { if (owned) cudaFree(base); }
};

size_t sort_bytes_for(int64_t n, cudaStream_t s) {
    size_t bytes = 0;
    if (cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (const uint32_t*)nullptr,
                                        (uint32_t*)nullptr, (int)n, 0, 63, s) != cudaSuccess)
        return 0;
    return bytes;
}

// The device-resident core: bounds b.pb (device, [n][6]) -> keys, sorted order, hierarchy, boxes, subtree sizes and
// depths in `b`, and the status on the host.  Returns LBVH_OK, _NAN_BOUND, _TOO_DEEP or _CUDA.
void core_reset(cudaStream_t s, int64_t n, Buffers& b) {
    cudaMemsetAsync(b.st, 0xFF, sizeof(b.st->cmin), s);
    cudaMemsetAsync(&b.st->cmax, 0, sizeof(Status) - sizeof(b.st->cmin), s);
    cudaMemsetAsync(b.parent, 0xFF, (size_t)(2 * n - 1) * sizeof(int32_t), s);
    if (n > 1) cudaMemsetAsync(b.arrive, 0, (size_t)(n - 1) * sizeof(uint32_t), s);
}

// build_core without the reset and the read-back: the kernels that run after core_reset (and anything that reports
// into the status block).  LBVH_OK or LBVH_CUDA.
int core_enqueue(cudaStream_t s, int64_t n, int m, Buffers& b, size_t sort_bytes, PhaseTimer& ph) {
    const int T = 256;
    lbvh_centroid_box<<<(unsigned)std::min<int64_t>(blocks_for(n, T), 4096), T, 0, s>>>(b.pb, n, b.st);
    lbvh_keys<<<blocks_for(n, T), T, 0, s>>>(b.pb, n, b.st, b.keys, b.ids);
    ph.mark(s, "keys");
    if (cub::DeviceRadixSort::SortPairs(b.sort_tmp, sort_bytes, b.keys, b.keys_sorted, b.ids, b.ids_sorted, (int)n, 0, 63, s)
        != cudaSuccess)
        return LBVH_CUDA;
    ph.mark(s, "sort");
    if (n > 1) lbvh_hierarchy<<<blocks_for(n - 1, T), T, 0, s>>>(b.keys_sorted, n, b.child, b.parent, b.first, b.count, b.axis);
    ph.mark(s, "hierarchy");
    lbvh_bottom_up<<<blocks_for(n, T), T, 0, s>>>(b.pb, b.ids_sorted, n, m, b.child, b.parent, b.count, b.arrive, b.box,
                                                   b.size, b.depth, b.st);
    return cudaGetLastError() == cudaSuccess ? LBVH_OK : LBVH_CUDA;
}

// the core's verdict from its status block on the host
int core_verdict(const Status& hs) {
    if (hs.nan) return LBVH_NAN_BOUND;
    if (hs.root_depth > TR_STACK_SIZE) return LBVH_TOO_DEEP;   // the walks' stacks would overflow
    return LBVH_OK;
}

// core_enqueue, the status read back, its verdict
int core_run(cudaStream_t s, int64_t n, int m, Buffers& b, size_t sort_bytes, Status& hs, PhaseTimer& ph) {
    if (core_enqueue(s, n, m, b, sort_bytes, ph) != LBVH_OK ||
        cudaMemcpyAsync(&hs, b.st, sizeof(Status), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess)
        return LBVH_CUDA;
    ph.mark(s, "bottom-up");
    return core_verdict(hs);
}

int build_core(cudaStream_t s, int64_t n, int m, Buffers& b, size_t sort_bytes, Status& hs, PhaseTimer& ph) {
    core_reset(s, n, b);
    return core_run(s, n, m, b, sort_bytes, hs, ph);
}

int build(cudaStream_t s, const float* hb, int64_t n, int m, trace_bvh** out, PhaseTimer& ph) {
    const int64_t nn = 2 * n - 1;
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return LBVH_CUDA;
    Buffers b;
    if (b.alloc(n, sort_bytes, true, true)) return LBVH_CUDA;
    const int T = 256;
    ph.mark(s, nullptr);
    if (cudaMemcpyAsync(b.pb, hb, (size_t)n * 6 * sizeof(float), cudaMemcpyHostToDevice, s) != cudaSuccess) return LBVH_CUDA;
    ph.mark(s, "upload");
    Status hs;
    if (const int rc = build_core(s, n, m, b, sort_bytes, hs, ph)) return rc;
    const int64_t n_nodes = hs.root_size;
    lbvh_emit<<<blocks_for(nn, T), T, 0, s>>>(n, m, b.child, b.parent, b.first, b.count, b.axis, b.box, b.size, 0u, 0u, b.nodes);
    if (cudaGetLastError() != cudaSuccess) return LBVH_CUDA;
    ph.mark(s, "emit");
    trace_bvh_node* hn = nullptr;
    uint32_t* ho = nullptr;
    trace_bvh* bvh = bvh_alloc(n_nodes, n, &hn, &ho);
    if (!bvh) return 2;
    if (cudaMemcpyAsync(hn, b.nodes, (size_t)n_nodes * sizeof(trace_bvh_node), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaMemcpyAsync(ho, b.ids_sorted, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess) {
        trace_bvh_free(bvh);
        return LBVH_CUDA;
    }
    ph.mark(s, "download");
    if (cudaStreamSynchronize(s) != cudaSuccess) { trace_bvh_free(bvh); return LBVH_CUDA; }
    *out = bvh;
    return LBVH_OK;
}

// ------------------------------------------------------------------ the shadow tree (traverse.cuh, traverse_shadow)
// A primitive's box: Julia min / max over its three vertices (the refit's leaf rule, refit.cu).  A NaN coordinate makes
// the whole box NaN, so the centroid pass refuses the input.
__global__ void lbvh_prim_bounds(const float4* __restrict__ prims, int64_t n, float* __restrict__ pb) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 A = prims[3 * i], B = prims[3 * i + 1], C = prims[3 * i + 2];
    float lo[3] = {TR_INF, TR_INF, TR_INF}, hi[3] = {-TR_INF, -TR_INF, -TR_INF};
    tri_box(xyz(A), xyz(B), xyz(C), lo, hi);
    const bool nan = A.x != A.x || A.y != A.y || A.z != A.z || B.x != B.x || B.y != B.y || B.z != B.z || C.x != C.x ||
                     C.y != C.y || C.z != C.z;
    for (int c = 0; c < 3; ++c) {
        pb[6 * i + c] = nan ? NAN : lo[c];
        pb[6 * i + 3 + c] = nan ? NAN : hi[c];
    }
}

// One 64-byte pair record per internal node, in Karras numbering (the root is pair 0): both children's boxes, their
// references (a pair index, or TR_REF_LEAF | primitive slot for a leaf, traverse.cuh) and the split axis as
// a bit in the first half - the layout of the upload's pair records (api.cu).  Pair references are shifted by
// pair_shift, primitive slots by leaf_shift.
__global__ void lbvh_emit_pairs(int64_t n, const uint32_t* __restrict__ child, const uint32_t* __restrict__ sorted_ids,
                                const uint8_t* __restrict__ axis, const float* __restrict__ box, uint32_t pair_shift,
                                uint32_t leaf_shift, float4* __restrict__ pairs) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    for (int k = 0; k < 2; ++k) {
        const int64_t v = child[2 * i + k];
        const float* bx = box + 6 * v;
        const uint32_t ref = v < n - 1 ? pair_shift + (uint32_t)v : (TR_REF_LEAF | (leaf_shift + sorted_ids[v - (n - 1)]));
        const uint32_t extra = k == 0 ? (1u << axis[i]) : 0u;
        pairs[4 * i + 2 * k] = make_float4(bx[0], bx[1], bx[2], bx[3]);
        pairs[4 * i + 2 * k + 1] = make_float4(bx[4], bx[5], __uint_as_float(ref), __uint_as_float(extra));
    }
}

// ------------------------------------------------------------------ mesh builds (trace_scene_upload_mesh_device, upload_device.cu)
// The inputs a triangle array brings beyond its vertices: any NaN normal (bit 0) and any material index >= n_materials
// (bit 1) into the status block, which the build reads back before anything is emitted.
__global__ void lbvh_mesh_validate(const float* __restrict__ nrm, const uint32_t* __restrict__ mat, int64_t n,
                                   uint32_t n_materials, Status* st) {
    uint32_t bad = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (nrm)
            for (int k = 0; k < 9; ++k) { const float x = nrm[9 * i + k]; if (x != x) bad |= 1u; }
        if ((mat ? mat[i] : 0u) >= n_materials) bad |= 2u;
    }
    bad = __reduce_or_sync(0xFFFFFFFFu, bad);
    if ((threadIdx.x & 31) == 0 && bad) atomicOr(&st->bad, bad);
}

// A triangle's box from the [n][3][3] vertex array: the rule of lbvh_prim_bounds (a NaN vertex makes the box NaN)
__global__ void lbvh_tri_bounds(const float* __restrict__ v, int64_t n, float* __restrict__ pb) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = v + 9 * i;
    bool nan = false;
    for (int k = 0; k < 9; ++k) nan |= p[k] != p[k];
    float lo[3] = {TR_INF, TR_INF, TR_INF}, hi[3] = {-TR_INF, -TR_INF, -TR_INF};
    tri_box(f3(p[0], p[1], p[2]), f3(p[3], p[4], p[5]), f3(p[6], p[7], p[8]), lo, hi);
    for (int c = 0; c < 3; ++c) {
        pb[6 * i + c] = nan ? NAN : lo[c];
        pb[6 * i + 3 + c] = nan ? NAN : hi[c];
    }
}

}  // namespace

// Scratch of one LBVH build over n primitives (bounds, keys, sort, hierarchy, boxes) in a caller-owned allocation;
// 0 when CUB cannot size its sort.  The shadow tree's build of the same n fits the same bytes.
size_t lbvh_scratch_bytes(int64_t n, cudaStream_t s) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return 0;
    Buffers b;
    b.carve(n, sort_bytes, true, false);
    return b.k.used;
}

// The shadow tree of an uploaded scene (api.cu): an LBVH with one primitive per leaf over the n >= 2 uploaded primitive
// records `prims` (device, BVH slot order, triangles only), written as n - 1 pair records to `pairs` (device).  Nothing
// crosses to the host but the build's status.  `scratch` (lbvh_scratch_bytes(n)) or nullptr: an allocation of its own.
// Returns LBVH_OK, _NAN_BOUND (a NaN vertex), _TOO_DEEP or _CUDA; *depth (may be NULL): the tree's levels, root = 1.
// pair_shift and leaf_shift move the references: a tree whose pairs start at pair pair_shift and whose primitives
// start at slot leaf_shift of a larger one.
namespace {
// the shadow tree's bounds and core over `b`, no read-back
int shadow_enqueue(cudaStream_t s, const void* prims, int64_t n, Buffers& b, size_t sort_bytes) {
    lbvh_prim_bounds<<<blocks_for(n, 256), 256, 0, s>>>(static_cast<const float4*>(prims), n, b.pb);
    core_reset(s, n, b);
    PhaseTimer quiet;
    return core_enqueue(s, n, 1, b, sort_bytes, quiet);
}
// after the status `hs` is on the host: its verdict, and the pair records when it is LBVH_OK
int shadow_emit(cudaStream_t s, const Status& hs, int64_t n, Buffers& b, void* pairs, int* depth, uint32_t pair_shift,
                uint32_t leaf_shift) {
    if (const int rc = core_verdict(hs)) return rc;
    lbvh_emit_pairs<<<blocks_for(n - 1, 256), 256, 0, s>>>(n, b.child, b.ids_sorted, b.axis, b.box, pair_shift, leaf_shift,
                                                           static_cast<float4*>(pairs));
    if (cudaGetLastError() != cudaSuccess) return LBVH_CUDA;
    if (depth) *depth = (int)hs.root_depth;
    return LBVH_OK;
}
}  // namespace

int shadow_tree_build(cudaStream_t s, const void* prims, int64_t n, void* pairs, void* scratch, int* depth,
                      uint32_t pair_shift, uint32_t leaf_shift) {
    if (n < 2 || n >= 0x40000000ll) return 1;
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return LBVH_CUDA;
    Buffers b;
    if (scratch) b.borrow(scratch, n, sort_bytes);
    else if (b.alloc(n, sort_bytes, true, false)) return LBVH_CUDA;
    Status hs;
    if (shadow_enqueue(s, prims, n, b, sort_bytes) != LBVH_OK ||
        cudaMemcpyAsync(&hs, b.st, sizeof(Status), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess)
        return LBVH_CUDA;
    if (const int rc = shadow_emit(s, hs, n, b, pairs, depth, pair_shift, leaf_shift)) return rc;
    return cudaStreamSynchronize(s) == cudaSuccess ? LBVH_OK : LBVH_CUDA;
}

size_t lbvh_status_bytes() { return sizeof(Status); }

const void* lbvh_status(void* scratch, int64_t n) {
    Buffers b;
    b.borrow(scratch, n, 0);                               // (the status block sits before anything sized by the sort)
    return b.st;
}

int shadow_tree_enqueue(cudaStream_t s, const void* prims, int64_t n, void* scratch) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (n < 2 || !sort_bytes) return LBVH_CUDA;
    Buffers b;
    b.borrow(scratch, n, sort_bytes);
    return shadow_enqueue(s, prims, n, b, sort_bytes);
}

int shadow_tree_emit(cudaStream_t s, const void* status, int64_t n, void* scratch, void* pairs, int* depth,
                     uint32_t pair_shift, uint32_t leaf_shift) {
    Status hs;
    memcpy(&hs, status, sizeof(hs));
    Buffers b;
    b.borrow(scratch, n, sort_bytes_for(n, s));
    return shadow_emit(s, hs, n, b, pairs, depth, pair_shift, leaf_shift);
}

// The tree of trace_scene_upload_mesh_device over `scratch` (lbvh_scratch_bytes(n), n >= 1): the status block reset,
// normals (NULL: none) and material indices (NULL: all 0) checked into it, the triangles' boxes, then the LBVH core
// and its status read back.  Returns LBVH_OK with *n_nodes, *depth (may be NULL: the tree's levels) and *order = the
// sorted triangle ids (slot -> triangle, device, inside the scratch), or the first refusal in the order vertices,
// normals, materials, depth.  Nothing is written outside the scratch before lbvh_mesh_emit (the preorder node records
// into `nodes`, device), so a refused input leaves the caller's buffers intact.
int lbvh_mesh_enqueue(cudaStream_t s, const float* v, const float* nrm, const uint32_t* mat, int64_t n_materials, int64_t n,
                      int m, void* scratch, PhaseTimer& ph) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return LBVH_CUDA;
    Buffers b;
    b.borrow(scratch, n, sort_bytes);
    core_reset(s, n, b);
    const int T = 256;
    const uint32_t nm = n_materials > 0xFFFFFFFFll ? 0xFFFFFFFFu : (uint32_t)n_materials;
    lbvh_mesh_validate<<<(unsigned)std::min<int64_t>(blocks_for(n, T), 4096), T, 0, s>>>(nrm, mat, n, nm, b.st);
    ph.mark(s, "validate");
    lbvh_tri_bounds<<<blocks_for(n, T), T, 0, s>>>(v, n, b.pb);
    ph.mark(s, "bounds");
    PhaseTimer quiet;                                      // the core's own phases are not the upload's
    const int rc = core_enqueue(s, n, m, b, sort_bytes, quiet);   // (its launch check covers the two kernels above)
    ph.mark(s, "build");
    return rc;
}

int lbvh_mesh_result(const void* status, void* scratch, int64_t n, int64_t* n_nodes, const uint32_t** order, int* depth) {
    Status hs;
    memcpy(&hs, status, sizeof(hs));
    if (hs.nan) return LBVH_NAN_BOUND;
    if (hs.bad & 1u) return LBVH_NAN_NORMAL;
    if (hs.bad & 2u) return LBVH_BAD_MATERIAL;
    if (const int rc = core_verdict(hs)) return rc;
    Buffers b;
    b.borrow(scratch, n, 0);                               // (ids_sorted sits before the sort's temp)
    *n_nodes = hs.root_size;
    *order = b.ids_sorted;
    if (depth) *depth = (int)hs.root_depth;
    return LBVH_OK;
}

int lbvh_mesh_build(cudaStream_t s, const float* v, const float* nrm, const uint32_t* mat, int64_t n_materials, int64_t n,
                    int m, void* scratch, PhaseTimer& ph, int64_t* n_nodes, const uint32_t** order, int* depth) {
    if (lbvh_mesh_enqueue(s, v, nrm, mat, n_materials, n, m, scratch, ph) != LBVH_OK) return LBVH_CUDA;
    std::vector<char> hs(lbvh_status_bytes());
    if (cudaMemcpyAsync(hs.data(), lbvh_status(scratch, n), hs.size(), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
        cudaStreamSynchronize(s) != cudaSuccess)
        return LBVH_CUDA;
    return lbvh_mesh_result(hs.data(), scratch, n, n_nodes, order, depth);
}

int lbvh_mesh_emit(cudaStream_t s, int64_t n, int m, void* scratch, void* nodes, uint32_t node_shift, uint32_t prim_shift) {
    const size_t sort_bytes = sort_bytes_for(n, s);
    if (!sort_bytes) return LBVH_CUDA;
    Buffers b;
    b.borrow(scratch, n, sort_bytes);
    const int T = 256;
    lbvh_emit<<<blocks_for(2 * n - 1, T), T, 0, s>>>(n, m, b.child, b.parent, b.first, b.count, b.axis, b.box, b.size,
                                                    node_shift, prim_shift, static_cast<trace_bvh_node*>(nodes));
    return cudaGetLastError() == cudaSuccess ? LBVH_OK : LBVH_CUDA;
}

extern "C" int trace_bvh_build_gpu(int device, const float* pb, int64_t n, int max_node_primitives, trace_bvh** out) {
    if (!out || n < 0 || (n > 0 && !pb)) return 1;
    *out = nullptr;
    if (n >= 0x40000000ll) return 1;
    const int m = max_node_primitives < 1 ? 1 : (max_node_primitives < 255 ? max_node_primitives : 255);
    int n_dev = 0, prev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || device < 0 || device >= n_dev || cudaGetDevice(&prev) != cudaSuccess) {
        cudaGetLastError();
        return LBVH_CUDA;                                    // no CPU fallback
    }
    if (n == 0) {
        trace_bvh_node* hn; uint32_t* ho;
        *out = bvh_alloc(0, 0, &hn, &ho);
        return *out ? 0 : 2;
    }
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return LBVH_CUDA; }
    cudaStream_t s;
    int rc = LBVH_CUDA;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) == cudaSuccess) {
        PhaseTimer ph;
        ph.on = getenv("TRACE_BVH_PROFILE") != nullptr;
        const auto t0 = std::chrono::steady_clock::now();
        rc = build(s, pb, n, m, out, ph);
        if (ph.on && rc == LBVH_OK) {
            char head[96];
            snprintf(head, sizeof(head), "bvh build gpu: n %lld, device %d", (long long)n, device);
            ph.print(head, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
        }
        cudaStreamDestroy(s);
    }
    cudaGetLastError();
    cudaSetDevice(prev);
    return rc;
}
