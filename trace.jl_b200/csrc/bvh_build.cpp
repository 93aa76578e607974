// bvh_build.cpp — host-side BVH build of libtrace_cuda.so (trace_bvh_build, include/trace_cuda.h).
//
// north_star: "The BVH is built on the host with the reference's SAH split logic, then flattened into a
// 32-byte-aligned LinearBVH node array".  The split logic is the reference's, quirks included
// (src/accel/bvh.jl:87-185, src/Trace.jl:128-137; SURVEY.md §9 Q16): 12 buckets that start as the point (0,0,0),
// a cost that weighs each side by its NUMBER OF BUCKETS, a partition that never tests the first element and splits
// [from..mid] | [mid+1..to], two-primitive nodes split at the smaller centroid, zero-primitive leaves kept.
// Unlike the reference's recursive, allocation-per-node build this one is iterative: SoA bounds/centroids, one index
// permutation that is partitioned in place, and nodes emitted directly in the flattened preorder (first child =
// parent + 1), so building the 10 M-triangle scene needs no recursion and no per-node heap traffic.  It is also
// multi-threaded (std::thread; TRACE_BVH_THREADS overrides the thread count): the passes over large nodes run in
// parallel and subtrees below 65 536 primitives are independent jobs - with the one-threaded result bit for bit.
// Compiled with -ffp-contract=off: the cost arithmetic must round like the reference's.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <memory>
#include <cstdlib>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/trace_cuda.h"

// (a std::vector would zero-fill 640 MB single-threaded for the 10 M-triangle tree before the parallel stitch writes it)
template <class T>
struct RawArray {
    std::unique_ptr<T[]> p;
    size_t n = 0;
    void resize(size_t m) { p.reset(new T[m]); n = m; }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    T* data() const { return p.get(); }
    T& operator[](size_t i) const { return p[i]; }
};
struct trace_bvh {
    RawArray<trace_bvh_node> nodes;
    RawArray<uint32_t> order;
};

namespace {

const float kInf = std::numeric_limits<float>::infinity();

// Julia's min/max on floats: NaN propagates, -0.0 orders below +0.0.
// Branch-free on x86 (the min / max passes are the build's inner loops): MINSS returns its SECOND operand when the two
// compare equal or unordered, so min(a, b) | min(b, a) is the smaller value when they differ, -0.0 for a +-0 tie (sign
// bits OR-ed) and a NaN when either is NaN (all-ones exponent, non-zero mantissa survive the OR); max(a, b) =
// -min(-a, -b) (sign flips are exact).
#if defined(__SSE2__)
inline float fmin_jl(float a, float b) {
    const __m128 x = _mm_set_ss(a), y = _mm_set_ss(b);
    return _mm_cvtss_f32(_mm_or_ps(_mm_min_ss(x, y), _mm_min_ss(y, x)));
}
inline float fmax_jl(float a, float b) { return -fmin_jl(-a, -b); }
#else
inline float fmin_jl(float a, float b) {
    if (a != a || b != b) return a + b;
    if (b < a) return b;
    if (a == b && std::signbit(b)) return b;
    return a;
}
inline float fmax_jl(float a, float b) {
    if (a != a || b != b) return a + b;
    if (b > a) return b;
    if (a == b && !std::signbit(b)) return b;
    return a;
}
#endif

struct Box {
    float lo[3], hi[3];
    void reset() { for (int k = 0; k < 3; ++k) { lo[k] = kInf; hi[k] = -kInf; } }
    void point(float v) { for (int k = 0; k < 3; ++k) { lo[k] = v; hi[k] = v; } }
    void grow(const float* l, const float* h) {
        for (int k = 0; k < 3; ++k) { lo[k] = fmin_jl(lo[k], l[k]); hi[k] = fmax_jl(hi[k], h[k]); }
    }
    void grow(const Box& b) { grow(b.lo, b.hi); }
    float area() const {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        return 2.0f * ((dx * dy + dx * dz) + dy * dz);
    }
    bool valid() const {
        for (int k = 0; k < 3; ++k) if (lo[k] == kInf || hi[k] == -kInf) return false;
        return true;
    }
    int widest() const {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (dx > dy && dx > dz) return 0;
        if (dy > dz) return 1;
        return 2;
    }
};

// ------------------------------------------------------------------ parallel helpers
// A fork-join over [0, n) in `parts` contiguous chunks.  The build runs a few thousand of these, so the workers are a
// persistent pool (one per process, grown on demand) woken through a condition variable, not threads spawned per call.
class ChunkPool {
  public:
    static ChunkPool& get() { static ChunkPool p; return p; }
    template <class F>
    void run(int64_t n, int parts, F f) {
        if (parts <= 1 || n < 2) { f(0, (int64_t)0, n); return; }
        std::unique_lock<std::mutex> entry(entry_mutex_);            // one fork-join at a time (builds may come from several host threads)
        grow(parts - 1);
        std::function<void(int)> job = [&](int p) { f(p, n * p / parts, n * (p + 1) / parts); };
        {
            std::lock_guard<std::mutex> lk(m_);
            job_ = &job; parts_ = parts; next_ = 1; pending_ = parts - 1; ++epoch_;
        }
        cv_.notify_all();
        f(0, (int64_t)0, n / parts);
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [&] { return pending_ == 0; });
        job_ = nullptr;
    }
    ~ChunkPool() {
        { std::lock_guard<std::mutex> lk(m_); stop_ = true; ++epoch_; }
        cv_.notify_all();
        for (auto& t : workers_) t.join();
    }
  private:
    void grow(int n) {
        while ((int)workers_.size() < n) workers_.emplace_back([this] { loop(); });
    }
    void loop() {
        for (;;) {
            std::unique_lock<std::mutex> lk(m_);
            cv_.wait(lk, [&] { return stop_ || (job_ != nullptr && next_ < parts_); });
            if (stop_) return;
            while (job_ != nullptr && next_ < parts_) {
                const int p = next_++;
                const std::function<void(int)>* job = job_;
                lk.unlock();
                (*job)(p);
                lk.lock();
                if (--pending_ == 0) done_.notify_all();
            }
        }
    }
    std::mutex entry_mutex_, m_;
    std::condition_variable cv_, done_;
    std::vector<std::thread> workers_;
    const std::function<void(int)>* job_ = nullptr;
    int parts_ = 0, next_ = 0, pending_ = 0;
    uint64_t epoch_ = 0;
    bool stop_ = false;
};
template <class F>
void parallel_chunks(int64_t n, int parts, F f) { ChunkPool::get().run(n, parts, f); }

int build_threads() {
    const char* e = getenv("TRACE_BVH_THREADS");
    int t = e ? atoi(e) : (int)std::thread::hardware_concurrency();
    return t < 1 ? 1 : (t > 64 ? 64 : t);
}

// Nodes with more primitives than this are split in the sequential "top" phase with their O(count) passes run in
// parallel; smaller ones become independent subtree jobs for the thread pool.
const int64_t kTopThreshold = 1 << 16;      // upper bound; build_tree lowers it for small inputs so that every thread gets jobs

struct Split { bool leaf; int axis; int64_t mid; trace_bvh_node node; };

// One primitive of the build: world bounds, centroid (bounds.jl: 0.5 lo + 0.5 hi) and its original index, 40 bytes.  The
// build permutes these RECORDS, not an index array: every pass over a node's range then streams contiguous memory (a
// subtree's working set is its own slice) instead of gathering 36 bytes per primitive from all over the input arrays -
// the gathers were ~80 % of the build time at 10 M triangles.
struct Rec { float b[6]; float c[3]; uint32_t id; };

// ---- the reference's split of perm[from..to] (src/accel/bvh.jl:87-185; quirks Q16).  `threads` > 1 runs the reductions
// and the bucket evaluation in parallel: min / max reductions are exact and order-independent, and the partition's
// swaps (whose ORDER defines the resulting permutation) stay sequential, so the tree is bit-identical to the
// one-threaded build.
// bounds of the primitives and of their centroids over rec[from .. from + count)
static void range_bounds(const Rec* rec, int64_t from, int64_t count, int parts, Box& all, Box& cb) {
    if (parts == 1) {
        all.reset(); cb.reset();
        for (int64_t i = from; i < from + count; ++i) { all.grow(rec[i].b, rec[i].b + 3); cb.grow(rec[i].c, rec[i].c); }
        return;
    }
    std::vector<Box> pa((size_t)parts), pc((size_t)parts);
    parallel_chunks(count, parts, [&](int p, int64_t b, int64_t e) {
        Box a, c; a.reset(); c.reset();
        for (int64_t i = from + b; i < from + e; ++i) { a.grow(rec[i].b, rec[i].b + 3); c.grow(rec[i].c, rec[i].c); }
        pa[(size_t)p] = a; pc[(size_t)p] = c;
    });
    all = pa[0]; cb = pc[0];
    for (int p = 1; p < parts; ++p) { all.grow(pa[(size_t)p]); cb.grow(pc[(size_t)p]); }
}

// Top-phase plumbing of a split (large nodes, passes run in parallel): the node's records are read from `src`; when the
// node is partitioned they are written - already permuted - into `dst` (the other one of the two record buffers), so no
// copy-back pass is needed, and the pass that moves them also accumulates the two children's boxes, which the children
// then take instead of a bounds pass of their own (min / max are exact and order-independent: same bits).
struct TopIO {
    const Rec* src; Rec* dst;
    const Box* pre_all; const Box* pre_cb;      // this node's boxes when the parent computed them (else null)
    bool moved = false;                          // the children's records live in dst
    Box child_all[2], child_cb[2];               // valid when moved
};

struct LiteralSplitter {
    static const bool kPingPong = true;
    Rec* rec; int max_prims;
    std::vector<uint8_t>* pred;        // scratch of the top phase (n entries each)
    uint32_t* idx; Rec* tmp;
    static const int NB = 12;

    Split operator()(int64_t from, int64_t to, int threads, TopIO* io = nullptr) const {
        Split r; r.leaf = false; r.axis = 0; r.mid = from;
        const int64_t count = to - from + 1;
        const int parts = (threads > 1 && count >= 32768) ? threads : 1;
        Rec* const rec = io ? const_cast<Rec*>(io->src) : this->rec;      // (shadows the member: the node's records)
        Box all, cb;
        if (io && io->pre_all) { all = *io->pre_all; cb = *io->pre_cb; }
        else range_bounds(rec, from, count, parts, all, cb);
        for (int k = 0; k < 3; ++k) { r.node.bmin[k] = all.lo[k]; r.node.bmax[k] = all.hi[k]; }
        if (count == 1) { r.leaf = true; return r; }
        const int axis = cb.widest();
        r.axis = axis;
        if (!cb.valid() || cb.lo[axis] == cb.hi[axis]) { r.leaf = true; return r; }
        // relative position of a centroid along `axis`, bounds.jl:134-143 (offset)
        const bool any_extent = cb.hi[0] > cb.lo[0] || cb.hi[1] > cb.lo[1] || cb.hi[2] > cb.lo[2];
        const float extent = cb.hi[axis] > cb.lo[axis] ? cb.hi[axis] - cb.lo[axis] : 1.0f;
        auto bucket = [&](const Rec& pr) -> int {
            float o = pr.c[axis] - cb.lo[axis];
            if (any_extent) o = o / extent;
            int b = (int)std::floor(12.0f * o);
            return b == NB ? NB - 1 : b;
        };
        if (count <= 2) {
            // partialsort!(view, 1, by = centroid[axis]) on two entries; mid = (from + to) ÷ 2 = from
            if (rec[to].c[axis] < rec[from].c[axis]) std::swap(rec[from], rec[to]);
            r.mid = (from + to) / 2;
            return r;
        }
        Box bk[NB];
        if (parts == 1) {
            Box acc[NB];
            for (int k = 0; k < NB; ++k) acc[k].reset();
            for (int64_t i = from; i <= to; ++i) acc[bucket(rec[i])].grow(rec[i].b, rec[i].b + 3);
            for (int k = 0; k < NB; ++k) { bk[k].point(0.0f); bk[k].grow(acc[k]); }
        } else {
            std::vector<Box> pbk((size_t)parts * NB);
            uint8_t* bkt = pred->data();                              // the partition below reuses the bucket numbers
            parallel_chunks(count, parts, [&](int p, int64_t b, int64_t e) {
                Box* acc = &pbk[(size_t)p * NB];
                for (int k = 0; k < NB; ++k) acc[k].reset();
                for (int64_t i = from + b; i < from + e; ++i) {
                    const int k = bucket(rec[i]);
                    acc[k].grow(rec[i].b, rec[i].b + 3);
                    bkt[i] = (uint8_t)k; idx[i] = (uint32_t)i;
                }
            });
            for (int k = 0; k < NB; ++k) { bk[k].point(0.0f); for (int p = 0; p < parts; ++p) bk[k].grow(pbk[(size_t)p * NB + k]); }
        }
        // prefix unions 0..i and suffix unions i..10 (bucket 11 never enters the right-hand side)
        Box pre[NB], suf[NB];
        pre[0] = bk[0];
        for (int k = 1; k < NB; ++k) { pre[k] = pre[k - 1]; pre[k].grow(bk[k]); }
        // the reference folds the right side left-to-right starting at bucket i+1; min/max are exact, so a suffix scan
        // yields the same box
        suf[NB - 2] = bk[NB - 2];
        for (int k = NB - 3; k >= 0; --k) { suf[k] = bk[k]; suf[k].grow(suf[k + 1]); }
        const float total_area = all.area();
        int best = 0;
        float best_cost = 0.0f;
        bool best_nan = false;
        for (int i = 0; i < NB - 1; ++i) {            // split after bucket i (0-based)
            float left = (float)(i + 1) * pre[i].area();
            float right = 0.0f;
            const int n_right = (NB - 1) - (i + 1);
            if (n_right > 0) right = (float)n_right * suf[i + 1].area();
            const float cost = 1.0f + (left + right) / total_area;
            if (i == 0) { best = 0; best_cost = cost; best_nan = cost != cost; }
            else if (!best_nan && (cost != cost || cost < best_cost)) { best = i; best_cost = cost; best_nan = cost != cost; }
        }
        if (!(count > max_prims || (double)best_cost < (double)count)) { r.leaf = true; return r; }
        // partition!, Trace.jl:128-137 (never tests the first element)
        int64_t left = from;
        if (parts > 1) {
            uint8_t* pr = pred->data();
            // The swaps' ORDER defines the permutation, so that loop stays sequential - but it runs on 4-byte positions
            // (branch-free), and the 40-byte records are moved afterwards, in parallel.  `left != i` only ever skips
            // i == from (left < i from then on).
            for (int64_t i = from + 1; i <= to; ++i) {
                const uint32_t p = (int)pr[i] <= best ? 1u : 0u, a = idx[i], b = idx[left];
                idx[i] = p ? b : a;
                idx[left] = p ? a : b;
                left += p;
            }
            if (io) {
                // one pass: permuted records into the other buffer + the children's boxes ([from, left] and (left, to])
                Rec* const dst = io->dst;
                std::vector<Box> pb((size_t)parts * 4);
                parallel_chunks(count, parts, [&](int p, int64_t b, int64_t e) {
                    Box* acc = &pb[(size_t)p * 4];
                    for (int k = 0; k < 4; ++k) acc[k].reset();
                    for (int64_t i = from + b; i < from + e; ++i) {
                        const Rec v = rec[idx[i]];
                        dst[i] = v;
                        const int side = i <= left ? 0 : 1;
                        acc[2 * side].grow(v.b, v.b + 3);
                        acc[2 * side + 1].grow(v.c, v.c);
                    }
                });
                for (int side = 0; side < 2; ++side) {
                    io->child_all[side] = pb[(size_t)2 * side]; io->child_cb[side] = pb[(size_t)2 * side + 1];
                    for (int p = 1; p < parts; ++p) { io->child_all[side].grow(pb[(size_t)p * 4 + 2 * side]); io->child_cb[side].grow(pb[(size_t)p * 4 + 2 * side + 1]); }
                }
                io->moved = true;
            } else {
                parallel_chunks(count, parts, [&](int, int64_t b, int64_t e) {
                    for (int64_t i = from + b; i < from + e; ++i) tmp[i] = rec[idx[i]];
                });
                parallel_chunks(count, parts, [&](int, int64_t b, int64_t e) {
                    memcpy(rec + from + b, tmp + from + b, (size_t)(e - b) * sizeof(Rec));
                });
            }
        } else {
            for (int64_t i = from; i <= to; ++i)
                if (left != i && bucket(rec[i]) <= best) { std::swap(rec[i], rec[left]); ++left; }
        }
        r.mid = left;
        return r;
    }
};

// ---- opt-in conventional binned SAH (SURVEY.md §8f.2): buckets start EMPTY, each side is weighted by its primitive
// COUNT (cost = 1/8 + (nL*aL + nR*aR)/A), a node becomes a leaf when that is cheaper and it holds <=
// max_node_primitives, the partition tests every element, and a degenerate split falls back to the median.
struct SahSplitter {
    static const bool kPingPong = false;
    Rec* rec; int max_prims;
    std::vector<uint8_t>* pred;
    uint32_t* idx; Rec* tmp;
    static const int NB = 16;

    Split operator()(int64_t from, int64_t to, int threads, TopIO* = nullptr) const {
        Split r; r.leaf = false; r.axis = 0;
        const int64_t count = to - from + 1;
        const int parts = (threads > 1 && count >= 32768) ? threads : 1;
        Box all, cb;
        range_bounds(rec, from, count, parts, all, cb);
        for (int k = 0; k < 3; ++k) { r.node.bmin[k] = all.lo[k]; r.node.bmax[k] = all.hi[k]; }
        const int axis = cb.widest();
        r.axis = axis;
        bool leaf = count == 1 || !cb.valid() || !(cb.hi[axis] > cb.lo[axis]);
        if (leaf && count > max_prims && count > 1) leaf = false;        // identical centroids: split at the median
        int64_t mid = (from + to) / 2;                                     // last index of the left side
        if (!leaf) {
            bool split_done = false;
            if (cb.valid() && cb.hi[axis] > cb.lo[axis] && count >= 2) {
                const float scale = (float)NB / (cb.hi[axis] - cb.lo[axis]);
                auto bucket = [&](const Rec& pr) -> int {
                    int b = (int)((pr.c[axis] - cb.lo[axis]) * scale);
                    return b < 0 ? 0 : (b >= NB ? NB - 1 : b);
                };
                std::vector<Box> pbk((size_t)parts * NB);
                std::vector<int64_t> pcnt((size_t)parts * NB, 0);
                parallel_chunks(count, parts, [&](int p, int64_t b, int64_t e) {
                    Box* bk = &pbk[(size_t)p * NB];
                    int64_t* cn = &pcnt[(size_t)p * NB];
                    for (int k = 0; k < NB; ++k) bk[k].reset();
                    for (int64_t i = from + b; i < from + e; ++i) {
                        const int k = bucket(rec[i]);
                        bk[k].grow(rec[i].b, rec[i].b + 3); cn[k]++;
                    }
                });
                Box bk[NB];
                int64_t cnt[NB];
                for (int k = 0; k < NB; ++k) {
                    bk[k].reset(); cnt[k] = 0;
                    for (int p = 0; p < parts; ++p) { if (pcnt[(size_t)p * NB + k]) bk[k].grow(pbk[(size_t)p * NB + k]); cnt[k] += pcnt[(size_t)p * NB + k]; }
                }
                float right_area[NB];
                int64_t right_cnt[NB];
                Box acc; acc.reset();
                int64_t c = 0;
                for (int k = NB - 1; k >= 1; --k) {
                    if (cnt[k]) acc.grow(bk[k]);
                    c += cnt[k];
                    right_area[k] = c ? acc.area() : 0.0f; right_cnt[k] = c;
                }
                acc.reset(); c = 0;
                const float total_area = all.area();
                float best_cost = kInf;
                int best = -1;
                for (int k = 0; k < NB - 1; ++k) {                          // split after bucket k
                    if (cnt[k]) acc.grow(bk[k]);
                    c += cnt[k];
                    if (c == 0 || right_cnt[k + 1] == 0) continue;
                    const float cost = 0.125f + ((float)c * acc.area() + (float)right_cnt[k + 1] * right_area[k + 1]) /
                                                    (total_area > 0.0f ? total_area : 1.0f);
                    if (cost < best_cost) { best_cost = cost; best = k; }
                }
                if (best >= 0 && (count > max_prims || best_cost < (float)count)) {
                    int64_t left = from;
                    for (int64_t i = from; i <= to; ++i)
                        if (bucket(rec[i]) <= best) { std::swap(rec[i], rec[left]); ++left; }
                    mid = left - 1;
                    split_done = mid >= from && mid < to;
                } else if (best >= 0 || count <= max_prims) {
                    leaf = count <= max_prims;
                }
            }
            if (!leaf && !split_done) {
                // median split along the axis (also: two primitives, or all centroids in one bucket)
                mid = (from + to) / 2;
                std::nth_element(rec + from, rec + mid, rec + to + 1, [&](const Rec& a, const Rec& b) { return a.c[axis] < b.c[axis]; });
            }
        }
        r.leaf = leaf; r.mid = mid;
        return r;
    }
};

struct Task { int64_t from, to; int64_t patch; };   // inclusive range into the permutation; node whose `offset` we are

struct LocalTree { std::vector<trace_bvh_node> nodes; std::vector<uint32_t> order; };

// sequential build of perm[from..to] into `out` with LOCAL indices (node 0 = the subtree's root, order starts at 0), nodes
// emitted in the flattened preorder (first child = parent + 1)
template <class Splitter>
int build_subtree(const Splitter& split, const Rec* rec, int64_t from, int64_t to, LocalTree& out) {
    std::vector<Task> todo;
    todo.push_back({from, to, -1});
    const int64_t node_limit = 8 * (to - from + 1) + 1024;     // a guard, never reached by terminating inputs
    while (!todo.empty()) {
        const Task t = todo.back();
        todo.pop_back();
        const int64_t slot = (int64_t)out.nodes.size();
        if (slot > node_limit) return 3;
        if (t.patch >= 0) out.nodes[(size_t)t.patch].offset = (uint32_t)slot;
        Split s = split(t.from, t.to, 1);
        const int64_t count = t.to - t.from + 1;
        if (s.leaf) {
            s.node.offset = (uint32_t)out.order.size();
            s.node.meta = TRACE_NODE_LEAF | (uint32_t)(count < 0 ? 0 : count);
            for (int64_t i = t.from; i <= t.to; ++i) out.order.push_back(rec[i].id);
            out.nodes.push_back(s.node);
        } else {
            s.node.offset = 0;
            s.node.meta = (uint32_t)s.axis << 30;
            out.nodes.push_back(s.node);
            todo.push_back({s.mid + 1, t.to, slot});     // second child: patched into `offset` when it is emitted
            todo.push_back({t.from, s.mid, -1});          // first child: emitted next, at slot + 1
        }
    }
    return 0;
}

// Whole build: (1) the top of the tree sequentially in preorder, each large node's passes in parallel; nodes below
// kTopThreshold primitives are set aside as jobs; (2) the jobs in parallel (disjoint ranges of the permutation);
// (3) stitch: item sizes -> preorder slots by a prefix sum, local indices rebased.  The result is the array the
// one-threaded build produces, bit for bit (tests/test_bvh_build.py compares them).
static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

template <class Splitter>
int build_tree(Splitter split, const Rec* rec, int64_t n, trace_bvh* bvh) {
    const int threads = build_threads();
    const bool prof = getenv("TRACE_BVH_PROFILE") != nullptr;
    const double t_begin = now_s();
    // ~16 jobs per thread (subtree sizes vary a lot: the literal tree is unbalanced), never below 4096 primitives
    const int64_t job_threshold = std::max<int64_t>(4096, std::min<int64_t>(kTopThreshold, n / (16 * (int64_t)threads)));
    struct Item { int kind; trace_bvh_node node; int64_t from, to; int64_t second_item; int job; const Rec* base; };   // kind 0 interior, 1 leaf, 2 job
    std::vector<Item> items;
    struct Job { int64_t from, to; Rec* base; };
    std::vector<Job> jobs;
    // `base`: which of the two record buffers holds the task's range (a partitioned top-phase node writes its children
    // into the other one); `boxes`: the parent computed this node's boxes while moving the records
    struct TopTask { int64_t from, to; int64_t patch_item; Rec* base; bool boxes; Box all, cb; };
    std::vector<TopTask> todo;
    Rec* const buf0 = const_cast<Rec*>(rec);
    Rec* const buf1 = split.tmp;
    { TopTask root; root.from = 0; root.to = n - 1; root.patch_item = -1; root.base = buf0; root.boxes = false; todo.push_back(root); }
    while (!todo.empty()) {
        const TopTask t = todo.back();
        todo.pop_back();
        const int64_t me = (int64_t)items.size();
        if (t.patch_item >= 0) items[(size_t)t.patch_item].second_item = me;
        const int64_t count = t.to - t.from + 1;
        if (threads == 1 ? false : count <= job_threshold) {
            items.push_back({2, trace_bvh_node(), t.from, t.to, -1, (int)jobs.size(), t.base});
            jobs.push_back({t.from, t.to, t.base});
            continue;
        }
        if (threads == 1 && me == 0) {          // one thread: the plain sequential build of the whole range
            items.push_back({2, trace_bvh_node(), t.from, t.to, -1, 0, t.base});
            jobs.push_back({t.from, t.to, t.base});
            continue;
        }
        TopIO io;
        io.src = t.base; io.dst = t.base == buf0 ? buf1 : buf0;
        io.pre_all = t.boxes ? &t.all : nullptr; io.pre_cb = t.boxes ? &t.cb : nullptr;
        const bool ping_pong = Splitter::kPingPong && buf1 != nullptr;
        Split s = split(t.from, t.to, threads, ping_pong ? &io : nullptr);
        if (s.leaf) {
            s.node.meta = TRACE_NODE_LEAF | (uint32_t)count;
            items.push_back({1, s.node, t.from, t.to, -1, -1, t.base});
        } else {
            s.node.meta = (uint32_t)s.axis << 30;
            items.push_back({0, s.node, t.from, t.to, -1, -1, t.base});
            const bool moved = ping_pong && io.moved;
            Rec* const child_base = moved ? io.dst : t.base;
            TopTask second, first;
            second.from = s.mid + 1; second.to = t.to; second.patch_item = me; second.base = child_base; second.boxes = moved;
            first.from = t.from; first.to = s.mid; first.patch_item = -1; first.base = child_base; first.boxes = moved;
            if (moved) { first.all = io.child_all[0]; first.cb = io.child_cb[0]; second.all = io.child_all[1]; second.cb = io.child_cb[1]; }
            todo.push_back(second);
            todo.push_back(first);
        }
    }
    const double t_top = now_s();
    std::vector<LocalTree> local(jobs.size());
    std::vector<int> rcs(jobs.size(), 0);
    {
        std::atomic<size_t> next(0);
        auto worker = [&]() {
            for (;;) {
                const size_t j = next.fetch_add(1);
                if (j >= jobs.size()) break;
                const int64_t cnt = jobs[j].to - jobs[j].from + 1;
                local[j].nodes.reserve((size_t)(2 * cnt + 16));
                local[j].order.reserve((size_t)cnt);
                Splitter mine = split;                       // the job's records may live in either buffer
                mine.rec = jobs[j].base;
                rcs[j] = build_subtree(mine, jobs[j].base, jobs[j].from, jobs[j].to, local[j]);
            }
        };
        const int nt = (int)std::min<size_t>((size_t)threads, std::max<size_t>(1, jobs.size()));
        std::vector<std::thread> th;
        for (int k = 1; k < nt; ++k) th.emplace_back(worker);
        worker();
        for (auto& t : th) t.join();
    }
    for (int rc : rcs) if (rc) return rc;
    const double t_jobs = now_s();
    // stitch
    std::vector<int64_t> node_base(items.size() + 1, 0), order_base(items.size() + 1, 0);
    for (size_t i = 0; i < items.size(); ++i) {
        const Item& it = items[i];
        node_base[i + 1] = node_base[i] + (it.kind == 2 ? (int64_t)local[(size_t)it.job].nodes.size() : 1);
        order_base[i + 1] = order_base[i] + (it.kind == 2 ? (int64_t)local[(size_t)it.job].order.size() : (it.kind == 1 ? it.to - it.from + 1 : 0));
    }
    if (node_base.back() > 0x7fffffffll) return 4;
    bvh->nodes.resize((size_t)node_base.back());
    bvh->order.resize((size_t)order_base.back());
    parallel_chunks((int64_t)items.size(), threads, [&](int, int64_t b, int64_t e) {
        for (int64_t i = b; i < e; ++i) {
            const Item& it = items[(size_t)i];
            if (it.kind == 0) {
                trace_bvh_node nd = it.node;
                nd.offset = (uint32_t)node_base[(size_t)it.second_item];
                bvh->nodes[(size_t)node_base[(size_t)i]] = nd;
            } else if (it.kind == 1) {
                trace_bvh_node nd = it.node;
                nd.offset = (uint32_t)order_base[(size_t)i];
                bvh->nodes[(size_t)node_base[(size_t)i]] = nd;
                for (int64_t k = it.from; k <= it.to; ++k) bvh->order[(size_t)(order_base[(size_t)i] + k - it.from)] = it.base[k].id;
            } else {
                const LocalTree& lt = local[(size_t)it.job];
                const uint32_t nb = (uint32_t)node_base[(size_t)i], ob = (uint32_t)order_base[(size_t)i];
                for (size_t k = 0; k < lt.nodes.size(); ++k) {
                    trace_bvh_node nd = lt.nodes[k];
                    nd.offset += (nd.meta >> 30) == 3 ? ob : nb;
                    bvh->nodes[(size_t)nb + k] = nd;
                }
                if (!lt.order.empty()) memcpy(&bvh->order[(size_t)ob], lt.order.data(), lt.order.size() * sizeof(uint32_t));
            }
        }
    });
    if (prof) fprintf(stderr, "bvh build: %d threads, top phase %.2f s (%zu items, %zu jobs), jobs %.2f s, stitch %.2f s\n", threads, t_top - t_begin,
                      items.size(), jobs.size(), t_jobs - t_top, now_s() - t_jobs);
    return 0;
}

template <class Splitter>
int build_entry(const float* pb, int64_t n, int max_prims, trace_bvh** out) {
    if (!out || n < 0 || (n > 0 && !pb)) return 1;
    *out = nullptr;
    if (n >= 0x40000000ll) return 1;
    trace_bvh* bvh = new (std::nothrow) trace_bvh();
    if (!bvh) return 2;
    if (n == 0) { *out = bvh; return 0; }
    try {
        std::unique_ptr<Rec[]> rec(new Rec[(size_t)n]);          // (no value-initialisation pass: filled in parallel below)
        std::vector<uint8_t> pred((size_t)n);
        const bool top_phase = build_threads() > 1 && n > 4096;      // scratch of the parallel partition
        std::unique_ptr<uint32_t[]> idx(top_phase ? new uint32_t[(size_t)n] : nullptr);
        std::unique_ptr<Rec[]> tmp(top_phase ? new Rec[(size_t)n] : nullptr);
        std::atomic<int> bad(0);
        parallel_chunks(n, build_threads(), [&](int, int64_t b, int64_t e) {
            for (int64_t i = b; i < e; ++i) {
                Rec& r = rec[(size_t)i];
                r.id = (uint32_t)i;
                for (int k = 0; k < 6; ++k) r.b[k] = pb[6 * i + k];
                for (int k = 0; k < 3; ++k) {
                    r.c[k] = 0.5f * pb[6 * i + k] + 0.5f * pb[6 * i + 3 + k];
                    if (r.c[k] != r.c[k]) bad.store(1, std::memory_order_relaxed);
                }
            }
        });
        // a NaN centroid has no bucket: the reference's Int64(floor(NaN)) throws an InexactError (bvh.jl:118); refuse the input
        if (bad.load()) { delete bvh; return 5; }
        Splitter split{rec.get(), max_prims, &pred, idx.get(), tmp.get()};
        const int rc = build_tree(split, rec.get(), n, bvh);
        if (rc) { delete bvh; return rc; }
    } catch (...) { delete bvh; return 2; }
    *out = bvh;
    return 0;
}

}  // namespace

extern "C" int trace_bvh_build(const float* pb, int64_t n, int max_node_primitives, trace_bvh** out) {
    return build_entry<LiteralSplitter>(pb, n, max_node_primitives < 255 ? max_node_primitives : 255, out);
}

// Opt-in alternative (SURVEY.md §8f.2): a conventional binned SAH over the same inputs, emitted in the same node format,
// so every kernel runs on it unchanged.  The closest hit of a ray does not depend on the tree (ties between equal t
// aside), so images agree; traversal work drops because the literal cost function is degenerate (Q16: depth 42 and
// 2 663 empty leaves on the caustic mesh).
extern "C" int trace_bvh_build_sah(const float* pb, int64_t n, int max_node_primitives, trace_bvh** out) {
    const int m = max_node_primitives < 1 ? 1 : (max_node_primitives < 255 ? max_node_primitives : 255);
    return build_entry<SahSplitter>(pb, n, m, out);
}

// The handle for builders outside this file (bvh_gpu.cu): arrays of the given sizes, left uninitialised for the caller
// to fill; nullptr when out of memory.
trace_bvh* bvh_alloc(int64_t n_nodes, int64_t n_prims, trace_bvh_node** nodes, uint32_t** order) {
    try {
        std::unique_ptr<trace_bvh> bvh(new trace_bvh());
        bvh->nodes.resize((size_t)n_nodes);
        bvh->order.resize((size_t)n_prims);
        *nodes = bvh->nodes.data();
        *order = bvh->order.data();
        return bvh.release();
    } catch (...) { return nullptr; }
}

extern "C" int64_t trace_bvh_num_nodes(const trace_bvh* b) { return b ? (int64_t)b->nodes.size() : 0; }
extern "C" int64_t trace_bvh_num_prims(const trace_bvh* b) { return b ? (int64_t)b->order.size() : 0; }
extern "C" int trace_bvh_copy(const trace_bvh* b, trace_bvh_node* nodes_out, uint32_t* order_out) {
    if (!b) return 1;
    if (nodes_out && !b->nodes.empty()) memcpy(nodes_out, b->nodes.data(), b->nodes.size() * sizeof(trace_bvh_node));
    if (order_out && !b->order.empty()) memcpy(order_out, b->order.data(), b->order.size() * sizeof(uint32_t));
    return 0;
}
extern "C" void trace_bvh_free(trace_bvh* b) { delete b; }
