// sets.cu — device-resident sorted sets: the Set concept of GMS as an object.
//
// Replaces (as a drop-in type for algorithms written against the Set concept, SURVEY.md 8b):
//   SortedSetBase<int32_t>            gms/representations/sets/sorted_set.h:22-270
//   SortedSetRefBase<int32_t>         gms/representations/sets/sorted_set_ref.h:10-80   (borrowed neighbourhoods)
//
// A set is an ascending, duplicate-free int32 array in HBM — owned, or borrowed from a graph's CSR like SortedSetRef.
// This file holds the object: construct (sorting what it is given), range, neighbourhood view, clone, find, add /
// remove, equality, copy to the host.  Its binary operations (vec_set_{union,intersect,intersect_count,difference},
// sets/sorted_set_operations.h:30-106) take SET HANDLES and leave their result on the device, so a chain such as the
// Bron-Kerbosch step  P' = P ∩ N(v), X' = X ∩ N(v), P = P \ {v}  (maximal_clique_enum/sequential/tomita.h:17-60) never
// returns to the host; they run on the same kernels as the batched neighbourhood API, in setops.cu.
#include "common.cuh"
#include "sort.cuh"
#include "isect.cuh"
#include "sets.cuh"

namespace gmsb {

namespace {

__global__ void k_iota(vid_t *__restrict__ out, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (vid_t)i;
}
// flags[0] = 1 when x is in the set; flags[1] = lower bound position of x
__global__ void k_find(const vid_t *__restrict__ p, int64_t n, vid_t x, int64_t *__restrict__ res) {
    int64_t lo = 0, hi = n;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (p[mid] < x) lo = mid + 1; else hi = mid; }
    res[0] = lo < n && p[lo] == x;
    res[1] = lo;
}
__global__ void k_equal(const vid_t *__restrict__ a, const vid_t *__restrict__ b, int64_t n, int *__restrict__ diff) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        if (a[i] != b[i]) *diff = 1;
}
__global__ void k_insert(const vid_t *__restrict__ in, int64_t n, int64_t pos, vid_t x, vid_t *__restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i <= n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = i < pos ? in[i] : (i == pos ? x : in[i - 1]);
}
__global__ void k_erase(const vid_t *__restrict__ in, int64_t n, int64_t pos, vid_t *__restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i + 1 < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = i < pos ? in[i] : in[i + 1];
}

}  // namespace

DevSet *set_from_device(const vid_t *src, int64_t count, bool sorted) {
    GMSB_REQUIRE(count >= 0 && (count == 0 || src != nullptr), "set: bad arguments");
    GMSB_REQUIRE(count < (int64_t(1) << 31), "set: more than 2^31 elements");
    Runtime &r = rt();
    auto *s = new DevSet();
    try {
        s->own.alloc((size_t)count);
        s->n = count;
        if (count) {
            if (sorted) {
                GMSB_CUDA(cudaMemcpyAsync(s->own.p, src, sizeof(vid_t) * count, cudaMemcpyDeviceToDevice, r.stream));
            } else {
                // SortedSetBase(const T*, size_t) sorts what it is given (sorted_set.h:64-66,265-268)
                DevBuf<vid_t> tmp((size_t)count);
                GMSB_CUDA(cudaMemcpyAsync(tmp.p, src, sizeof(vid_t) * count, cudaMemcpyDeviceToDevice, r.stream));
                size_t bytes = 0;
                GMSB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, tmp.p, s->own.p, (int)count, 0, 32, r.stream));
                DevBuf<uint8_t> scratch(bytes);
                GMSB_CUDA(cub::DeviceRadixSort::SortKeys(scratch.p, bytes, tmp.p, s->own.p, (int)count, 0, 32, r.stream));
                r.launches += 5;
                GMSB_CUDA(cudaStreamSynchronize(r.stream));
            }
        }
        s->p = s->own.p;
        GMSB_CUDA(cudaStreamSynchronize(r.stream));
    } catch (...) { delete s; throw; }
    return s;
}

DevSet *set_from_host(const vid_t *elems, int64_t count) {
    GMSB_REQUIRE(count >= 0 && (count == 0 || elems != nullptr), "set_from_host: bad arguments");
    for (int64_t i = 0; i < count; ++i) GMSB_REQUIRE(elems[i] >= 0, "set_from_host: negative element");
    bool sorted = true;
    for (int64_t i = 1; i < count && sorted; ++i) sorted = elems[i - 1] < elems[i];
    DevBuf<vid_t> tmp((size_t)count);
    tmp.upload(elems, (size_t)count);
    return set_from_device(tmp.p, count, sorted);
}

DevSet *set_range(int64_t bound) {
    GMSB_REQUIRE(bound >= 0 && bound < (int64_t(1) << 31), "set_range: bad bound");
    Runtime &r = rt();
    auto *s = new DevSet();
    try {
        s->own.alloc((size_t)bound);
        s->n = bound;
        s->p = s->own.p;
        if (bound) { k_iota<<<grid_for(bound, 256), 256, 0, r.stream>>>(s->own.p, bound); launched(); }
        GMSB_CUDA(cudaStreamSynchronize(r.stream));
    } catch (...) { delete s; throw; }
    return s;
}

DevSet *set_neighbourhood(Graph &g, vid_t v) {
    GMSB_REQUIRE(v >= 0 && v < g.n, "set_neighbourhood: vertex out of range");
    eid_t be[2];
    GMSB_CUDA(cudaMemcpyAsync(be, g.off.p + v, 2 * sizeof(eid_t), cudaMemcpyDeviceToHost, rt().stream));
    GMSB_CUDA(cudaStreamSynchronize(rt().stream));
    auto *s = new DevSet();
    s->p = g.nbr.p + be[0];
    s->n = be[1] - be[0];
    return s;
}

DevSet *set_clone(const DevSet &a) { return set_from_device(a.p, a.n, true); }

void set_to_host(const DevSet &a, vid_t *out) {
    if (a.n == 0) return;
    GMSB_REQUIRE(out != nullptr, "set_to_host: null output");
    GMSB_CUDA(cudaMemcpyAsync(out, a.p, sizeof(vid_t) * a.n, cudaMemcpyDeviceToHost, rt().stream));
    GMSB_CUDA(cudaStreamSynchronize(rt().stream));
}

static void find_in(const DevSet &a, vid_t x, int64_t res[2]) {
    Runtime &r = rt();
    DevBuf<int64_t> d(2);
    k_find<<<1, 1, 0, r.stream>>>(a.p, a.n, x, d.p); launched();
    d.download(res, 2);
}
bool set_contains(const DevSet &a, vid_t x) {
    if (a.n == 0) return false;
    int64_t res[2];
    find_in(a, x, res);
    return res[0] != 0;
}
bool set_equal(const DevSet &a, const DevSet &b) {
    if (a.n != b.n) return false;
    if (a.n == 0 || a.p == b.p) return true;
    Runtime &r = rt();
    DevBuf<int> diff(1);
    diff.zero();
    k_equal<<<grid_for(a.n, 256), 256, 0, r.stream>>>(a.p, b.p, a.n, diff.p); launched();
    return diff.get(0) == 0;
}
// add / remove keep the set sorted (sorted_set.h:222-243); a borrowed view becomes an owning set first
void set_add(DevSet &a, vid_t x) {
    GMSB_REQUIRE(x >= 0, "set_add: negative element");
    Runtime &r = rt();
    int64_t res[2] = {0, 0};
    if (a.n) find_in(a, x, res);
    if (res[0]) return;
    DevBuf<vid_t> grown((size_t)a.n + 1);
    k_insert<<<grid_for(a.n + 1, 256), 256, 0, r.stream>>>(a.p, a.n, res[1], x, grown.p); launched();
    GMSB_CUDA(cudaStreamSynchronize(r.stream));
    a.own = std::move(grown);
    a.p = a.own.p;
    a.n += 1;
}
void set_remove(DevSet &a, vid_t x) {
    if (a.n == 0) return;
    Runtime &r = rt();
    int64_t res[2];
    find_in(a, x, res);
    if (!res[0]) return;
    DevBuf<vid_t> shrunk((size_t)a.n - 1);
    if (a.n > 1) { k_erase<<<grid_for(a.n, 256), 256, 0, r.stream>>>(a.p, a.n, res[1], shrunk.p); launched(); }
    GMSB_CUDA(cudaStreamSynchronize(r.stream));
    a.own = std::move(shrunk);
    a.p = a.own.p;
    a.n -= 1;
}

}  // namespace gmsb
