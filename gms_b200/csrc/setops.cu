// setops.cu — SortedSet algebra on the device, batched over neighbourhood pairs of a graph and over device-resident sets
// (sets.cu), and the vertex-similarity measures built on it.
//
// Replaces:
//   SortedSetBase::intersect_count / intersect      gms/representations/sets/sorted_set.h:160-182
//   SortedSetBase::union_with / union_count / difference   sorted_set.h:104-109,140,184-189
//   vec_set_{union,intersect,intersect_count,difference}   sets/sorted_set_operations.h:30-106
//   GMS::VertexSim::vertex_similarity<Metric>       gms/algorithms/set_based/vertex_similarity/vertex_similarity.h:30-221
//
// One warp per pair (A_i, B_i).  Both input forms run on the same two kernels, templated on where pair i's lists come
// from: PairLists (N(pa[i]), N(pb[i]) of a graph; the ids are checked on the device) and SpanLists (one left set
// against right[i]: set handles, or the neighbourhoods of a set's members).
//   k_set_count   |A ∩ B| by merge path or galloping (isect.cuh: warp_intersect_count); |A ∪ B|, |A \ B| follow.
//   k_set_op<OP>  A op B materialised, ascending, in two passes: sizes, then the elements at their scanned offsets.
// The similarity scores are IEEE doubles computed from integer counts with the same expressions as the reference, so
// Jaccard, Overlap, CommNeigh, TotalNeigh and PrefAtt are bit-exact; Resource sums 1/deg(w) in ascending-w order like
// the reference (bit-exact); AdamicAdar additionally depends on log() and agrees to a few ulp.
#include "common.cuh"
#include "sort.cuh"
#include "isect.cuh"
#include "ops.cuh"
#include "sets.cuh"

#include <tuple>
#include <vector>

namespace gmsb {

namespace {

constexpr int kWarps = 8;

// pair i = (N(pa[i]), N(pb[i])); an id outside the graph raises *bad and the pair is skipped
struct PairLists {
    const eid_t *off;
    const vid_t *nbr;
    int64_t n;
    const vid_t *pa, *pb;
    int *bad;
    __device__ __forceinline__ bool lists(int64_t i, const vid_t *&a, int &na, const vid_t *&b, int &nb) const {
        const vid_t va = pa[i], vb = pb[i];
        if (va < 0 || vb < 0 || va >= n || vb >= n) { *bad = 1; return false; }
        const eid_t oa = off[va], ob = off[vb];
        a = nbr + oa; na = (int)(off[va + 1] - oa);
        b = nbr + ob; nb = (int)(off[vb + 1] - ob);
        return true;
    }
    auto args() const { return std::make_tuple(off, nbr, n, pa, pb, bad); }   // host: the kernel arguments
    // after a kernel that read this source: throws if a pair named a vertex outside the graph
    void check(const char *what) const {
        int flag = 0;
        GMSB_CUDA(cudaMemcpyAsync(&flag, bad, sizeof flag, cudaMemcpyDeviceToHost, rt().stream));
        GMSB_CUDA(cudaStreamSynchronize(rt().stream));
        GMSB_REQUIRE(flag == 0, std::string(what) + ": vertex id out of range");
    }
};

// pair i = (left, right[i]); set handles are valid by construction and member neighbourhoods are checked when built
struct SpanLists {
    Span left;
    const Span *right;
    __device__ __forceinline__ bool lists(int64_t i, const vid_t *&a, int &na, const vid_t *&b, int &nb) const {
        a = left.p; na = (int)left.n;
        b = right[i].p; nb = (int)right[i].n;
        return true;
    }
    auto args() const { return std::make_tuple(left, right); }
    void check(const char *) const {}
};

// The kernels below take a source's pointers as __restrict__ parameters and build the source inside: loads through
// pointers that arrive inside a struct are not compiled as read-only (LDG.CONSTANT) loads.

// out[i] = |A ∩ B|, |A ∪ B| = |A| + |B| - |A ∩ B| (sorted_set.h:140) or |A \ B| = |A| - |A ∩ B|
template <typename Src>
__device__ __forceinline__ void set_count(const Src &src, int64_t np, gmsb_set_op_kind op,
                                          unsigned long long *__restrict__ out) {
    __shared__ vid_t stage[kWarps][kMergeTile + 2];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < np; i += nwarps) {
        const vid_t *a, *b;
        int na, nb;
        if (!src.lists(i, a, na, b, nb)) { if (lane == 0) out[i] = 0; continue; }
        const unsigned long long c = warp_sum(warp_intersect_count(a, na, b, nb, lane, stage[wib]));
        if (lane == 0)
            out[i] = op == GMSB_SET_INTERSECT ? c
                   : op == GMSB_SET_UNION     ? (unsigned long long)na + (unsigned long long)nb - c
                                              : (unsigned long long)na - c;
    }
}
__global__ void __launch_bounds__(kWarps * 32)
k_set_count(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n, const vid_t *__restrict__ pa,
            const vid_t *__restrict__ pb, int *__restrict__ bad, int64_t np, gmsb_set_op_kind op,
            unsigned long long *__restrict__ out) {
    set_count(PairLists{off, nbr, n, pa, pb, bad}, np, op, out);
}
__global__ void __launch_bounds__(kWarps * 32)
k_set_count(Span left, const Span *__restrict__ right, int64_t np, gmsb_set_op_kind op,
            unsigned long long *__restrict__ out) {
    set_count(SpanLists{left, right}, np, op, out);
}

// Materialising A op B, ascending, two passes (out_elems == nullptr: counts[i] only; then write at out_off[i]).
// Lanes walk a list in chunks of 32 and binary-search the other; ballots keep the order.
//   intersect: elements of the shorter list found in the longer one      (std::set_intersection)
//   difference: elements of A not found in B                              (std::set_difference)
//   union: every element knows its place without a merge — an element x of A sits after the |A<x| + |B<x| - |A∩B<x|
//          smaller ones, i.e. at j + lower_bound(B, x) - (common elements among A[0..j)); an element of B that is not
//          in A likewise                                                   (std::set_union)
template <gmsb_set_op_kind OP, typename Src>
__device__ __forceinline__ void set_op(const Src &src, int64_t np, int64_t *__restrict__ counts,
                                       const int64_t *__restrict__ out_off, vid_t *__restrict__ out_elems) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < np; i += nwarps) {
        const vid_t *a, *b;
        int na, nb;
        if (!src.lists(i, a, na, b, nb)) continue;
        if (OP == GMSB_SET_INTERSECT && na > nb) { const vid_t *t = a; a = b; b = t; const int tn = na; na = nb; nb = tn; }
        const int64_t w = out_elems ? out_off[i] : 0;
        int c = 0;                           // elements kept so far; for union, common elements seen so far
        for (int j0 = 0; j0 < na; j0 += 32) {
            const int j = j0 + lane;
            bool hit = false;
            int lo = 0;
            vid_t x = 0;
            if (j < na) {
                x = a[j];
                lo = lower_bound_dev(b, nb, x);
                hit = lo < nb && b[lo] == x;
            }
            const bool keep = OP == GMSB_SET_INTERSECT ? hit : (OP == GMSB_SET_DIFFERENCE ? (j < na && !hit) : j < na);
            const unsigned mask = __ballot_sync(0xffffffffu, OP == GMSB_SET_UNION ? hit : keep);
            const int before = __popc(mask & ((1u << lane) - 1));
            if (out_elems && keep) out_elems[OP == GMSB_SET_UNION ? w + j + lo - (c + before) : w + c + before] = x;
            c += __popc(mask);
        }
        if (OP == GMSB_SET_UNION) {
            if (!out_elems) { if (lane == 0) counts[i] = (int64_t)na + nb - c; continue; }
            int common = 0;
            for (int t0 = 0; t0 < nb; t0 += 32) {
                const int t = t0 + lane;
                bool hit = false;
                int lo = 0;
                vid_t x = 0;
                if (t < nb) {
                    x = b[t];
                    lo = lower_bound_dev(a, na, x);
                    hit = lo < na && a[lo] == x;
                }
                const unsigned hmask = __ballot_sync(0xffffffffu, hit);
                if (t < nb && !hit) out_elems[w + t + lo - (common + __popc(hmask & ((1u << lane) - 1)))] = x;
                common += __popc(hmask);
            }
        } else if (!out_elems && lane == 0) {
            counts[i] = c;
        }
    }
}
template <gmsb_set_op_kind OP>
__global__ void __launch_bounds__(kWarps * 32)
k_set_op(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n, const vid_t *__restrict__ pa,
         const vid_t *__restrict__ pb, int *__restrict__ bad, int64_t np, int64_t *__restrict__ counts,
         const int64_t *__restrict__ out_off, vid_t *__restrict__ out_elems) {
    set_op<OP>(PairLists{off, nbr, n, pa, pb, bad}, np, counts, out_off, out_elems);
}
template <gmsb_set_op_kind OP>
__global__ void __launch_bounds__(kWarps * 32)
k_set_op(Span left, const Span *__restrict__ right, int64_t np, int64_t *__restrict__ counts,
         const int64_t *__restrict__ out_off, vid_t *__restrict__ out_elems) {
    set_op<OP>(SpanLists{left, right}, np, counts, out_off, out_elems);
}

// neighbourhoods of the listed vertices as the right-hand spans
__global__ void k_neighbourhood_spans(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n,
                                      const vid_t *__restrict__ verts, int64_t nv, Span *__restrict__ out,
                                      int *__restrict__ bad) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
        const vid_t v = verts[i];
        if (v < 0 || v >= n) { *bad = 1; out[i] = Span{nullptr, 0}; continue; }
        out[i] = Span{nbr + off[v], off[v + 1] - off[v]};
    }
}

// Similarity of one pair; lane 0 writes the score.
__global__ void __launch_bounds__(kWarps * 32)
k_pair_similarity(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n, int metric, int64_t np,
                  const vid_t *__restrict__ pa, const vid_t *__restrict__ pb, double *__restrict__ out,
                  int *__restrict__ bad) {
    const PairLists src{off, nbr, n, pa, pb, bad};
    __shared__ vid_t stage[kWarps][kMergeTile + 2];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < np; i += nwarps) {
        const vid_t *a, *b;
        int na, nb;
        if (!src.lists(i, a, na, b, nb)) { if (lane == 0) out[i] = 0; continue; }
        double score;
        if (metric == GMSB_SIM_PREF_ATT) {
            score = (double)((unsigned long long)na * (unsigned long long)nb);            // vertex_similarity.h:153-156
        } else if (metric == GMSB_SIM_ADAMIC_ADAR || metric == GMSB_SIM_RESOURCE) {
            // sum over w in A∩B, ascending w, of 1/log(deg w) or 1/deg w  (vertex_similarity.h:95-126)
            const vid_t *s = a, *l = b;
            int ns = na, nl = nb;
            if (ns > nl) { const vid_t *t = s; s = l; l = t; int tn = ns; ns = nl; nl = tn; }
            double sum = 0;
            for (int j0 = 0; j0 < ns; j0 += 32) {
                const int j = j0 + lane;
                bool hit = false;
                double term = 0;
                if (j < ns) {
                    const vid_t x = s[j];
                    int lo = lower_bound_dev(l, nl, x);
                    hit = lo < nl && l[lo] == x;
                    if (hit) {
                        const double dw = (double)(off[x + 1] - off[x]);
                        term = metric == GMSB_SIM_ADAMIC_ADAR ? 1. / log(dw) : 1.0 / dw;
                    }
                }
                unsigned mask = __ballot_sync(0xffffffffu, hit);
                while (mask) {                         // sequential, ascending: same rounding order as the reference
                    const int src_lane = __ffs(mask) - 1;
                    sum += __shfl_sync(0xffffffffu, term, src_lane);
                    mask &= mask - 1;
                }
            }
            score = sum;
        } else {
            unsigned long long c = warp_sum(warp_intersect_count(a, na, b, nb, lane, stage[wib]));
            const double cd = (double)c;
            if (metric == GMSB_SIM_JACCARD)                                              // :30-37 (sic: plus)
                score = (na == 0 && nb == 0) ? 1.0 : cd / (double)((unsigned long long)na + (unsigned long long)nb + cd);
            else if (metric == GMSB_SIM_OVERLAP)                                         // :64-66
                score = cd / (double)(unsigned long long)(na < nb ? na : nb);
            else if (metric == GMSB_SIM_COMM_NEIGH)                                      // :138-141
                score = cd;
            else                                                                         // TotalNeigh = |A ∪ B|
                score = (double)((unsigned long long)na + (unsigned long long)nb - c);
        }
        if (lane == 0) out[i] = score;
    }
}

// undirected edges u<v in CSR order
__global__ void k_count_upper(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n,
                              int64_t *__restrict__ cnt) {
    for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < n; u += (int64_t)gridDim.x * blockDim.x) {
        const eid_t b = off[u], e = off[u + 1];
        // lists are ascending: entries > u form a suffix
        int lo = lower_bound_dev(nbr + b, (int)(e - b), (vid_t)(u + 1));
        cnt[u] = (e - b) - lo;
        if (u == 0) cnt[n] = 0;
    }
}
__global__ void k_emit_upper(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n,
                             const int64_t *__restrict__ base, vid_t *__restrict__ pa, vid_t *__restrict__ pb) {
    int lane = threadIdx.x & 31;
    int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t u = warp; u < n; u += nwarps) {
        const eid_t e = off[u + 1];
        const int64_t c = base[u + 1] - base[u];
        const eid_t s0 = e - c;
        for (int64_t j = lane; j < c; j += 32) { pa[base[u] + j] = (vid_t)u; pb[base[u] + j] = nbr[s0 + j]; }
    }
}

}  // namespace

template <typename Src>
static void count_sets(gmsb_set_op_kind op, const Src &src, int64_t np, const char *what, uint64_t *out) {
    Runtime &r = rt();
    DevBuf<unsigned long long> dout(np);
    const int grid = (int)std::min<int64_t>(ceil_div(np, kWarps), (int64_t)r.sm_count * 16);
    std::apply([&](auto... s) { k_set_count<<<grid, kWarps * 32, 0, r.stream>>>(s..., np, op, dout.p); }, src.args());
    launched();
    dout.download(reinterpret_cast<unsigned long long *>(out), np);
    src.check(what);
}

template <typename Src>
static void launch_set_op(gmsb_set_op_kind op, const Src &src, int64_t np, int64_t *counts, const int64_t *out_off,
                          vid_t *out_elems) {
    Runtime &r = rt();
    const int grid = (int)std::min<int64_t>(ceil_div(np, kWarps), (int64_t)r.sm_count * 16);
    std::apply([&](auto... s) {
        if (op == GMSB_SET_INTERSECT)
            k_set_op<GMSB_SET_INTERSECT><<<grid, kWarps * 32, 0, r.stream>>>(s..., np, counts, out_off, out_elems);
        else if (op == GMSB_SET_UNION)
            k_set_op<GMSB_SET_UNION><<<grid, kWarps * 32, 0, r.stream>>>(s..., np, counts, out_off, out_elems);
        else
            k_set_op<GMSB_SET_DIFFERENCE><<<grid, kWarps * 32, 0, r.stream>>>(s..., np, counts, out_off, out_elems);
    }, src.args());
    launched();
}

// A_i op B_i for np >= 1 pairs: the count pass, the exclusive scan of the sizes (copied to offs[0..np] on the host)
// and, with `write`, the elements at those offsets, left on the device.  A bad pair id throws before offs[1..np] is
// written; a total above `cap` throws after it.
template <typename Src>
static DevBuf<vid_t> set_op_pairs(gmsb_set_op_kind op, const Src &src, int64_t np, const char *what, int64_t *offs,
                                  bool write, int64_t cap) {
    DevBuf<int64_t> cnt(np + 1), pos(np + 1);
    cnt.zero();
    launch_set_op(op, src, np, cnt.p, nullptr, nullptr);
    src.check(what);
    exclusive_sum(cnt.p, pos.p, np + 1);
    pos.download(offs, np + 1);
    const int64_t total = offs[np];
    DevBuf<vid_t> elems;
    if (!write) return elems;
    GMSB_REQUIRE(cap >= total, std::string(what) + ": output capacity too small");
    if (total == 0) return elems;
    elems.alloc(total);
    launch_set_op(op, src, np, nullptr, pos.p, elems.p);
    return elems;
}

// ---- neighbourhood pairs ---------------------------------------------------------------------------------------------
static void count_batch(Graph &g, gmsb_set_op_kind op, const char *what, int64_t np, const vid_t *a, const vid_t *b,
                        uint64_t *out) {
    if (np == 0) return;
    DevBuf<vid_t> da(np), db(np);
    DevBuf<int> bad(1);
    bad.zero();
    da.upload(a, np); db.upload(b, np);
    count_sets(op, PairLists{g.off.p, g.nbr.p, g.n, da.p, db.p, bad.p}, np, what, out);
}
void intersect_count_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, uint64_t *out) {
    count_batch(g, GMSB_SET_INTERSECT, "intersect_count_batch", np, a, b, out);
}
void union_count_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, uint64_t *out) {
    count_batch(g, GMSB_SET_UNION, "union_count_batch", np, a, b, out);
}

static void set_batch(Graph &g, gmsb_set_op_kind op, const char *what, int64_t np, const vid_t *a, const vid_t *b,
                      int64_t *out_offsets, vid_t *out_elems, int64_t cap) {
    out_offsets[0] = 0;
    if (np == 0) return;
    DevBuf<vid_t> da(np), db(np);
    DevBuf<int> bad(1);
    bad.zero();
    da.upload(a, np); db.upload(b, np);
    const DevBuf<vid_t> elems = set_op_pairs(op, PairLists{g.off.p, g.nbr.p, g.n, da.p, db.p, bad.p}, np, what,
                                             out_offsets, out_elems != nullptr, cap);
    if (elems.n) elems.download(out_elems, elems.n);
}
void intersect_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, int64_t *out_offsets, vid_t *out_elems,
                     int64_t cap) {
    set_batch(g, GMSB_SET_INTERSECT, "intersect_batch", np, a, b, out_offsets, out_elems, cap);
}
void difference_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, int64_t *out_offsets, vid_t *out_elems,
                      int64_t cap) {
    set_batch(g, GMSB_SET_DIFFERENCE, "difference_batch", np, a, b, out_offsets, out_elems, cap);
}
void union_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, int64_t *out_offsets, vid_t *out_elems,
                 int64_t cap) {
    set_batch(g, GMSB_SET_UNION, "union_batch", np, a, b, out_offsets, out_elems, cap);
}

// ---- one device set against many -------------------------------------------------------------------------------------
static Span span_of(const DevSet &s) { return Span{s.p, s.n}; }

static DevBuf<Span> upload_spans(int64_t np, DevSet *const *bs) {
    std::vector<Span> h((size_t)np);
    for (int64_t i = 0; i < np; ++i) { GMSB_REQUIRE(bs[i] != nullptr, "set op: null set handle"); h[i] = span_of(*bs[i]); }
    DevBuf<Span> d((size_t)np);
    d.upload(h.data(), (size_t)np);
    return d;
}

void set_op_count_many(gmsb_set_op_kind op, const DevSet &a, int64_t np, DevSet *const *bs, uint64_t *out) {
    if (np == 0) return;
    const DevBuf<Span> d = upload_spans(np, bs);
    count_sets(op, SpanLists{span_of(a), d.p}, np, "set_op_count_many", out);
}

void set_op_count_members(gmsb_set_op_kind op, const DevSet &a, Graph &g, const DevSet &members, uint64_t *out) {
    if (members.n == 0) return;
    Runtime &r = rt();
    DevBuf<Span> d((size_t)members.n);
    DevBuf<int> bad(1);
    bad.zero();
    k_neighbourhood_spans<<<grid_for(members.n, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, g.n, members.p, members.n,
                                                                        d.p, bad.p);
    launched();
    GMSB_REQUIRE(bad.get(0) == 0, "set op: member outside the graph");
    count_sets(op, SpanLists{span_of(a), d.p}, members.n, "set_op_count_neighbourhoods", out);
}

void set_op_many(gmsb_set_op_kind op, const DevSet &a, int64_t np, DevSet *const *bs, DevSet **outs) {
    if (np == 0) return;
    const DevBuf<Span> d = upload_spans(np, bs);
    std::vector<int64_t> ho((size_t)np + 1);
    const DevBuf<vid_t> elems = set_op_pairs(op, SpanLists{span_of(a), d.p}, np, "set_op_many", ho.data(), true,
                                             INT64_MAX);
    std::vector<DevSet *> made;
    try {
        for (int64_t i = 0; i < np; ++i) {
            made.push_back(set_from_device(elems.p + ho[i], ho[i + 1] - ho[i], true));
            outs[i] = made.back();
        }
    } catch (...) { for (auto *m : made) delete m; throw; }
}

// ---- similarity ------------------------------------------------------------------------------------------------------
void pair_similarity_device(Graph &g, int metric, int64_t np, const vid_t *da, const vid_t *db, double *out) {
    Runtime &r = rt();
    DevBuf<double> dout(np);
    DevBuf<int> bad(1);
    bad.zero();
    const PairLists src{g.off.p, g.nbr.p, g.n, da, db, bad.p};
    int grid = (int)std::min<int64_t>(ceil_div(np, kWarps), (int64_t)r.sm_count * 16);
    k_pair_similarity<<<grid, kWarps * 32, 0, r.stream>>>(g.off.p, g.nbr.p, g.n, metric, np, da, db, dout.p, bad.p);
    launched();
    dout.download(out, np);
    src.check("pair_similarity");
}

void pair_similarity(Graph &g, int metric, int64_t np, const vid_t *a, const vid_t *b, double *out) {
    if (np == 0) return;
    DevBuf<vid_t> da(np), db(np);
    da.upload(a, np); db.upload(b, np);
    pair_similarity_device(g, metric, np, da.p, db.p, out);
}

void upper_edge_base(Graph &g, DevBuf<int64_t> &base, int64_t *m_out) {
    Runtime &r = rt();
    const int64_t n = g.n;
    DevBuf<int64_t> cnt(n + 1);
    base.alloc(n + 1);
    *m_out = 0;
    if (n) {
        k_count_upper<<<grid_for(n, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, n, cnt.p); launched();
        exclusive_sum(cnt.p, base.p, n + 1);
        *m_out = base.get(n);
    }
}
void emit_upper_pairs(Graph &g, const int64_t *base_dev, vid_t *pa, vid_t *pb) {
    k_emit_upper<<<grid_for(g.n * 32, 256), 256, 0, rt().stream>>>(g.off.p, g.nbr.p, g.n, base_dev, pa, pb); launched();
}

void edge_similarity(Graph &g, int metric, double *out, int64_t *m_out) {
    GMSB_REQUIRE(!g.directed, "edge_similarity: graph must be undirected");
    Runtime &r = rt();
    const int64_t n = g.n;
    int64_t m = 0;
    DevBuf<int64_t> base;
    upper_edge_base(g, base, &m);
    if (m_out) *m_out = m;
    if (!out || m == 0) return;
    if (metric != GMSB_SIM_ADAMIC_ADAR && metric != GMSB_SIM_RESOURCE) {
        // these five depend on the graph only through |N(a) ∩ N(b)| = the edge's triangle support: one pass of the
        // oriented triangle schedule instead of one symmetric intersection per edge (tc_support.cu)
        DevBuf<double> dout(m);
        edge_scores_from_support(g, metric, base.p, dout.p);
        dout.download(out, m);
        return;
    }
    DevBuf<vid_t> pa(m), pb(m);
    k_emit_upper<<<grid_for(n * 32, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, n, base.p, pa.p, pb.p); launched();
    pair_similarity_device(g, metric, m, pa.p, pb.p, out);
}

}  // namespace gmsb
