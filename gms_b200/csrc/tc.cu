// tc.cu — triangle counting on the degree-oriented DAG: schedule + the three intersection kernels.
//
// Replaces  GMS::TriangleCount::{Seq,Par}::count_total   gms/algorithms/set_based/triangle_count/parallel/total.h:8-24
// whose inner loop is  vec_set_intersect_count           gms/representations/sets/sorted_set_operations.h:45-71
//
// Formulation.  In rank space a triangle {u<v<w} is the wedge u->v, u->w closed by the edge v->w, so
//     TC = sum over oriented edges (u,v) of | suffix(N+(u), after v)  ∩  N+(v) |
// (the elements of N+(u) up to and including v can never be in N+(v), whose members are all > v).  Every edge is
// therefore a pair (suffix descriptor, v); descriptors are grouped by v so that one CTA can keep N+(v) on chip:
//
//   bitmap  — v is a hub: N+(v) becomes a bitmap over (v, last(N+(v))] in shared memory; the CTA streams the
//             suffixes of all in-neighbours with coalesced loads and does one bit probe per element.
//   gallop  — skewed light pair: each lane binary-searches one element of the shorter list in the longer one.
//   merge   — balanced light pair: warp-cooperative merge path, lists staged through shared memory, every lane
//             walks an equal share of the merge diagonal.
//
// The choice is made per edge on the device when the schedule ("plan") is built: hub-ness of v first, then the
// length ratio of the two lists.  Counts are integers, so every variant returns the same value.
#include "common.cuh"
#include "sort.cuh"
#include "orient.cuh"
#include "isect.cuh"
#include "tc_plan.cuh"
#include <cooperative_groups.h>
#include <cstdlib>
#include <cstring>

namespace gmsb {

void delete_plan(TcPlan *p) { delete p; }

namespace {

// ---- plan construction -----------------------------------------------------------------------------------------
// The schedule groups the suffix descriptors of all oriented edges (u,v) by their closing vertex v and, inside v,
// by length class.  It is a counting sort keyed on (v, class) — the transposed (in-edge) index of the DAG — built in
// two streaming passes over the oriented CSR instead of a radix sort of |E+| (key, descriptor) pairs:
//   pass 1  k_plan_count    one RED per edge into the 64-bit counter of (v, class): descriptors << 38 | suffix lengths
//           k_classify      per vertex: hub or light, number of CTA items (cost-balanced), segment sizes
//           two scans       item numbers and descriptor segments of the hubs
//           k_plan_layout   per vertex: the counters become absolute write cursors (or a LIGHT / DEAD mark), items written
//   pass 2  k_plan_scatter  one ATOM per edge into an owned hub takes the descriptor's slot in v's segment; edges into
//                           light vertices are appended to the merge / gallop lists instead (warp-aggregated cursors)
// With part_count > 1 a device builds ITS SHARE of the schedule only.  An edge (u,v) belongs to the device that owns its
// closing vertex v, and ownership is a function of the id alone — plan_owner: the vertices are dealt in snake order from
// the top of rank space, where the hubs are, heaviest first — so every pass skips foreign edges right after loading v:
// no gather, no atomic, no write.  Counters, classification, segments, items, descriptor writes and the item order cover
// the own vertices only, and every statistic of the schedule is this device's share (the shares add up).
// Round 1 emitted 251 M (key, descriptor) pairs at scale 24 and radix-sorted them (4 onesweep passes over 12 B per
// pair + 2 x 251 M 64-bit atomics for the per-vertex work) and then flagged / scanned / compacted the light edges.
constexpr int kCntShift = 38;                                  // counter word = (descriptors << 38) | sum of lengths
constexpr unsigned long long kWorkMask = (1ull << kCntShift) - 1ull;
constexpr unsigned long long kPosLight = 1ull << 63;           // cursor marks: edges into a light vertex ...
constexpr unsigned long long kPosDead = 1ull << 62;            // ... and into a vertex that closes no triangle
// What the scatter pass needs to know about the closing vertex v of an edge, one byte per vertex (the array stays in
// the L2; the 24-byte cursor triples do not).  Only edges into a hub this device owns touch a cursor.
constexpr uint8_t kDead = 0;        // no incoming descriptor can close a triangle
constexpr uint8_t kLight = 1;       // edges go to the merge / gallop lists
constexpr uint8_t kHub = 2;         // hub whose descriptor segment this device builds
constexpr uint8_t kElsewhere = 3;   // vertex owned by another device (part_count > 1)

// owner of closing vertex v among the devices: rank space puts the highest degrees last, so counting from the top deals
// the hubs out in (nearly) descending order of work; the snake order evens out the steps between neighbours (owner.cuh)
__device__ __forceinline__ int plan_owner(vid_t v, int64_t n, const OwnerDeal &od) {
    return deal_owner(od, (uint32_t)(n - 1 - (int64_t)v));
}

__device__ __forceinline__ uint32_t len_class(eid_t len) { return len <= kShortLen ? 0u : (len <= kMidLen ? 1u : 2u); }

// One edge (u,v) of the count pass, both forms: len = suffix length after v, du = d+(u); sums as in k_plan_count's acc.
__device__ __forceinline__ void count_edge(vid_t v, eid_t len, unsigned long long du, const int32_t *__restrict__ dplus,
                                           unsigned long long *__restrict__ cw, unsigned long long &deg2,
                                           unsigned long long &wedges, unsigned long long &kept, unsigned long long &ku) {
    const int dv = dplus[v];
    deg2 += du + (unsigned long long)dv;
    if (len > 0 && dv > 0) {
        atomicAdd(&cw[3 * (int64_t)v + len_class(len)], (1ull << kCntShift) | (unsigned long long)len);
        wedges += (unsigned long long)len; kept++; ku += du;
    }
}

__device__ __forceinline__ void flush_counts(unsigned long long *__restrict__ acc, unsigned long long deg2,
                                             unsigned long long wedges, unsigned long long kept, unsigned long long ku) {
    for (int o = 16; o; o >>= 1) {
        deg2 += __shfl_xor_sync(0xffffffffu, deg2, o);
        wedges += __shfl_xor_sync(0xffffffffu, wedges, o);
        kept += __shfl_xor_sync(0xffffffffu, kept, o);
        ku += __shfl_xor_sync(0xffffffffu, ku, o);
    }
    if ((threadIdx.x & 31) == 0 && deg2) {
        atomicAdd(&acc[0], deg2); atomicAdd(&acc[1], wedges); atomicAdd(&acc[2], kept); atomicAdd(&acc[3], ku);
    }
}

template <int G>
__global__ void __launch_bounds__(256)
k_plan_count(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const int32_t *__restrict__ dplus,
             int64_t n, int part_index, OwnerDeal od, unsigned long long *__restrict__ cw /* 3n */,
             unsigned long long *__restrict__ acc /* over the own edges: [0]=sum d+(u)+d+(v)  [1]=wedges  [2]=kept edges
                                                     [3]=sum d+(u), kept edges */) {
    const int sub = threadIdx.x % G;
    const int64_t grp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    const int64_t ngrp = ((int64_t)gridDim.x * blockDim.x) / G;
    unsigned long long deg2 = 0, wedges = 0, kept = 0, ku = 0;
    for (int64_t u = grp; u < n; u += ngrp) {
        const eid_t b = off[u], e = off[u + 1];
        const unsigned long long du = (unsigned long long)(e - b);
        for (eid_t s = b + sub; s < e; s += G) {
            const vid_t v = nbr[s];
            if (od.parts > 1 && plan_owner(v, n, od) != part_index) continue;
            count_edge(v, e - s - 1, du, dplus, cw, deg2, wedges, kept, ku);
        }
    }
    flush_counts(acc, deg2, wedges, kept, ku);
}

// The same pass as an element-wise stream over the edge slots, given Dag::spos (position and suffix length per slot,
// built once per DAG by k_slot_positions): no row is walked, so a device that owns 1/P of the closing vertices pays for
// a coalesced read of two arrays plus 1/P of the gathers and atomics.  Measured at scale 24
// (profiles/r2o_partition_balance.jsonl): schedule of one part of 8 3.1-3.3 ms against 3.8-3.9 ms with the row walks,
// but 11.4 against 10.6 ms for the whole schedule — so the element-wise form is used from 4 parts on.
__global__ void __launch_bounds__(256)
k_slot_positions(const eid_t *__restrict__ off, int64_t n, uint32_t *__restrict__ spos) {
    constexpr int G = 8;
    const int sub = threadIdx.x % G;
    const int64_t grp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    const int64_t ngrp = ((int64_t)gridDim.x * blockDim.x) / G;
    for (int64_t u = grp; u < n; u += ngrp) {
        const eid_t b = off[u], e = off[u + 1];
        for (eid_t s = b + sub; s < e; s += G) spos[s] = ((uint32_t)(s - b) << 16) | (uint32_t)(e - s - 1);
    }
}

constexpr int kFlatUnroll = 4;
__global__ void __launch_bounds__(256)
k_plan_count_flat(const vid_t *__restrict__ nbr, const uint32_t *__restrict__ spos, const int32_t *__restrict__ dplus,
                  int64_t m, int64_t n, int part_index, OwnerDeal od, unsigned long long *__restrict__ cw /* 3n */,
                  unsigned long long *__restrict__ acc) {
    unsigned long long deg2 = 0, wedges = 0, kept = 0, ku = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t s0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s0 < m; s0 += kFlatUnroll * stride) {
        vid_t vs[kFlatUnroll];
        uint32_t sps[kFlatUnroll];
#pragma unroll
        for (int q = 0; q < kFlatUnroll; ++q) {                       // independent streaming loads first
            const int64_t s = s0 + q * stride;
            vs[q] = s < m ? nbr[s] : -1;
            sps[q] = s < m ? spos[s] : 0u;
        }
#pragma unroll
        for (int q = 0; q < kFlatUnroll; ++q) {
            const vid_t v = vs[q];
            if (v < 0 || (od.parts > 1 && plan_owner(v, n, od) != part_index)) continue;
            const eid_t len = (eid_t)(sps[q] & 0xffffu);
            const unsigned long long du = (unsigned long long)(sps[q] >> 16) + (unsigned long long)len + 1ull;
            count_edge(v, len, du, dplus, cw, deg2, wedges, kept, ku);
        }
    }
    flush_counts(acc, deg2, wedges, kept, ku);
}

struct PlanParams {
    int variant;
    int hub_bits;
    long long hub_min_work;
};

// Work target of one hub item: list elements probed plus 4 per descriptor, and never less than 16 x d+(v), the cost of
// setting and clearing the bitmap.  Half of it bought nothing at scale 24 (profiles/r2m_tile_order_sweep.jsonl: 35.2-35.3
// ms of counting kernels, with address tiles, against 34.35 ms for this target with positional tiles).
constexpr long long kItemCost = 262144;

// Per vertex: hub or not, and into how many CTA items its descriptor group is cut.
__global__ void k_classify(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n,
                           const unsigned long long *__restrict__ cw, PlanParams pp, int part_index, OwnerDeal od,
                           int64_t *__restrict__ nitems /* n+1 */, int64_t *__restrict__ seg /* n+1 */,
                           unsigned long long *__restrict__ cls /* [0]=hub edges [1]=hub wedges [2]=sum cnt*d+(v), hubs
                                                                  [3]=sum cnt*d+(v), all  [4]=light edges */,
                           int *__restrict__ mx /* [0]=max span words [1]=max d+ of a hub */,
                           uint8_t *__restrict__ vstate /* n: kDead / kLight / kHub / kElsewhere */) {
    int mxw = 0, mxd = 0;
    unsigned long long he = 0, hw = 0, hb = 0, ab = 0, le = 0;
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v <= n; v += (int64_t)gridDim.x * blockDim.x) {
        int64_t k = 0, sg = 0;
        if (v < n && od.parts > 1 && plan_owner((vid_t)v, n, od) != part_index) {
            vstate[v] = kElsewhere;
        } else if (v < n) {
            const unsigned long long w0 = cw[3 * v], w1 = cw[3 * v + 1], w2 = cw[3 * v + 2];
            const int64_t cnt = (int64_t)((w0 >> kCntShift) + (w1 >> kCntShift) + (w2 >> kCntShift));
            uint8_t state = kDead;
            if (cnt > 0) {
                const long long work = (long long)((w0 & kWorkMask) + (w1 & kWorkMask) + (w2 & kWorkMask));
                const eid_t ob = off[v], oe = off[v + 1];
                const unsigned long long dv = (unsigned long long)(oe - ob);
                ab += (unsigned long long)cnt * dv;
                bool hub = false;
                if (pp.variant == GMSB_TC_AUTO || pp.variant == GMSB_TC_BITMAP) {
                    const int64_t span = (int64_t)nbr[oe - 1] - v;          // bit x = w - v - 1, x in [0, span)
                    hub = span <= pp.hub_bits && (pp.variant == GMSB_TC_BITMAP || work >= pp.hub_min_work);
                    if (hub) {
                        const long long setup = 16ll * (long long)dv;
                        const long long target = kItemCost > setup ? kItemCost : setup;
                        const long long cost = work + 4ll * cnt;
                        k = (cost + target - 1) / target;
                        if (k < 1) k = 1;
                        if (k > cnt) k = cnt;
                        const int64_t chunk = (cnt + k - 1) / k;
                        k = (cnt + chunk - 1) / chunk;                      // no empty trailing items
                        sg = cnt;
                        mxw = max(mxw, (int)((span + 31) >> 5));
                        mxd = max(mxd, (int)dv);
                        he += (unsigned long long)cnt; hw += (unsigned long long)work; hb += (unsigned long long)cnt * dv;
                    }
                }
                if (!hub) le += (unsigned long long)cnt;
                state = hub ? kHub : kLight;
            }
            vstate[v] = state;
        }
        nitems[v] = k;
        seg[v] = sg;
    }
    for (int o = 16; o; o >>= 1) {
        mxw = max(mxw, __shfl_xor_sync(0xffffffffu, mxw, o));
        mxd = max(mxd, __shfl_xor_sync(0xffffffffu, mxd, o));
        he += __shfl_xor_sync(0xffffffffu, he, o); hw += __shfl_xor_sync(0xffffffffu, hw, o);
        hb += __shfl_xor_sync(0xffffffffu, hb, o); ab += __shfl_xor_sync(0xffffffffu, ab, o);
        le += __shfl_xor_sync(0xffffffffu, le, o);
    }
    if ((threadIdx.x & 31) == 0) {
        if (mxw) { atomicMax(&mx[0], mxw); atomicMax(&mx[1], mxd); }
        if (he) { atomicAdd(&cls[0], he); atomicAdd(&cls[1], hw); atomicAdd(&cls[2], hb); }
        if (ab) atomicAdd(&cls[3], ab);
        if (le) atomicAdd(&cls[4], le);
    }
}

// Counters -> write cursors; items of the hubs (a slice of the descriptor segment each, with its class boundaries).
__global__ void k_plan_layout(int64_t n, unsigned long long *__restrict__ cw, const int64_t *__restrict__ nitems,
                              const int64_t *__restrict__ item_base, const int64_t *__restrict__ segbase,
                              const uint8_t *__restrict__ vstate, Item *__restrict__ items) {
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c0 = (int64_t)(cw[3 * v] >> kCntShift), c1 = (int64_t)(cw[3 * v + 1] >> kCntShift),
                      c2 = (int64_t)(cw[3 * v + 2] >> kCntShift);
        const int64_t cnt = c0 + c1 + c2, k = nitems[v];
        const uint8_t state = vstate[v];
        if (state == kElsewhere) continue;                      // another device's vertex: its counters were never touched
        if (state == kDead) { cw[3 * v] = kPosDead; cw[3 * v + 1] = kPosDead; cw[3 * v + 2] = kPosDead; continue; }
        if (state == kLight) { cw[3 * v] = kPosLight; cw[3 * v + 1] = kPosLight; cw[3 * v + 2] = kPosLight; continue; }
        const int64_t b = segbase[v];
        cw[3 * v] = (unsigned long long)b;
        cw[3 * v + 1] = (unsigned long long)(b + c0);
        cw[3 * v + 2] = (unsigned long long)(b + c0 + c1);
        const int64_t chunk = (cnt + k - 1) / k, w = item_base[v];
        for (int64_t j = 0; j < k; ++j) {
            const int64_t s = j * chunk;                           // first descriptor of the slice, relative to b
            const int64_t c = cnt - s < chunk ? cnt - s : chunk;
            Item it;
            it.v = (int32_t)v; it.begin = b + s; it.count = (int32_t)c; it.pad[0] = 0; it.pad[1] = 0;
            const int64_t a0 = c0 - s, a1 = c0 + c1 - s;
            it.n0 = (int32_t)(a0 < 0 ? 0 : (a0 > c ? c : a0));
            it.n1 = (int32_t)(a1 < 0 ? 0 : (a1 > c ? c : a1));
            items[w + j] = it;
        }
    }
}

// Appends a light edge to the merge or the gallop list: one cursor bump per coalesced group of lanes.
__device__ __forceinline__ void append_light(unsigned long long *__restrict__ cursor, uint64_t *__restrict__ l_desc,
                                             vid_t *__restrict__ l_v, uint64_t ds, vid_t v) {
    namespace cg = cooperative_groups;
    cg::coalesced_group act = cg::coalesced_threads();
    unsigned long long base = 0;
    if (act.thread_rank() == 0) base = atomicAdd(cursor, (unsigned long long)act.size());
    const unsigned long long i = act.shfl(base, 0) + act.thread_rank();
    l_desc[i] = ds; l_v[i] = v;
}

// One edge (u,v) of the scatter pass, both forms: slot s of v in N+(u), len = suffix length after v, du = d+(u).  An edge
// into a hub takes its descriptor's slot in v's segment (du is summed for bytes_bitmap); a light edge goes to the gallop
// list when the two lists are skewed by at least `ratio`, to the merge list otherwise.
__device__ __forceinline__ void scatter_edge(bool hub, vid_t v, eid_t s, eid_t len, unsigned long long du,
                                             const int32_t *__restrict__ dplus, unsigned long long *__restrict__ pos,
                                             uint64_t *__restrict__ desc, int variant, int ratio,
                                             uint64_t *__restrict__ m_desc, vid_t *__restrict__ m_v,
                                             uint64_t *__restrict__ g_desc, vid_t *__restrict__ g_v,
                                             unsigned long long *__restrict__ cursors, unsigned long long &hub_u) {
    const uint64_t ds = ((uint64_t)(s + 1) << kLenBits) | (uint64_t)len;
    if (hub) {
        hub_u += du;
        desc[atomicAdd(&pos[3 * (int64_t)v + len_class(len)], 1ull)] = ds;
        return;
    }
    const long long a = (long long)len, dv = dplus[v];
    const long long lo = a < dv ? a : dv, hi = a < dv ? dv : a;
    const bool gallop = variant == GMSB_TC_GALLOP || (variant != GMSB_TC_MERGE && hi >= (long long)ratio * lo);
    if (gallop) append_light(&cursors[1], g_desc, g_v, ds, v);
    else append_light(&cursors[0], m_desc, m_v, ds, v);
}

template <int G>
__global__ void __launch_bounds__(256)
k_plan_scatter(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const int32_t *__restrict__ dplus,
               const uint8_t *__restrict__ vstate, int64_t n, unsigned long long *__restrict__ pos /* 3n */,
               uint64_t *__restrict__ desc, int variant, int ratio, int part_index, OwnerDeal od,
               uint64_t *__restrict__ m_desc, vid_t *__restrict__ m_v, uint64_t *__restrict__ g_desc,
               vid_t *__restrict__ g_v, unsigned long long *__restrict__ cursors /* [0]=merge [1]=gallop */,
               unsigned long long *__restrict__ acc /* [0] = sum of d+(u) over the own hub edges */) {
    const int sub = threadIdx.x % G;
    const int64_t grp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    const int64_t ngrp = ((int64_t)gridDim.x * blockDim.x) / G;
    unsigned long long hub_u = 0;
    for (int64_t u = grp; u < n; u += ngrp) {
        const eid_t b = off[u], e = off[u + 1];
        for (eid_t s = b + sub; s < e; s += G) {
            const eid_t len = e - s - 1;
            if (len <= 0) continue;
            const vid_t v = nbr[s];
            if (od.parts > 1 && plan_owner(v, n, od) != part_index) continue;
            const uint8_t state = vstate[v];
            if (state == kDead) continue;
            scatter_edge(state == kHub, v, s, len, (unsigned long long)(e - b), dplus, pos, desc, variant, ratio, m_desc,
                         m_v, g_desc, g_v, cursors, hub_u);
        }
    }
    for (int o = 16; o; o >>= 1) hub_u += __shfl_xor_sync(0xffffffffu, hub_u, o);
    if ((threadIdx.x & 31) == 0 && hub_u) atomicAdd(&acc[0], hub_u);
}

// element-wise form of the scatter pass (see k_plan_count_flat); descriptors reach their segments in ascending slot order
__global__ void __launch_bounds__(256)
k_plan_scatter_flat(const vid_t *__restrict__ nbr, const uint32_t *__restrict__ spos, const int32_t *__restrict__ dplus,
                    const uint8_t *__restrict__ vstate, int64_t m, int64_t n, unsigned long long *__restrict__ pos /* 3n */,
                    uint64_t *__restrict__ desc, int variant, int ratio, int part_index, OwnerDeal od,
                    uint64_t *__restrict__ m_desc, vid_t *__restrict__ m_v, uint64_t *__restrict__ g_desc,
                    vid_t *__restrict__ g_v, unsigned long long *__restrict__ cursors /* [0]=merge [1]=gallop */,
                    unsigned long long *__restrict__ acc /* [0] = sum of d+(u) over the own hub edges */) {
    unsigned long long hub_u = 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t s0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s0 < m; s0 += kFlatUnroll * stride) {
        vid_t vs[kFlatUnroll];
        uint32_t sps[kFlatUnroll];
#pragma unroll
        for (int q = 0; q < kFlatUnroll; ++q) {
            const int64_t s = s0 + q * stride;
            vs[q] = s < m ? nbr[s] : -1;
            sps[q] = s < m ? spos[s] : 0u;
        }
#pragma unroll
        for (int q = 0; q < kFlatUnroll; ++q) {
            const vid_t v = vs[q];
            const int64_t s = s0 + q * stride;
            const eid_t len = (eid_t)(sps[q] & 0xffffu);
            if (v < 0 || len <= 0 || (od.parts > 1 && plan_owner(v, n, od) != part_index)) continue;
            const uint8_t state = vstate[v];
            if (state == kDead) continue;
            const unsigned long long du = (unsigned long long)(sps[q] >> 16) + (unsigned long long)len + 1ull;
            scatter_edge(state == kHub, v, s, len, du, dplus, pos, desc, variant, ratio, m_desc, m_v, g_desc, g_v, cursors,
                         hub_u);
        }
    }
    for (int o = 16; o; o >>= 1) hub_u += __shfl_xor_sync(0xffffffffu, hub_u, o);
    if ((threadIdx.x & 31) == 0 && hub_u) atomicAdd(&acc[0], hub_u);
}

// Order key of an item: window class, then the L2 tile its suffixes start in (tile-major order keeps the lists that
// concurrently running CTAs stream inside the L2), then heaviest vertex first.  Window classes: 0 = NEAR (everything
// after v, up to n-1, fits the small window: no element can fall outside the bitmap), 1 = small window, 2 = wide.
// The tile is named by the slice's position inside v's descriptor segment (descriptors arrive in roughly ascending u),
// on a scale of ntiles = one per kTileSlots slots of the neighbour array: slices at the same relative position of
// different hubs advance through the array together, which the L2 rewards more than tiles read off the suffixes' start
// addresses (DESIGN.md §3.1).
constexpr int kNearWords = kSmallWindowBytes / 4 - 1;
constexpr int64_t kTileSlots = int64_t(1) << 24;
__global__ void k_item_keys(const Item *__restrict__ items, int64_t cnt, int64_t n, int64_t ntiles, int vbits, int tbits,
                            const int64_t *__restrict__ nitems, const int64_t *__restrict__ item_base,
                            const eid_t *__restrict__ off, const vid_t *__restrict__ nbr,
                            uint64_t *__restrict__ keys, unsigned long long *__restrict__ cls_count /* 3 */,
                            int *__restrict__ cls_words /* 3 */) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
        const Item it = items[i];
        const int64_t k = nitems[it.v], j = i - item_base[it.v];
        const uint64_t tile = (uint64_t)(j * ntiles / k);
        int words = (int)(((int64_t)nbr[off[it.v + 1] - 1] - it.v + 31) >> 5);
        // a NEAR window starts at the multiple of 32 at or below v + 1 and holds every id up to n - 1
        const int64_t reach_words = ((n - 1 - (((int64_t)it.v + 1) & ~int64_t(31))) >> 5) + 1;
        int cls = (words + 1) * 4 > kSmallWindowBytes ? 2 : 1;
        if (reach_words <= kNearWords) { cls = 0; words = (int)reach_words; }
        atomicAdd(&cls_count[cls], 1ull);
        atomicMax(&cls_words[cls], words);
        // packed into as few bits as the graph needs: the radix sort below runs one pass per 8 key bits
        keys[i] = ((uint64_t)cls << (tbits + vbits)) | ((tile & ((1ull << tbits) - 1ull)) << vbits) |
                  (uint64_t)(uint32_t)(n - 1 - it.v);
    }
}

// ---- counting kernels ----------------------------------------------------------------------------------------------
// Hub bitmap kernel.  Persistent CTAs (one wave, grid = SMs x resident CTAs) pull items (v, slice of v's incoming
// suffix descriptors) from a global ticket, heaviest first.  The shared-memory bitmap is zeroed ONCE per CTA; each
// item sets the bits of N+(v), streams its suffixes, then clears exactly the words it set — so the per-item cost
// is O(d+(v)) and independent of how wide the window (v, last(N+(v))] is.  Inside an item the warps pull
// descriptors from shared-memory tickets, one per length class (suffix lengths vary by 1000x): a lane, an 8-lane
// group or the whole warp takes one descriptor, so short suffixes do not pay a warp's worth of control overhead.
// List elements are read with coalesced, 4-deep predicated loads and cost ONE branch-free probe each:
// out-of-window elements and predicated-off slots are pointed at the always-zero guard word.
constexpr int kDescChunk = 4;

// The streaming loops take fewer instructions per probe than round 1's (which were issue-bound: 72 % issue-active, 20.7
// warp instructions per 32 probes; 33.7 ms against 32.0 ms at scale 24, DESIGN.md §3.1):
//   * NEAR items — hubs whose whole possible range (v, n-1] fits the window, which is where 99 % of the work is (hubs
//     are the last vertices in rank space) — need no clamp: every element of a suffix is inside the bitmap, and slots
//     that are predicated off are pointed at the guard word with a constant instead of a min;
//   * the long-suffix loop runs its full 128-element blocks without per-element bounds (one predicated tail block);
//   * the bit is taken with a wrapping funnel shift (no `& 31`).
// 128-bit loads do not pay here: a suffix starts at an arbitrary 4-byte offset, and the scalar head and tail an int4 body
// needs cost more issue slots than they save (37.7 ms against 32.0 ms, DESIGN.md §3.1).
//     In a NEAR item the window starts at a multiple of 32 (base = (v + 1) & ~31), so the bit number inside a word is
//     the element's own low five bits and the subtraction of the base moves into the (per-item) bitmap pointer:
//     element e -> word (bm - base / 32)[e >> 5], bit e & 31.  SASS per probe: LDG, SHF, LOP3, LDS, SHF.W, LOP3 + IADD3 / 2.
template <bool NEAR>
__device__ __forceinline__ uint32_t probe2(const uint32_t *bm, uint32_t e, uint32_t base, uint32_t cap_words) {
    if constexpr (NEAR) {
        return __funnelshift_r(bm[e >> 5], 0u, e) & 1u;               // bm is already shifted by -base/32 words
    } else {
        const uint32_t x = e - base;
        return __funnelshift_r(bm[min(x >> 5, cap_words)], 0u, x) & 1u;
    }
}

// G lanes cooperate on one descriptor; the warp takes 32/G descriptors per ticket (4 when G == 32).
template <int G, bool NEAR>
__device__ __forceinline__ uint32_t stream_class2(const uint64_t *__restrict__ dptr, int lo, int hi, int *ticket,
                                                  const vid_t *__restrict__ nbr, const uint32_t *bm, uint32_t base,
                                                  uint32_t cap_words, int lane) {
    uint32_t hits = 0;
    if (lo >= hi) return 0;
    // a slot that is predicated off probes the guard word: element base + 32 * cap_words (NEAR), or one that clamps
    const uint32_t off_x = NEAR ? base + (cap_words << 5) : base - 1u;
    constexpr int BATCH = G == 32 ? kDescChunk : 32 / G;
    for (;;) {
        int d0 = 0;
        if (lane == 0) d0 = atomicAdd(ticket, BATCH);
        d0 = __shfl_sync(0xffffffffu, d0, 0) + lo;
        if (d0 >= hi) break;
        if constexpr (G == 32) {
            const int nd = min(BATCH, hi - d0);
            const uint64_t mine = lane < nd ? __ldcs(&dptr[d0 + lane]) : 0ull;
            for (int k = 0; k < nd; ++k) {
                const uint64_t ds = __shfl_sync(0xffffffffu, mine, k);
                const vid_t *__restrict__ p = nbr + (ds >> kLenBits);
                const int len = (int)(ds & kLenMask);
                const vid_t *__restrict__ q = p + lane;
                for (int t = len >> 7; t > 0; --t, q += 128) {               // full 128-element blocks, no bounds
                    const uint32_t x0 = (uint32_t)q[0], x1 = (uint32_t)q[32],
                                   x2 = (uint32_t)q[64], x3 = (uint32_t)q[96];
                    hits += probe2<NEAR>(bm, x0, base, cap_words) + probe2<NEAR>(bm, x1, base, cap_words) +
                            probe2<NEAR>(bm, x2, base, cap_words) + probe2<NEAR>(bm, x3, base, cap_words);
                }
                const int rem = len & 127;
                if (rem) {
                    const uint32_t x0 = lane < rem ? (uint32_t)q[0] : off_x;
                    const uint32_t x1 = lane + 32 < rem ? (uint32_t)q[32] : off_x;
                    const uint32_t x2 = lane + 64 < rem ? (uint32_t)q[64] : off_x;
                    const uint32_t x3 = lane + 96 < rem ? (uint32_t)q[96] : off_x;
                    hits += probe2<NEAR>(bm, x0, base, cap_words) + probe2<NEAR>(bm, x1, base, cap_words) +
                            probe2<NEAR>(bm, x2, base, cap_words) + probe2<NEAR>(bm, x3, base, cap_words);
                }
            }
        } else {
            const int idx = d0 + lane / G, sub = lane % G;
            const uint64_t ds = idx < hi ? __ldcs(&dptr[idx]) : 0ull;
            const vid_t *__restrict__ p = nbr + (ds >> kLenBits);
            const int len = (int)(ds & kLenMask);
            if constexpr (G == 1) {
#pragma unroll
                for (int j = 0; j < kShortLen; ++j)
                    hits += probe2<NEAR>(bm, j < len ? (uint32_t)p[j] : off_x, base, cap_words);
            } else {
                for (int j = sub; j < len; j += 4 * G) {
                    const uint32_t x0 = (uint32_t)p[j];
                    const uint32_t x1 = j + G < len ? (uint32_t)p[j + G] : off_x;
                    const uint32_t x2 = j + 2 * G < len ? (uint32_t)p[j + 2 * G] : off_x;
                    const uint32_t x3 = j + 3 * G < len ? (uint32_t)p[j + 3 * G] : off_x;
                    hits += probe2<NEAR>(bm, x0, base, cap_words) + probe2<NEAR>(bm, x1, base, cap_words) +
                            probe2<NEAR>(bm, x2, base, cap_words) + probe2<NEAR>(bm, x3, base, cap_words);
                }
            }
        }
    }
    return hits;
}

template <int BLOCK, int MINB, bool NEAR>
__global__ void __launch_bounds__(BLOCK, MINB)
k_tc_bitmap2(const Item *__restrict__ items, int64_t count, uint32_t cap_words,
             const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const uint64_t *__restrict__ desc,
             unsigned long long *__restrict__ total, unsigned int *__restrict__ ticket) {
    extern __shared__ uint32_t bm[];                  // cap_words + 1 words
    __shared__ unsigned long long red[BLOCK / 32];
    __shared__ unsigned int s_item;
    __shared__ int s_next[3];
    const int tid = threadIdx.x, lane = tid & 31;
    for (uint32_t i = tid; i <= cap_words; i += BLOCK) bm[i] = 0u;
    unsigned long long hits64 = 0;
    for (;;) {
        if (tid == 0) { s_item = atomicAdd(ticket, 1u); s_next[0] = 0; s_next[1] = 0; s_next[2] = 0; }
        __syncthreads();                              // ticket visible; previous item's clears done
        const int64_t it = (int64_t)s_item;
        if (it >= count) break;
        const Item item = items[it];                                      // plan order: L2 tile, then heaviest
        const vid_t v = item.v;
        const eid_t ob = off[v], oe = off[v + 1];
        const uint32_t base = NEAR ? (((uint32_t)v + 1u) & ~31u) : (uint32_t)v + 1u;       // first element of the window
        for (eid_t j = ob + tid; j < oe; j += BLOCK) {
            const uint32_t x = (uint32_t)nbr[j] - base;
            atomicOr(&bm[x >> 5], 1u << (x & 31));
        }
        __syncthreads();                              // bitmap of N+(v) complete
        const uint64_t *__restrict__ dptr = desc + item.begin;
        const uint32_t *bmv = NEAR ? bm - (base >> 5) : bm;           // NEAR: indexed by the element's own word number
        uint32_t hits = stream_class2<32, NEAR>(dptr, item.n1, item.count, &s_next[2], nbr, bmv, base, cap_words, lane);
        hits += stream_class2<8, NEAR>(dptr, item.n0, item.n1, &s_next[1], nbr, bmv, base, cap_words, lane);
        hits += stream_class2<1, NEAR>(dptr, 0, item.n0, &s_next[0], nbr, bmv, base, cap_words, lane);
        hits64 += hits;
        __syncthreads();                              // every probe of this item done
        for (eid_t j = ob + tid; j < oe; j += BLOCK) bm[((uint32_t)nbr[j] - base) >> 5] = 0u;
    }
    unsigned long long s = block_sum(hits64, red);
    if (tid == 0 && s) atomicAdd(total, s);
}

// Galloping kernel: one warp per light edge (isect.cuh: warp_gallop_count).
__global__ void __launch_bounds__(256)
k_tc_gallop(const uint64_t *__restrict__ desc, const vid_t *__restrict__ vs,
            int64_t count, const eid_t *__restrict__ off, const vid_t *__restrict__ nbr,
            unsigned long long *__restrict__ total) {
    __shared__ unsigned long long red[8];
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    uint32_t hits = 0;
    for (int64_t i = warp; i < count; i += nwarps) {
        const uint64_t ds = desc[i];
        const vid_t v = vs[i];
        const eid_t ob = off[v];
        hits += warp_gallop_count(nbr + (ds >> kLenBits), (int)(ds & kLenMask), nbr + ob, (int)(off[v + 1] - ob), lane);
    }
    unsigned long long s = block_sum(hits, red);
    if (threadIdx.x == 0 && s) atomicAdd(total, s);
}

// Balanced light pairs, one warp per edge: merge path — lists staged through shared memory, every lane walks a share of
// the merge diagonal.  A block-compare intersection (32 x 32 comparisons by rotating one block past the other) was
// measured slower (scale 24, every edge forced through this kernel: 1066 ms against 534 ms; light edges of the auto
// schedule 3.59 against 3.19 ms): its 32-step rotation costs the same for a block of three elements as for a full one,
// and the light lists are short.
constexpr int kMergeWarps = 8;

__global__ void __launch_bounds__(kMergeWarps * 32)
k_tc_merge(const uint64_t *__restrict__ desc, const vid_t *__restrict__ vs,
           int64_t count, const eid_t *__restrict__ off, const vid_t *__restrict__ nbr,
           unsigned long long *__restrict__ total) {
    __shared__ vid_t stage[kMergeWarps][kMergeTile + 2];
    __shared__ unsigned long long red[kMergeWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    uint32_t hits = 0;
    for (int64_t i = warp; i < count; i += nwarps) {
        const uint64_t ds = desc[i];
        const vid_t v = vs[i];
        const eid_t ob = off[v];
        hits += warp_merge_count(nbr + (ds >> kLenBits), (int)(ds & kLenMask), nbr + ob, (int)(off[v + 1] - ob), lane,
                                 stage[wib]);
    }
    unsigned long long s = block_sum(hits, red);
    if (threadIdx.x == 0 && s) atomicAdd(total, s);
}

// ---- host side ---------------------------------------------------------------------------------------------------
gmsb_tc_options normalise(const gmsb_tc_options *in) {
    gmsb_tc_options o{};
    if (in) o = *in;
    if (o.part_count <= 0) { o.part_count = 1; o.part_index = 0; }
    if (o.hub_bitmap_bits <= 0) o.hub_bitmap_bits = 512 * 1024;      // 64 KB of shared memory
    if (o.gallop_ratio <= 0) o.gallop_ratio = 8;
    if (o.hub_min_work <= 0) o.hub_min_work = 1024;
    GMSB_REQUIRE(o.reserved[0] == 0 && o.reserved[1] == 0 && o.reserved[2] == 0 &&
                     (o.reserved[3] == 0 || o.reserved[3] == 2 || o.reserved[3] == 3),
                 "tc: reserved[0..2] must be 0 and reserved[3] one of 0, 2, 3");
    return o;
}

bool same_plan(const gmsb_tc_options &a, const gmsb_tc_options &b) {
    return a.variant == b.variant && a.hub_bitmap_bits == b.hub_bitmap_bits && a.gallop_ratio == b.gallop_ratio &&
           a.hub_min_work == b.hub_min_work && a.part_index == b.part_index &&
           a.part_count == b.part_count;      // a schedule holds one device's share
    // (reserved[3] picks the form of the edge passes, and both forms build the same schedule)
}

TcPlan *build_plan(Dag &d, const gmsb_tc_options &opt) {
    Runtime &r = rt();
    auto *p = new TcPlan();
    try {
        p->opt = opt;
        const int64_t n = d.n, m = d.m;
        const int pi = opt.part_index;
        const OwnerDeal od = make_owner_deal(opt.part_count);
        GMSB_REQUIRE(d.max_dplus < (1 << kLenBits), "tc: out-degree too large for the descriptor format");
        GMSB_REQUIRE(m < (int64_t(1) << (64 - kLenBits)), "tc: too many edges for the descriptor format");
        // the per-(vertex, class) counter packs (descriptors << 38 | sum of suffix lengths)
        GMSB_REQUIRE(d.max_deg < (int64_t(1) << (64 - kCntShift - 1)) &&
                         (double)d.max_deg * (double)d.max_dplus < (double)(1ull << kCntShift),
                     "tc: in-degree x out-degree too large for the schedule counters");
        size_t smem_cap = r.smem_optin ? r.smem_optin : 48 * 1024;
        int hub_bits = opt.hub_bitmap_bits;
        if ((size_t)hub_bits / 8 > smem_cap - 1024) hub_bits = (int)((smem_cap - 1024) * 8);
        if (m == 0 || n == 0) return p;
        PhaseTrace tr("GMSB_TC_TRACE");

        constexpr int G = 8;                    // lanes per vertex in the two edge passes (mean d+ is ~16, median far less)
        DevBuf<unsigned long long> cw(3 * (size_t)n), acc(4), cls(5);
        DevBuf<int> mx(2);
        cw.zero(); acc.zero(); cls.zero(); mx.zero();
        // element-wise passes from 4 parts on (lists shorter than 65536), row walks otherwise;
        // reserved[3]: 2 forces the row walks, 3 the element-wise form
        const bool flat = d.max_dplus < 65536 && opt.reserved[3] != 2 && (opt.part_count >= 4 || opt.reserved[3] == 3);
        if (flat && d.spos.p == nullptr) {              // once per DAG
            d.spos.alloc(m);
            k_slot_positions<<<grid_for(n * 8, 256), 256, 0, r.stream>>>(d.off.p, n, d.spos.p); launched();
        }
        if (flat)
            k_plan_count_flat<<<grid_for(m, 256), 256, 0, r.stream>>>(d.nbr.p, d.spos.p, d.dplus.p, m, n, pi, od, cw.p,
                                                                     acc.p);
        else
            k_plan_count<G><<<grid_for(n * G, 256), 256, 0, r.stream>>>(d.off.p, d.nbr.p, d.dplus.p, n, pi, od, cw.p, acc.p);
        launched();
        tr.mark("plan: count pass");
        DevBuf<int64_t> nitems(n + 1), seg(n + 1), item_base(n + 1), segbase(n + 1);
        DevBuf<uint8_t> vstate(n);
        PlanParams pp{opt.variant, hub_bits, (long long)opt.hub_min_work};
        k_classify<<<grid_for(n + 1, 256), 256, 0, r.stream>>>(d.off.p, d.nbr.p, n, cw.p, pp, pi, od, nitems.p, seg.p,
                                                              cls.p, mx.p, vstate.p);
        launched();
        unsigned long long h_acc[4], h_cls[5];
        int h_mx[2];
        acc.download(h_acc, 4);
        cls.download(h_cls, 5);
        mx.download(h_mx, 2);
        p->algorithmic_bytes = 4ull * h_acc[0];
        p->wedges = h_acc[1];
        p->n_desc = (int64_t)h_acc[2];
        p->bytes_kept = 4ull * (h_acc[3] + h_cls[3]);
        p->wedges_bitmap = h_cls[1];
        p->max_span_words = h_mx[0];
        p->max_hub_dplus = h_mx[1];
        const int64_t n_light = (int64_t)h_cls[4];
        if (p->n_desc == 0) return p;
        exclusive_sum(nitems.p, item_base.p, n + 1);
        exclusive_sum(seg.p, segbase.p, n + 1);
        tr.mark("plan: classify + scans");
        p->n_items = item_base.get(n);
        p->n_bitmap_edges = segbase.get(n);
        p->items.alloc(p->n_items);
        p->desc.alloc(p->n_bitmap_edges);
        k_plan_layout<<<grid_for(n, 256), 256, 0, r.stream>>>(n, cw.p, nitems.p, item_base.p, segbase.p, vstate.p,
                                                             p->items.p);
        launched();
        // both light lists are sized for all of this device's light edges; the scatter pass decides merge / gallop per edge
        p->m_desc.alloc(n_light); p->m_v.alloc(n_light); p->g_desc.alloc(n_light); p->g_v.alloc(n_light);
        DevBuf<unsigned long long> cursors(2), hub_u(1);
        cursors.zero(); hub_u.zero();
        // (A variant that kept the cursors of the last 4096 vertices in shared memory per 2048-vertex tile — one global
        // ATOM per non-empty counter and tile instead of one per edge — was measured slower at scale 24: 14.8 ms
        // against 9.4 ms; the two passes over the tile and the 48 KB of shared cursors per CTA cost more than the
        // returns of the global atomics.)
        if (flat)
            k_plan_scatter_flat<<<grid_for(m, 256), 256, 0, r.stream>>>(
                d.nbr.p, d.spos.p, d.dplus.p, vstate.p, m, n, cw.p, p->desc.p, opt.variant, opt.gallop_ratio, pi, od,
                p->m_desc.p, p->m_v.p, p->g_desc.p, p->g_v.p, cursors.p, hub_u.p);
        else
            k_plan_scatter<G><<<grid_for(n * G, 256), 256, 0, r.stream>>>(
                d.off.p, d.nbr.p, d.dplus.p, vstate.p, n, cw.p, p->desc.p, opt.variant, opt.gallop_ratio, pi, od,
                p->m_desc.p, p->m_v.p, p->g_desc.p, p->g_v.p, cursors.p, hub_u.p);
        launched();
        unsigned long long h_cur[2];
        cursors.download(h_cur, 2);
        p->n_merge = (int64_t)h_cur[0];
        p->n_gallop = (int64_t)h_cur[1];
        p->bytes_bitmap = 4ull * (hub_u.get(0) + h_cls[2]);
        tr.mark("plan: layout + scatter pass");
        if (p->n_items) {
            // order: tile-major, heaviest first inside a tile
            DevBuf<uint64_t> ik(p->n_items), ik2(p->n_items);
            DevBuf<Item> items2(p->n_items);
            const int64_t ntiles = std::max<int64_t>(1, (m + kTileSlots - 1) / kTileSlots);
            DevBuf<unsigned long long> ccnt(3);
            DevBuf<int> cwords(3);
            ccnt.zero(); cwords.zero();
            const int vbits = bits_for((uint64_t)n);
            const int tbits = bits_for((uint64_t)(ntiles - 1));
            const int key_bits = 2 + tbits + vbits;                 // class | tile | n - 1 - v
            k_item_keys<<<grid_for(p->n_items, 256), 256, 0, r.stream>>>(p->items.p, p->n_items, n, ntiles, vbits, tbits,
                                                                        nitems.p, item_base.p, d.off.p, d.nbr.p, ik.p,
                                                                        ccnt.p, cwords.p);
            launched();
            unsigned long long h_cc[3];
            ccnt.download(h_cc, 3);
            cwords.download(p->cls_words, 3);
            for (int c = 0; c < 3; ++c) p->cls_items[c] = (int64_t)h_cc[c];
            size_t bytes = 0;
            GMSB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, ik.p, ik2.p, p->items.p, items2.p, p->n_items, 0,
                                                      key_bits, r.stream));
            DevBuf<uint8_t> tmp(bytes);
            GMSB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, bytes, ik.p, ik2.p, p->items.p, items2.p, p->n_items, 0,
                                                      key_bits, r.stream));
            r.launches += (uint64_t)((key_bits + 7) / 8 + 1);
            GMSB_CUDA(cudaStreamSynchronize(r.stream));
            p->items = std::move(items2);
        }
        GMSB_CUDA(cudaStreamSynchronize(r.stream));
        tr.mark("plan: item order");
    } catch (...) { delete p; throw; }
    return p;
}

}  // namespace

gmsb_tc_options normalise_tc_options(const gmsb_tc_options *in) { return normalise(in); }

TcPlan &ensure_plan(Graph &g, const gmsb_tc_options &opt) {
    GMSB_REQUIRE(!g.directed, "triangle kernels need an undirected graph");
    GMSB_REQUIRE(opt.variant >= GMSB_TC_AUTO && opt.variant <= GMSB_TC_BITMAP, "tc: bad variant");
    if (!opt.reuse_plan && !g.dag_pinned) { delete g.dag; g.dag = nullptr; }
    if (!g.dag) g.dag = build_degree_dag(g);
    Dag &d = *g.dag;
    // reuse_plan == 2: the oriented representation stays (the FromCGraph analogue), the kernel-specific schedule is rebuilt
    if (d.plan && (opt.reuse_plan == 2 || !same_plan(d.plan->opt, opt))) { delete_plan(d.plan); d.plan = nullptr; }
    if (!d.plan) d.plan = build_plan(d, opt);
    return *d.plan;
}

void tc_total(Graph &g, const gmsb_tc_options &opt_in, uint64_t *out, gmsb_tc_stats *stats) {
    GMSB_REQUIRE(!g.directed, "tc_total: graph must be undirected");
    GMSB_REQUIRE(out != nullptr, "tc_total: null output");
    Runtime &r = rt();
    gmsb_tc_options opt = normalise(&opt_in);
    GMSB_REQUIRE(opt.part_index >= 0 && opt.part_index < opt.part_count, "tc_total: bad partition");
    const uint64_t launches0 = r.launches;
    DevTimer t_orient, t_bm, t_mg, t_gl;

    t_orient.start();
    TcPlan &p = ensure_plan(g, opt);
    Dag &d = *g.dag;
    t_orient.stop();

    DevBuf<unsigned long long> total(1);
    total.zero();
    // the schedule holds this device's share only (the edges into the vertices it owns: ownership does not depend on
    // the order the scatter pass's atomics ran in)
    const int64_t my_items = p.n_items, my_merge = p.n_merge, my_gallop = p.n_gallop;
    // GMSB_TC_TRACE=1: after every counting launch, one line with the triangles it added (read off the running total,
    // so each launch is followed by a synchronisation while tracing)
    const bool trace = std::getenv("GMSB_TC_TRACE") != nullptr;
    unsigned long long traced = 0;
    auto trace_class = [&](const char *cls, const char *unit, int64_t cnt, int words) {
        if (!trace) return;
        const unsigned long long now = total.get(0);
        if (words >= 0)
            std::fprintf(stderr, "[gmsb tc] class=%s %s=%lld words=%d triangles=%llu\n", cls, unit, (long long)cnt,
                         words, now - traced);
        else
            std::fprintf(stderr, "[gmsb tc] class=%s %s=%lld triangles=%llu\n", cls, unit, (long long)cnt, now - traced);
        traced = now;
    };

    t_bm.start();
    if (my_items) {
        GMSB_REQUIRE(p.n_items < (int64_t(1) << 31), "tc: too many bitmap items");
        DevBuf<unsigned int> tickets(3);
        tickets.zero();
        // one persistent wave per window class (the ticket's free is stream-ordered after the kernels)
        auto launch = [&](const char *cls, auto kern, int BLOCK, const Item *items, int64_t cnt, int cap_words,
                          unsigned int *ticket) {
            const int64_t mine = cnt;
            if (mine == 0) return;
            const size_t smem = ((size_t)cap_words + 1) * 4;
            if (smem > 48 * 1024)
                GMSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int resident = 0;
            GMSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, BLOCK, smem));
            GMSB_REQUIRE(resident >= 1, "tc: bitmap kernel does not fit on an SM");
            const int grid = (int)std::min<int64_t>(mine, (int64_t)r.sm_count * resident);
            kern<<<grid, BLOCK, smem, r.stream>>>(items, mine, (uint32_t)cap_words, d.off.p, d.nbr.p,
                                                  p.desc.p, total.p, ticket);
            launched();
            trace_class(cls, "items", mine, cap_words);
        };
        const Item *it0 = p.items.p, *it1 = it0 + p.cls_items[0], *it2 = it1 + p.cls_items[1];
        // small windows (<= 55 KB of bitmap): four CTAs of 512 threads per SM = 64 resident warps; wide: three
        launch("near", k_tc_bitmap2<512, 4, true>, 512, it0, p.cls_items[0], p.cls_words[0], tickets.p);
        launch("small", k_tc_bitmap2<512, 4, false>, 512, it1, p.cls_items[1], p.cls_words[1], tickets.p + 1);
        launch("wide", k_tc_bitmap2<512, 3, false>, 512, it2, p.cls_items[2], p.cls_words[2], tickets.p + 2);
    }
    t_bm.stop();
    t_mg.start();
    if (my_merge) {
        int grid = (int)std::min<int64_t>(ceil_div(my_merge, kMergeWarps), (int64_t)r.sm_count * 16);
        k_tc_merge<<<grid, kMergeWarps * 32, 0, r.stream>>>(p.m_desc.p, p.m_v.p, my_merge, d.off.p, d.nbr.p, total.p);
        launched();
        trace_class("merge", "edges", my_merge, -1);
    }
    t_mg.stop();
    t_gl.start();
    if (my_gallop) {
        int grid = (int)std::min<int64_t>(ceil_div(my_gallop, 8), (int64_t)r.sm_count * 16);
        k_tc_gallop<<<grid, 256, 0, r.stream>>>(p.g_desc.p, p.g_v.p, my_gallop, d.off.p, d.nbr.p, total.p);
        launched();
        trace_class("gallop", "edges", my_gallop, -1);
    }
    t_gl.stop();
    *out = total.get(0);

    if (stats) {
        gmsb_tc_stats s{};
        s.triangles = *out;
        s.algorithmic_bytes = p.algorithmic_bytes;            // every figure of the schedule is this device's share
        s.wedges_checked = p.wedges;
        s.oriented_edges = d.m;
        s.edges_bitmap = p.n_bitmap_edges;                    // this device's share, like bitmap_items
        s.edges_merge = p.n_merge;
        s.edges_gallop = p.n_gallop;
        s.ms_orient = t_orient.ms();
        s.ms_bitmap = t_bm.ms();
        s.ms_merge = t_mg.ms();
        s.ms_gallop = t_gl.ms();
        s.ms_count = s.ms_bitmap + s.ms_merge + s.ms_gallop;
        s.launches = (int32_t)(r.launches - launches0);
        s.max_dplus = d.max_dplus;
        s.bytes_bitmap = p.bytes_bitmap;
        s.bytes_light = p.bytes_kept - p.bytes_bitmap;
        s.wedges_bitmap = p.wedges_bitmap;
        s.bitmap_items = p.n_items;
        s.bitmap_smem_bytes = (p.max_span_words + 1) * 4;
        *stats = s;
    }
    if (!opt.reuse_plan) {
        if (g.dag_pinned) { delete_plan(g.dag->plan); g.dag->plan = nullptr; }
        else { delete g.dag; g.dag = nullptr; }
    }
}

}  // namespace gmsb
