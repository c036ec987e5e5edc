// kclique_lane.cuh — lane-parallel k-clique kernels (included by kclique.cu).
//
// Replaces: KClique::KcListing::listing + Parallelize::{node,edge}
//           (gms/algorithms/non_set_based/k_clique_list/kernels/kclisting.h:92-114,
//            parallelizationStrategy/parallelize.h:39-121).
//
// The warp-cooperative kernels in kclique.cu spend a whole warp on every search-tree node; deep in the tree the
// candidate sets have a few dozen members and most lanes idle.  Here every LANE owns a subtree:
//   * the sub-problem of a vertex u is its |S| x |S| bit matrix (S = N+(u)) in shared memory, rows of 64-bit words
//     with an odd pitch (conflict-free when 32 lanes read the same word of 32 different rows);
//   * 33 <= d+(u) <= 512 : the matrix itself is the compact problem; tasks (second vertex, residue class of the
//     third vertex) are dealt to the lanes of the CTA through a shared ticket;
//   * d+(u) > 512 : the CTA walks the top of the tree together (one AND per level, a handful of barriers) until the
//     candidate set has <= 512 members, re-indexes that set into a second, compact matrix (<= 8 words per row) and
//     deals its tasks to the lanes; with two vertices left the pairs are counted straight off the big matrix;
//   * 129 <= d+(u) <= 512 and four or more vertices left below the second one: a warp re-indexes the second
//     vertex's row once more into its own small matrix (warp_tasks).
// A lane keeps its candidate sets in registers (kclique_lane_core.cuh); only the path is remembered per level, the
// parent's set is recomputed on the way back, so there is no per-lane stack memory at all.
#pragma once
#include "common.cuh"
#include "isect.cuh"
#include "kclique_lane_core.cuh"

namespace gmsb {
namespace lane {

__device__ __forceinline__ int split_for(int c, int block) {
    int sl = 0;
    while (sl < 6 && (c << sl) < 16 * block) ++sl;       // >= 16 tasks per lane keeps the tail short
    return sl;
}

// Lanes of the calling warp(s) pull tasks [0, t_end) of the compact graph cm from *counter (zeroed by the caller) and
// count the `need`-cliques (need >= 3) of those tasks.  Task t = (first member, residue class of the second member,
// kclique_lane_core.cuh): the member is t >> split_log2, or alist[t >> split_log2] when a list of members is given.
// All 32 lanes of every calling warp must be here.  Returns this lane's partial count.
template <int NW>
__device__ __forceinline__ u64 lane_tasks(const u64 *cm, int pitch, unsigned t_end, int need, int split_log2,
                                          unsigned *counter, int lane, const unsigned short *alist) {
    u64 total = 0;
    LaneState<NW> s;
    s.level = -1;
    bool exhausted = false;
    for (;;) {
        const bool want = s.level < 0 && !exhausted;
        const unsigned idle = __ballot_sync(0xffffffffu, want);
        if (idle) {
            const int leader = __ffs(idle) - 1;
            unsigned base = 0;
            if (lane == leader) base = atomicAdd(counter, (unsigned)__popc(idle));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (want) {
                const unsigned t = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
                if (t >= t_end) exhausted = true;
                else {
                    const unsigned m = t >> split_log2;
                    lane_begin<NW>(s, cm, pitch, alist ? (int)alist[m] : (int)m, (int)(t & ((1u << split_log2) - 1u)),
                                   split_log2);
                }
            }
        }
        if (__all_sync(0xffffffffu, s.level < 0)) break;
        if (s.level >= 0) {
            u64 Q[NW];
            if (need == 3) {
#pragma unroll
                for (int w = 0; w < NW; ++w) Q[w] = s.cur[w] & s.stripe;
                total += leaf_pairs<NW>(cm, pitch, Q, s.cur);
                s.level = -1;
            } else {
                if (lane_advance<NW>(s, cm, pitch, need, Q)) total += leaf_pairs<NW>(cm, pitch, Q, Q);
            }
        }
    }
    return total;
}

// Flat form of lane_tasks (kclique_lane_core.cuh: FlatState).  The warp alternates between (1) a refill decision —
// two ballots; lanes that ran dry are refilled together once they are a quarter of the lanes that still have work, or
// nobody has a job, so that the tree walk and the task ticket are paid once per batch of lanes — and (2) a burst of
// kFlatBurst leaf operations per lane with no warp-level bookkeeping in between (a lane that runs dry inside a burst
// idles for at most kFlatBurst - 1 operations).  All 32 lanes of every calling warp must be here.
constexpr int kFlatBurst = 4;
template <int NW>
__device__ __forceinline__ u64 lane_tasks_flat(const u64 *cm, int pitch, unsigned t_end, int need, int split_log2,
                                               unsigned *counter, int lane, const unsigned short *alist) {
    FlatState<NW> s;
    flat_init<NW>(s);
    u64 total = 0;
    for (;;) {
        const bool dry = s.w1 >= NW;                 // a lane with a job always has a member left in s.bits
        const unsigned live = __ballot_sync(0xffffffffu, !dry);
        const unsigned want = __ballot_sync(0xffffffffu, dry && !s.exhausted);
        if (flat_should_refill(__popc(want), __popc(live))) {
            if (dry && !s.exhausted) {
                flat_refill<NW>(s, cm, pitch, need, split_log2, t_end, counter, alist);
                flat_skip<NW>(s);
            }
            continue;
        }
        if (live == 0) break;
        unsigned cnt = 0;
#pragma unroll
        for (int r = 0; r < kFlatBurst; ++r) {
            if (s.w1 < NW) {
                cnt += flat_step<NW>(s, cm, pitch);
                if (s.bits == 0) flat_skip<NW>(s);
            }
        }
        total += cnt;
    }
    return total;
}

// ---- third level: per-warp compact matrix ------------------------------------------------------------------------------
// Deep in the tree the candidate sets hold 3-5 members per 64-bit word of the parent's index space, so every AND +
// popcount there is mostly zeros.  A WARP therefore re-indexes a candidate set of <= kC3Max = 192 members into a
// matrix M3 of its own (rows of 1-3 dense words) and its lanes search M3 with the flat loop; a larger set is expanded
// one member at a time by the warp (one AND per child) until its children fit.  The sets live in the warp's box in
// shared memory, in the index space of the parent matrix cm (<= 8 words).
constexpr int kBoxLevels = 8;                // expansions stop at need == 3 and need <= kMaxNeed = 9: at most 6 deep
struct WarpBox {
    u64 m3[kC3Max * kP3];
    u64 sets[kBoxLevels][8];
    int prefix[8];
    int cursor[kBoxLevels];
    unsigned short list[kC3Max];
    unsigned counter;
    unsigned pad;
};
struct CtaBigRows {                          // members of cm whose row does not fit M3
    unsigned short list[kCMax];
    unsigned count;
    unsigned counter;                        // ticket of the (row, word) units of the second phase
};

// rare fallback: triangles (need == 3) inside a set that is too large for M3, lane per first member, in cm's space
__device__ __forceinline__ u64 lane_triangles_in_set(const u64 *cm, int pitch, int nw, const u64 *set, int lane) {
    u64 total = 0;
#pragma unroll 1
    for (int p = lane; p < nw * 64; p += 32) {
        if (!((set[p >> 6] >> (p & 63)) & 1ull)) continue;
        const u64 *rp = cm + (size_t)p * pitch;
#pragma unroll 1
        for (int w1 = p >> 6; w1 < nw; ++w1) {
            u64 bits = set[w1] & rp[w1];
            while (bits) {
                const int x = (w1 << 6) + __ffsll((long long)bits) - 1;
                bits &= bits - 1;
                const u64 *rx = cm + (size_t)x * pitch;
#pragma unroll 1
                for (int w = w1; w < nw; ++w) total += (u64)__popcll(set[w] & rp[w] & rx[w]);
            }
        }
    }
    return total;
}

// `need`-cliques (need >= 1) among the members of box->sets[level0] (nw valid words, the rest zero), by the whole warp.
// Returns this lane's partial count.
__device__ __forceinline__ u64 warp_set_count(const u64 *cm, int pitch, int nw, WarpBox *box, int level0, int need0, int lane) {
    u64 total = 0;
    int level = level0, need = need0;
    bool fresh = true;
    for (;;) {
        const u64 *set = box->sets[level];
        if (fresh) {
            fresh = false;
            const u64 mine = lane < nw ? set[lane] : 0ull;
            const int pc = __popcll(mine);
            int incl = pc;
#pragma unroll
            for (int o = 1; o < 8; o <<= 1) {
                const int x = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += x;
            }
            const int c = __shfl_sync(0xffffffffu, incl, 7);          // lanes >= nw add 0
            bool expand = false;
            if (c >= need) {
                if (need == 1) {
                    if (lane == 0) total += (u64)c;
                } else if (need == 2) {
                    for (int p = lane; p < nw * 64; p += 32) {
                        if (!((set[p >> 6] >> (p & 63)) & 1ull)) continue;
                        const u64 *rp = cm + (size_t)p * pitch;
                        for (int w = p >> 6; w < nw; ++w) total += (u64)__popcll(set[w] & rp[w]);
                    }
                } else if (c <= kC3Max && need >= 4) {
                    // re-index the set into M3 and search it with the flat lane loop
                    __syncwarp();
                    if (lane == 0) box->counter = 0u;
                    if (lane < 8) box->prefix[lane] = incl - pc;
                    __syncwarp();
                    for (int p = lane; p < nw * 64; p += 32)
                        if ((set[p >> 6] >> (p & 63)) & 1ull)
                            box->list[compact_index(set, box->prefix, p)] = (unsigned short)p;
                    __syncwarp();
                    const int nw3 = (c + 63) >> 6;                    // 1..3 words per row of M3
                    for (int m = lane; m < c; m += 32) {
                        const int pa = box->list[m];
                        compact_row(set, box->prefix, nw, cm + (size_t)pa * pitch, pa, box->m3 + (size_t)m * kP3, nw3);
                    }
                    __syncwarp();
                    const int sl = split_for(c, 32);
                    const unsigned t3 = (unsigned)c << sl;
                    // inside an M3 the alternating loop is the faster one (scale 20, k = 7, 257..512 class: 51.5 s
                    // against 59.2 s with the flat loop: 32 lanes drain a <= 192-member matrix in a few refills, so the
                    // batched refill has little to amortise); the flat loop wins where a CTA's lanes share one matrix
                    total += nw3 == 1   ? lane_tasks<1>(box->m3, kP3, t3, need, sl, &box->counter, lane, nullptr)
                             : nw3 == 2 ? lane_tasks<2>(box->m3, kP3, t3, need, sl, &box->counter, lane, nullptr)
                                        : lane_tasks<3>(box->m3, kP3, t3, need, sl, &box->counter, lane, nullptr);
                    __syncwarp();
                } else if (need == 3 || level + 1 >= kBoxLevels) {
                    // (the second condition cannot occur for need0 <= kMaxNeed; it keeps the stack in bounds)
                    if (need == 3) total += lane_triangles_in_set(cm, pitch, nw, set, lane);
                } else {
                    expand = true;
                }
            }
            if (!expand) {
                if (level == level0) break;
                --level; ++need;
                continue;
            }
            __syncwarp();
            if (lane == 0) box->cursor[level] = -1;
            __syncwarp();
        }
        // next member of this level's set after the cursor (every lane computes the same answer)
        int v = -1;
        {
            const int from = box->cursor[level] + 1;
            int w = from >> 6;
            if (w < nw) {
                u64 m = set[w] & (~0ull << (from & 63));
                while (!m && ++w < nw) m = set[w];
                if (m) v = (w << 6) + __ffsll((long long)m) - 1;
            }
        }
        if (v < 0) {
            if (level == level0) break;
            --level; ++need;
            continue;
        }
        __syncwarp();
        if (lane == 0) box->cursor[level] = v;
        if (lane < 8) box->sets[level + 1][lane] = lane < nw ? (set[lane] & cm[(size_t)v * pitch + lane]) : 0ull;
        __syncwarp();
        ++level; --need;
        fresh = true;
    }
    return total;
}

// `need`-cliques (need >= 5) of the compact graph cm[c][pitch] (nw valid words per row, rows readable — zero padded —
// up to NWP words) by ALL threads of the CTA through per-warp third-level matrices; *counter and *big are zeroed by the
// caller (and a barrier passed).  The members a are dealt to the warps: row a (<= kC3Max members) becomes the warp's
// set with need - 1 vertices left.  Rows that do not fit an M3 go on a list and are searched afterwards in cm itself
// by all lanes of the CTA, 64 residue-class tasks per row.
template <int NWP, bool FLATBIG>
__device__ __forceinline__ u64 count_compact_boxes(const u64 *cm, int pitch, int nw, int c, int need, unsigned *counter,
                                                   WarpBox *box, CtaBigRows *big, int lane) {
    u64 total = 0;
    for (;;) {
        unsigned a = 0;
        if (lane == 0) a = atomicAdd(counter, 1u);
        a = __shfl_sync(0xffffffffu, a, 0);
        if (a >= (unsigned)c) break;
        const u64 *ra = cm + (size_t)a * pitch;
        const u64 mine = lane < nw ? ra[lane] : 0ull;
        int c3 = __popcll(mine);
#pragma unroll
        for (int o = 4; o; o >>= 1) c3 += __shfl_xor_sync(0xffffffffu, c3, o);
        c3 = __shfl_sync(0xffffffffu, c3, 0);             // lanes 0..7 hold the sum of the 8 words
        if (c3 < need - 1) continue;
        if (c3 > kC3Max) {
            if (lane == 0) big->list[atomicAdd(&big->count, 1u)] = (unsigned short)a;
            continue;
        }
        __syncwarp();
        if (lane < 8) box->sets[0][lane] = mine;
        __syncwarp();
        total += warp_set_count(cm, pitch, nw, box, 0, need - 1, lane);
    }
    __syncthreads();
    const unsigned t_end = big->count << 6;
    if constexpr (FLATBIG) total += lane_tasks_flat<NWP>(cm, pitch, t_end, need, 6, &big->counter, lane, big->list);
    else total += lane_tasks<NWP>(cm, pitch, t_end, need, 6, &big->counter, lane, big->list);
    return total;
}

// `need`-cliques (need >= 3) of the compact graph cm[c][pitch] (NW valid words per row) by ALL threads of the CTA:
// per-warp third-level matrices when the rows are long and the search below a member is deep enough to pay for
// another re-indexing (building a matrix below d chosen vertices costs about one operation per (d+2)-clique, the search
// one per (k-1)-clique: it pays for d <= k - 4, i.e. need >= 5 here); else per-lane tasks over every member.
template <int NW>
__device__ __forceinline__ u64 count_compact(const u64 *cm, int pitch, int c, int need, int block, unsigned *counter,
                                             WarpBox *box, CtaBigRows *big, int lane) {
    if constexpr (NW >= 3) {
        if (box && need >= 5) return count_compact_boxes<NW, false>(cm, pitch, NW, c, need, counter, box, big, lane);
    }
    const int sl = split_for(c, block);
    if constexpr (NW <= 2) return lane_tasks_flat<NW>(cm, pitch, (unsigned)c << sl, need, sl, counter, lane, nullptr);
    else return lane_tasks<NW>(cm, pitch, (unsigned)c << sl, need, sl, counter, lane, nullptr);
}

// rows of the bit matrix of S (|S| = D): warp per member i streams N+(S[i]) and looks every element up in S
template <int BLOCK>
__device__ __forceinline__ void build_rows(const vid_t *S, int D, u64 *M, int pitch, const eid_t *__restrict__ off,
                                           const vid_t *__restrict__ nbr, int tid) {
    const int lane = tid & 31, warp = tid >> 5;
    uint32_t *M32 = reinterpret_cast<uint32_t *>(M);
    for (int i = warp; i < D; i += BLOCK / 32) {
        const vid_t vi = S[i];
        const eid_t mb = off[vi];
        const int md = (int)(off[vi + 1] - mb);
        for (int j = lane; j < md; j += 32) {
            const vid_t w = nbr[mb + j];
            int lo = i + 1, hi = D;                     // members after i only (ids ascend with position)
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (S[mid] < w) lo = mid + 1; else hi = mid;
            }
            if (lo < D && S[lo] == w) atomicOr(&M32[(size_t)i * pitch * 2 + (lo >> 5)], 1u << (lo & 31));
        }
    }
}

// ---- 33 <= d+ <= 64*NWB ---------------------------------------------------------------------------------------------
template <int NWB, int BLOCK, int MINB>
__global__ void __launch_bounds__(BLOCK, MINB)
k_kclique_lane_mid(const vid_t *__restrict__ verts, int64_t count, const eid_t *__restrict__ off,
                   const vid_t *__restrict__ nbr, int k, unsigned long long *__restrict__ total,
                   unsigned int *__restrict__ ticket, int pi, int P) {
    constexpr int DMAX = 64 * NWB;
    constexpr int PITCH = pitch_for(NWB);
    __shared__ vid_t S[DMAX];
    __shared__ u64 M[DMAX * PITCH];
    __shared__ unsigned long long red[BLOCK / 32];
    __shared__ unsigned int s_item, s_counter;
    __shared__ CtaBigRows s_big;
    extern __shared__ u64 dyn64[];                  // one WarpBox per warp (classes with rows of >= 3 words)
    const int tid = threadIdx.x, lane = tid & 31;
    WarpBox *box = NWB >= 3 ? reinterpret_cast<WarpBox *>(dyn64) + (tid >> 5) : nullptr;
    u64 acc = 0;
    for (;;) {
        __syncthreads();
        if (tid == 0) { s_item = atomicAdd(ticket, 1u); s_counter = 0; s_big.count = 0; s_big.counter = 0; }
        __syncthreads();
        const int64_t t = pi + (int64_t)s_item * P;
        if (t >= count) break;
        const vid_t u = verts[t];
        const eid_t ob = off[u];
        const int D = (int)(off[u + 1] - ob);
        for (int j = tid; j < D; j += BLOCK) S[j] = nbr[ob + j];
        for (int j = tid; j < D * PITCH; j += BLOCK) M[j] = 0ull;
        __syncthreads();
        build_rows<BLOCK>(S, D, M, PITCH, off, nbr, tid);
        __syncthreads();
        // u is the first clique vertex; k-1 more inside the matrix
        acc += count_compact<NWB>(M, PITCH, D, k - 1, BLOCK, &s_counter, box, &s_big, lane);
    }
    const unsigned long long s = block_sum(acc, red);
    if (tid == 0 && s) atomicAdd(total, s);
}

// ---- d+ > 512 ---------------------------------------------------------------------------------------------------------
constexpr int kStackLevels = 16;

__host__ __device__ inline int huge_pitch(int maxD) { return ((maxD + 63) >> 6) | 1; }
// dynamic shared memory of k_kclique_lane_huge in 64-bit words (matrix included unless it is spilled to global)
__host__ __device__ inline size_t huge_smem_words(int maxD, bool matrix_in_smem) {
    const size_t P1 = (size_t)huge_pitch(maxD);
    return (matrix_in_smem ? (size_t)maxD * P1 : 0) + (size_t)kCMax * pitch_for(8) + (size_t)kStackLevels * P1 +
           (size_t)((maxD + 1) >> 1) + ((P1 + 2) >> 1) + (size_t)(kCMax / 4);
}

// index t of the vertex that work item `item` belongs to: item_base[t] <= item < item_base[t + 1] (item_base is the
// exclusive scan of the items per vertex, nverts + 1 entries)
__device__ __forceinline__ int64_t item_vertex(const int64_t *item_base, int64_t nverts, int64_t item) {
    int64_t lo_t = 0, hi_t = nverts;
    while (hi_t - lo_t > 1) {
        const int64_t mid = (lo_t + hi_t) >> 1;
        if (item_base[mid] <= item) lo_t = mid; else hi_t = mid;
    }
    return lo_t;
}

// The CTA walks the top of the search tree below u and S[i] together (k_kclique_lane_huge, k_kclique_lane_pair).
// M1 is the bit matrix of S (|S| = D, W1 valid words per row, pitch P1); stack[level] = candidates after (level + 2)
// chosen vertices, and the caller has written stack[0] = row i of M1 and passed a barrier.  A set with one or two
// vertices left is counted straight off M1; one of <= kCMax members is re-indexed into the compact matrix M2 and
// counted by the kernel's own step; a larger set is expanded one member at a time.  What differs between the kernels:
//   PAD                 rows of M2 are zero padded from 3..8 words to 4 or 8 (else exactly nwb words);
//   reset()             thread 0, before the barrier that precedes M2: zero the kernel's tickets;
//   count(M2, pitch2, nwb, nwp, c, need, acc)   all threads: acc plus this thread's share of the need-cliques of M2
//                       (c members, nwb valid words per row, nwp readable).
// All threads of the CTA must be here.  Returns acc plus this thread's partial count.
template <int BLOCK, bool PAD, class Reset, class Count>
__device__ __forceinline__ u64 cta_walk(const u64 *M1, int P1, int W1, int D, int k, u64 *stack, u64 *M2, int *prefix,
                                        unsigned short *list, int &s_c, const Reset &reset, const Count &count, u64 acc) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int level = 0;
    bool fresh = true;
    int cursor[kStackLevels];
    for (;;) {
        const u64 *set = stack + (size_t)level * P1;
        if (fresh) {
            fresh = false;
            if (warp == 0) {
                int pc = 0;
                for (int w = lane; w < W1; w += 32) pc += __popcll(set[w]);
                for (int o = 16; o; o >>= 1) pc += __shfl_xor_sync(0xffffffffu, pc, o);
                if (lane == 0) s_c = pc;
            }
            __syncthreads();
            const int c = s_c;
            const int need = k - level - 2;
            bool expand = false;
            if (c >= need) {
                if (need == 1) {
                    if (tid == 0) acc += (u64)c;
                } else if (need == 2) {
                    // pairs straight off the big matrix: thread per member
                    unsigned cnt = 0;
                    for (int p = tid; p < D; p += BLOCK) {
                        const int w0 = p >> 6;
                        if ((set[w0] >> (p & 63)) & 1ull) {
                            const u64 *row = M1 + (size_t)p * P1;
                            for (int w = w0; w < W1; ++w) cnt += (unsigned)__popcll(set[w] & row[w]);
                        }
                    }
                    acc += cnt;
                } else if (c <= kCMax) {
                    // re-index the set into the compact matrix and deal its subtrees to the lanes
                    if (warp == 0) {
                        int carry = 0;
                        for (int base = 0; base < P1; base += 32) {
                            const int w = base + lane;
                            const int v = w < W1 ? __popcll(set[w]) : 0;
                            int incl = v;
                            for (int o = 1; o < 32; o <<= 1) {
                                const int x = __shfl_up_sync(0xffffffffu, incl, o);
                                if (lane >= o) incl += x;
                            }
                            if (w < P1) prefix[w] = carry + incl - v;
                            carry += __shfl_sync(0xffffffffu, incl, 31);
                        }
                    }
                    if (tid == 0) reset();
                    __syncthreads();
                    for (int p = tid; p < D; p += BLOCK)
                        if ((set[p >> 6] >> (p & 63)) & 1ull)
                            list[compact_index(set, prefix, p)] = (unsigned short)p;
                    __syncthreads();
                    const int nwb = (c + 63) >> 6;         // 1..8 words per compact row
                    const int nwp = PAD ? (nwb <= 2 ? nwb : (nwb <= 4 ? 4 : 8)) : nwb;
                    const int pitch2 = pitch_for(nwp);
                    for (int a = tid; a < c; a += BLOCK) {
                        const int pa = list[a];
                        compact_row(set, prefix, W1, M1 + (size_t)pa * P1, pa, M2 + (size_t)a * pitch2, nwp);
                    }
                    __syncthreads();
                    acc = count(M2, pitch2, nwb, nwp, c, need, acc);
                } else {
                    expand = true;
                }
            }
            if (!expand) {
                if (level == 0) break;
                --level;
                continue;
            }
            cursor[level] = -1;
        }
        // next member of this level's set after the cursor (every thread computes the same answer)
        int v = -1;
        {
            const int from = cursor[level] + 1;
            int w = from >> 6;
            if (w < W1) {
                u64 m = set[w] & (~0ull << (from & 63));
                while (!m && ++w < W1) m = set[w];
                if (m) v = (w << 6) + __ffsll((long long)m) - 1;
            }
        }
        if (v < 0) {
            if (level == 0) break;
            --level;
            continue;
        }
        cursor[level] = v;
        __syncthreads();          // everyone is done with the deeper levels before they are overwritten
        u64 *child = stack + (size_t)(level + 1) * P1;
        for (int w = tid; w < P1; w += BLOCK) child[w] = set[w] & M1[(size_t)v * P1 + w];
        __syncthreads();
        ++level;
        fresh = true;
    }
    return acc;
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK, 1)
k_kclique_lane_huge(const vid_t *__restrict__ verts, const int64_t *__restrict__ item_base, int64_t nverts,
                    int64_t count, const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int k, int maxD,
                    unsigned long long *__restrict__ total, unsigned int *__restrict__ ticket,
                    u64 *__restrict__ spill, int pi, int P) {
    extern __shared__ u64 smem64[];
    const int P1 = huge_pitch(maxD);
    u64 *M1 = spill ? spill + (size_t)blockIdx.x * ((size_t)maxD * P1) : smem64;
    u64 *sp = smem64 + (spill ? 0 : (size_t)maxD * P1);
    u64 *M2 = sp;                  sp += (size_t)kCMax * pitch_for(8);
    u64 *stack = sp;               sp += (size_t)kStackLevels * P1;
    vid_t *S = reinterpret_cast<vid_t *>(sp);            sp += (maxD + 1) >> 1;
    int *prefix = reinterpret_cast<int *>(sp);           sp += (P1 + 2) >> 1;
    unsigned short *list = reinterpret_cast<unsigned short *>(sp);
    __shared__ unsigned long long red[BLOCK / 32];
    __shared__ unsigned int s_item, s_counter;
    __shared__ int s_c;
    const int tid = threadIdx.x, lane = tid & 31;
    // compact step: rows of exactly nwb words, per-lane tasks over every member
    auto reset = [&] { s_counter = 0; };
    auto count_m2 = [&](const u64 *M2, int pitch2, int nwb, int, int c, int need, u64 acc) {
        const int sl = split_for(c, BLOCK);
        switch (nwb) {
            case 1: acc += lane_tasks<1>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
            case 2: acc += lane_tasks<2>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
            case 3: acc += lane_tasks<3>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
            case 4: acc += lane_tasks<4>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
            case 5: acc += lane_tasks<5>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
            case 6: acc += lane_tasks<6>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
            case 7: acc += lane_tasks<7>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
            default: acc += lane_tasks<8>(M2, pitch2, (unsigned)c << sl, need, sl, &s_counter, lane, nullptr); break;
        }
        return acc;
    };
    u64 acc = 0;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(ticket, 1u);
        __syncthreads();
        const int64_t item = pi + (int64_t)s_item * P;
        if (item >= count) break;
        const int64_t t = item_vertex(item_base, nverts, item);
        const int part = (int)(item - item_base[t]), nparts = (int)(item_base[t + 1] - item_base[t]);
        const vid_t u = verts[t];
        const eid_t ob = off[u];
        const int D = (int)(off[u + 1] - ob);
        const int W1 = (D + 63) >> 6;
        for (int j = tid; j < D; j += BLOCK) S[j] = nbr[ob + j];
        for (size_t j = tid; j < (size_t)D * P1; j += BLOCK) M1[j] = 0ull;
        __syncthreads();
        build_rows<BLOCK>(S, D, M1, P1, off, nbr, tid);
        for (int i = part; i < D; i += nparts) {
            __syncthreads();
            for (int w = tid; w < P1; w += BLOCK) stack[w] = M1[(size_t)i * P1 + w];
            __syncthreads();
            acc = cta_walk<BLOCK, false>(M1, P1, W1, D, k, stack, M2, prefix, list, s_c, reset, count_m2, acc);
        }
    }
    const unsigned long long s = block_sum(acc, red);
    if (tid == 0 && s) atomicAdd(total, s);
}

// ---- d+ > 512, decoupled (round 2) -------------------------------------------------------------------------------------
// k_kclique_lane_huge keeps the vertex's big matrix M1 in shared memory (up to 142 KB at scale 22), which leaves room
// for one CTA per SM and nothing for per-warp third-level matrices.  Here the two jobs are separated:
//   phase 1  k_kclique_m1_build   M1 of every d+ > 128 vertex is written to global memory (0.5 GB at scale 22; the
//                                 rows a CTA needs stay in the L2);
//   phase 2  k_kclique_lane_pair  (k >= 7: at least five vertices left below u and S[i], so that third-level matrices
//                                 pay) work item = (vertex u, member i): the CTA reads row i of M1 — the candidates after
//                                 choosing u and S[i] —, walks further down together only while that set has more than
//                                 512 members, re-indexes it into a compact matrix M2 in shared memory and counts in
//                                 M2 exactly as the 257..512 class does (count_compact: per-warp M3 boxes, flat lanes).
// Shared memory per CTA is M2 + boxes (~85 KB at 256 threads): two CTAs per SM, items ~100x finer than a vertex
// part, and no limit on d+ other than the memory for M1.
__host__ __device__ inline size_t pair_smem_words(int maxD, int warps) {
    const size_t P1 = (size_t)huge_pitch(maxD);
    return (size_t)kCMax * pitch_for(8) + (size_t)kStackLevels * P1 + ((P1 + 2) >> 1) + (size_t)(kCMax / 4) +
           (size_t)warps * ((sizeof(WarpBox) + 7) / 8);
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK)
k_kclique_m1_build(const vid_t *__restrict__ verts, int64_t first, int64_t nverts, const eid_t *__restrict__ off,
                   const vid_t *__restrict__ nbr, const int64_t *__restrict__ m1_off, u64 *__restrict__ m1, int maxD) {
    extern __shared__ u64 smem64[];
    const int P1max = huge_pitch(maxD);
    constexpr int NWARPS = BLOCK / 32;
    u64 *rowbuf = smem64;                                               // NWARPS x P1max
    vid_t *S = reinterpret_cast<vid_t *>(smem64 + (size_t)NWARPS * P1max);   // maxD
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int64_t t = blockIdx.x; t < nverts; t += gridDim.x) {
        const vid_t u = verts[first + t];
        const eid_t ob = off[u];
        const int D = (int)(off[u + 1] - ob);
        const int P1 = huge_pitch(D);
        u64 *M1 = m1 + m1_off[t];
        __syncthreads();
        for (int j = tid; j < D; j += BLOCK) S[j] = nbr[ob + j];
        __syncthreads();
        u64 *rb = rowbuf + (size_t)warp * P1max;
        uint32_t *rb32 = reinterpret_cast<uint32_t *>(rb);
        for (int i = warp; i < D; i += NWARPS) {
            for (int w = lane; w < P1; w += 32) rb[w] = 0ull;
            __syncwarp();
            const vid_t vi = S[i];
            const eid_t mb = off[vi];
            const int md = (int)(off[vi + 1] - mb);
            for (int j = lane; j < md; j += 32) {
                const vid_t w = nbr[mb + j];
                int lo = i + 1, hi = D;                     // members after i only (ids ascend with position)
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (S[mid] < w) lo = mid + 1; else hi = mid;
                }
                if (lo < D && S[lo] == w) atomicOr(&rb32[lo >> 5], 1u << (lo & 31));
            }
            __syncwarp();
            for (int w = lane; w < P1; w += 32) M1[(size_t)i * P1 + w] = rb[w];
            __syncwarp();
        }
    }
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK, 2)
k_kclique_lane_pair(const vid_t *__restrict__ verts, int64_t first, const int64_t *__restrict__ item_base,
                    int64_t nverts, int64_t count, const eid_t *__restrict__ off, const int64_t *__restrict__ m1_off,
                    const u64 *__restrict__ m1, int k, int maxD, unsigned long long *__restrict__ total,
                    unsigned int *__restrict__ ticket, int pi, int P) {
    extern __shared__ u64 smem64[];
    const int P1max = huge_pitch(maxD);
    u64 *sp = smem64;
    u64 *M2 = sp;                  sp += (size_t)kCMax * pitch_for(8);
    u64 *stack = sp;               sp += (size_t)kStackLevels * P1max;
    int *prefix = reinterpret_cast<int *>(sp);           sp += (P1max + 2) >> 1;
    unsigned short *list = reinterpret_cast<unsigned short *>(sp);    sp += kCMax / 4;
    __shared__ unsigned long long red[BLOCK / 32];
    __shared__ unsigned int s_item, s_counter;
    __shared__ int s_c;
    __shared__ CtaBigRows s_big;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    WarpBox *box = reinterpret_cast<WarpBox *>(sp) + warp;
    // compact step: rows padded to 4 or 8 words; per-warp M3 boxes where five or more vertices are left, else flat lanes
    auto reset = [&] { s_counter = 0; s_big.count = 0; s_big.counter = 0; };
    auto count_m2 = [&](const u64 *M2, int pitch2, int nwb, int nwp, int c, int need, u64 acc) {
        if (nwp == 8 && need >= 5) {
            acc += count_compact_boxes<8, true>(M2, pitch2, nwb, c, need, &s_counter, box, &s_big, lane);
        } else if (nwp == 4 && need >= 5) {
            acc += count_compact_boxes<4, true>(M2, pitch2, nwb, c, need, &s_counter, box, &s_big, lane);
        } else if (nwp >= 4) {       // too shallow for another re-indexing: flat lanes on M2 itself
            const int sl = split_for(c, BLOCK);
            const unsigned t_end = (unsigned)c << sl;
            acc += nwp == 4 ? lane_tasks_flat<4>(M2, pitch2, t_end, need, sl, &s_counter, lane, nullptr)
                            : lane_tasks_flat<8>(M2, pitch2, t_end, need, sl, &s_counter, lane, nullptr);
        } else {
            const int sl = split_for(c, BLOCK);
            const unsigned t_end = (unsigned)c << sl;
            acc += nwb == 1 ? lane_tasks_flat<1>(M2, pitch2, t_end, need, sl, &s_counter, lane, nullptr)
                            : lane_tasks_flat<2>(M2, pitch2, t_end, need, sl, &s_counter, lane, nullptr);
        }
        return acc;
    };
    u64 acc = 0;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(ticket, 1u);
        __syncthreads();
        const int64_t item = pi + (int64_t)s_item * P;
        if (item >= count) break;
        const int64_t t = item_vertex(item_base, nverts, item);
        const int i = (int)(item - item_base[t]);
        const vid_t u = verts[first + t];
        const int D = (int)(off[u + 1] - off[u]);
        const int P1 = huge_pitch(D), W1 = (D + 63) >> 6;
        const u64 *__restrict__ M1 = m1 + m1_off[t];
        for (int w = tid; w < P1; w += BLOCK) stack[w] = M1[(size_t)i * P1 + w];
        __syncthreads();
        // the CTA walks down together while the candidate set has more than 512 members
        acc = cta_walk<BLOCK, true>(M1, P1, W1, D, k, stack, M2, prefix, list, s_c, reset, count_m2, acc);
    }
    const unsigned long long s = block_sum(acc, red);
    if (tid == 0 && s) atomicAdd(total, s);
}

}  // namespace lane
}  // namespace gmsb
