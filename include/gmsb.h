/*
 * gmsb.h — C ABI of gms-b200: the B200-native replacement for GraphMineSuite's set-intersection hot path.
 *
 * GMS (spcl/gms) is header-only C++ and has no ABI of its own (SURVEY.md §8b); the entry points below are what a
 * binding for this path has to reach, one per reference interface that is replaced.  Citations are
 * file:line relative to the reference tree.  The C++ facade in include/gms_b200/ wraps these in GMS-named
 * templates (CudaSetGraph, GMS::TriangleCount::Par::count_total, ...); INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every function returns 0 on success or a negative gmsb_status; gmsb_last_error() gives the message of the
 *     last failure on the calling thread;
 *   - handles are opaque; all array arguments are HOST pointers owned by the caller unless the name ends in
 *     `_device` (then they are device pointers on the current device);
 *   - vertex ids are int32 (gms/common/types.h:9), offsets int64, counts uint64 / int64 as in the reference;
 *   - one host thread per handle at a time; handles live on the process's primary device (gmsb_set_device) and the
 *     library launches on the stream given by gmsb_set_stream (default: the legacy stream 0); the *_multi entry
 *     points spread one call over the devices of gmsb_set_devices;
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry point fails with
 *     GMSB_ERR_CUDA.
 */
#ifndef GMSB_H_
#define GMSB_H_

#include <stdint.h>

#if defined(__GNUC__)
#define GMSB_API __attribute__((visibility("default")))
#else
#define GMSB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gmsb_graph_s *gmsb_graph_t;

typedef enum {
    GMSB_OK = 0,
    GMSB_ERR_INVALID = -1,   /* bad argument (null pointer, negative size, directed graph where undirected needed) */
    GMSB_ERR_CUDA = -2,      /* CUDA runtime failure, incl. "no device" */
    GMSB_ERR_OOM = -3,
    GMSB_ERR_UNSUPPORTED = -4
} gmsb_status;

/* ---- runtime -------------------------------------------------------------------------------------------- */
GMSB_API const char *gmsb_last_error(void);
GMSB_API int gmsb_version(void);
GMSB_API int gmsb_device_count(int *count);
GMSB_API int gmsb_set_device(int device);
GMSB_API int gmsb_set_stream(void *cuda_stream);            /* cudaStream_t; NULL = legacy default stream */
GMSB_API int gmsb_synchronize(void);
/* Device memory is cached in size-class free lists between calls (driver allocation of GBs costs more than the
 * kernels); this returns every cached block to the driver. */
GMSB_API int gmsb_trim_memory(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
GMSB_API int gmsb_launch_count(uint64_t *count);

/* ---- several GPUs in one process ------------------------------------------------------------------------------ */
/* gmsb_set_devices(n, ids): the devices the *_multi entry points below work on; ids[0] becomes the process's primary
 * device, where graph handles live.  The handle's CSR is replicated to the other devices over NVLink on first use
 * (cached), one host thread per device runs the partitioned kernels, scalar counts are summed on the host and array
 * results go through NCCL (libnccl.so.2, loaded on first use): vertex_count2 is one ncclAllReduce(int64[n]), the
 * per-edge similarity one ncclAllReduce(uint32[m]) of the edge supports followed by edge-partitioned scoring
 * (SURVEY.md 8e).  Same results as the single-device entry points. */
GMSB_API int gmsb_set_devices(int n, const int *ids);
GMSB_API int gmsb_tc_total_multi(gmsb_graph_t g, uint64_t *out);
GMSB_API int gmsb_tc_vertex2_multi(gmsb_graph_t g, int64_t *out_n);
GMSB_API int gmsb_kclique_count_multi(gmsb_graph_t g, int k, uint64_t *out);
GMSB_API int gmsb_edge_similarity_multi(gmsb_graph_t g, int metric, double *out, int64_t *m_out);

/* ---- synthetic inputs (host side; input preparation, never timed) ---------------------------------------------- */
/* Generator::MakeRMatEL + PermuteIDs                    gms/third_party/gapbs/generator.h:81-114,52-62
 * m edges of a 2^scale-vertex R-MAT graph, mt19937 reseeded with 27491095 + block every 2^18 edges; the reference's
 * "kronecker" is a=.57 b=.19 c=.19 with permute=1. Bit-identical to the reference for those constants. */
GMSB_API int gmsb_generate_rmat(int scale, int64_t m, float a, float b, float c, int permute, int32_t *src,
                                int32_t *dst);
/* Generator::MakeUniformEL                              gms/third_party/gapbs/generator.h:64-79 */
GMSB_API int gmsb_generate_uniform(int scale, int64_t m, int32_t *src, int32_t *dst);

/* ---- graph construction (replaces gapbs CSRGraph / Builder + SetGraph::FromCGraph) ---------------------------- */
/* SetGraph<Set>::FromCGraph(const CSRGraph&)            gms/representations/graphs/set_graph.h:87-89,153-181
 * Lists must be ascending and duplicate-free (what SquishGraph leaves, gapbs/builder.h:206-235). */
GMSB_API int gmsb_graph_from_csr(int64_t n, const int64_t *offsets, const int32_t *nbrs, int directed, gmsb_graph_t *out);
GMSB_API int gmsb_graph_from_csr_device(int64_t n, const int64_t *offsets, const int32_t *nbrs, int directed,
                               gmsb_graph_t *out);
/* Same, with construction flags.  GMSB_BUILD_ORIENT (undirected graphs): the degree-oriented representation that
 * the triangle / clique / similarity entry points work on is built together with the graph — BenchmarkKernelBk calls
 * SGraph::FromCGraph once and then the kernel (gms/common/benchmark.h:105-118); here the upload of the host arrays is
 * chunked and the ranking, validation and relabelling passes run on the chunks that have already arrived.  Use pinned
 * host memory for the copies to overlap. */
typedef enum { GMSB_BUILD_DEFAULT = 0, GMSB_BUILD_ORIENT = 1 } gmsb_build_flags;
GMSB_API int gmsb_graph_from_csr_ex(int64_t n, const int64_t *offsets, const int32_t *nbrs, int directed, int flags,
                                    gmsb_graph_t *out);
/* Sharded form of the same construction for one process per device (torchrun ranks, MPI ranks): SURVEY.md 8e keeps the
 * CSR replicated, but what the triangle kernels read is the ORIENTED representation only, so each device uploads and
 * orients one vertex range and the finished rows are exchanged instead of the host arrays being read N times.
 *   gmsb_shard_begin   device part_index of part_count uploads the offsets and the neighbour slots of its vertex range
 *                      (ranges of equal slot counts), ranks the vertices (PpParallel::getDegreeOrdering), keeps each
 *                      row's higher-ranked neighbours, relabelled and sorted; *piece_len = entries of its piece.
 *                      offsets_dev (may be NULL): the complete offsets already on this device — a caller that uploads
 *                      1/part_count of them per device and all-gathers saves (part_count - 1) x 8(n+1) bytes of host
 *                      traffic; `offsets` (host) is then read at a handful of positions only
 *   gmsb_shard_export  writes the piece (rows packed in original-id order) to piece_dev and d+ of the range's vertices
 *                      to dplus_all_dev[range] (an int32[n] the caller zeroed)
 *   (caller)           all-gather of the pieces into pieces_dev[part * piece_stride ...], piece_stride >= every
 *                      piece_len; all-reduce(sum) of dplus_all_dev
 *   gmsb_shard_finish  rows into rank order; the handle it returns answers gmsb_tc_total[_ex] / gmsb_tc_vertex2 and the
 *                      size queries — its symmetric lists are incomplete, every other operator returns GMSB_ERR_INVALID
 * Lists longer than 8192 after orientation are not supported here (GMSB_ERR_INVALID): use gmsb_graph_from_csr_ex. */
typedef struct gmsb_shard_s *gmsb_shard_t;
GMSB_API int gmsb_shard_begin(int64_t n, const int64_t *offsets, const int32_t *nbrs, const int64_t *offsets_dev,
                              int part_index, int part_count, gmsb_shard_t *out, int64_t *piece_len);
GMSB_API int gmsb_shard_export(gmsb_shard_t s, int32_t *piece_dev, int32_t *dplus_all_dev);
GMSB_API int gmsb_shard_finish(gmsb_shard_t s, const int32_t *pieces_dev, int64_t piece_stride, const int32_t *dplus_all_dev,
                               gmsb_graph_t *out);
GMSB_API int gmsb_shard_free(gmsb_shard_t s);
/* BuilderBase::MakeGraphFromEL + SquishGraph            gms/third_party/gapbs/builder.h:279-298,237-251
 * n = max id + 1; symmetrize inserts both directions; lists sorted, de-duplicated, self loops removed —
 * done by an on-GPU radix sort of 64-bit (u<<32|v) keys. */
GMSB_API int gmsb_graph_from_edgelist(int64_t m, const int32_t *src, const int32_t *dst, int symmetrize, gmsb_graph_t *out);
GMSB_API int gmsb_graph_from_edgelist_device(int64_t m, const int32_t *src, const int32_t *dst, int symmetrize,
                                    gmsb_graph_t *out);
/* BuilderBase::RelabelByDegree (degree desc, id desc)   gms/third_party/gapbs/builder.h:1699-1735 */
GMSB_API int gmsb_graph_relabel_by_degree(gmsb_graph_t g, gmsb_graph_t *out);
GMSB_API int gmsb_graph_num_nodes(gmsb_graph_t g, int64_t *n);
GMSB_API int gmsb_graph_num_slots(gmsb_graph_t g, int64_t *slots);     /* CSR entries: 2m undirected, m directed */
GMSB_API int gmsb_graph_is_directed(gmsb_graph_t g, int *directed);
GMSB_API int gmsb_graph_export_csr(gmsb_graph_t g, int64_t *offsets, int32_t *nbrs);
GMSB_API int gmsb_graph_free(gmsb_graph_t g);

/* ---- preprocessing: orderings and orientation ------------------------------------------------------------------- */
/* PpParallel::getDegreeOrdering<G,useRankFormat>        gms/algorithms/preprocessing/parallel/degree.h:26-61
 * (degree asc, id asc); rank_format=0: out[i] = vertex at position i; 1: out[v] = position of v. */
GMSB_API int gmsb_order_degree(gmsb_graph_t g, int rank_format, int32_t *out);
/* PpSequential::getDegeneracyOrderingDanischHeap        gms/algorithms/preprocessing/sequential/degeneracy_danisch.h:12-56
 * a valid min-degree-peeling order in the reference's convention rank = n - (removal index); ties are
 * implementation-defined in the reference too. */
GMSB_API int gmsb_order_degeneracy(gmsb_graph_t g, int32_t *out_rank);
/* PpParallel::getDegeneracyOrderingApproxCGraph<boundary_function::averageDegree, useRankFormat>(g, out, epsilon)
 *                                                       gms/algorithms/preprocessing/parallel/degeneracy_approx_csr.h:13-78
 * rounds remove every vertex with residual degree <= (1+eps)*average; inside a round vertices are ordered by that
 * degree (ties by id; unspecified in the reference). Ascending convention: first removed = position / rank 0. */
GMSB_API int gmsb_order_degeneracy_approx(gmsb_graph_t g, double epsilon, int rank_format, int32_t *out);
/* Core number of every vertex: the largest k such that v belongs to the k-core (the maximal subgraph of minimum
 * degree >= k); 0 for an isolated vertex; max over v = the degeneracy.  Undirected graphs only.  GMS has no per-vertex
 * core numbers (its verifiers report the maximum of an order); the value is what the peel of gmsb_order_degeneracy
 * reaches when it removes the vertex. */
GMSB_API int gmsb_core_numbers(gmsb_graph_t g, int32_t *out_n);
/* Truss number of every undirected edge a<b, in the CSR order of gmsb_edge_similarity: the largest k such that the
 * edge belongs to the k-truss (the maximal subgraph in which every edge lies in >= k-2 triangles of the subgraph);
 * 2 for an edge in no triangle.  Two-pass like gmsb_edge_similarity: out may be NULL, *m_out = number of edges.
 * Undirected graphs with fewer than 2^31 edges only (GMSB_ERR_INVALID otherwise). */
GMSB_API int gmsb_truss_numbers(gmsb_graph_t g, int32_t *out, int64_t *m_out);
/* getDegeneracyOrderingApprox{CGraph,SGraph}<boundary, useRankFormat>
 *                                                       degeneracy_approx_csr.h:13-78 (push), degeneracy_approx_set.h:14-85 (pull)
 * boundary = one of boundary_function::{averageDegree, minDegree, probMinDegree, probMedianDegree}
 * (boundary_function.h:15-91).  pull = 1 is the Set form: every remaining vertex subtracts |N(v) ∩ X|, X the set removed
 * in the round, one intersect_count per vertex against the shared set X.  Push and pull give the same order.  The two
 * sampled rules draw with WyRand from `seed` (the reference seeds from the clock: not reproducible there). */
typedef enum { GMSB_ADG_AVERAGE = 0, GMSB_ADG_MIN = 1, GMSB_ADG_PROB_MIN = 2, GMSB_ADG_PROB_MEDIAN = 3 } gmsb_adg_boundary;
GMSB_API int gmsb_order_degeneracy_approx_ex(gmsb_graph_t g, double epsilon, int rank_format, int boundary, int pull,
                                             uint64_t seed, int32_t *out);
/* WorthRelabelling(g): the CLI's auto-relabel heuristic    gms/third_party/gapbs/benchmark.h:158-176, cli/cli.h:174-181
 * (average degree >= 10 and mean/1.3 > median over 1000 mt19937-sampled non-isolated vertices). */
GMSB_API int gmsb_graph_worth_relabelling(gmsb_graph_t g, int *out);
/* PpSequential::InduceDirectedGraph(g, ranking)         gms/algorithms/preprocessing/sequential/apply_order.h:10-35
 * relabels u -> ranking[u], keeps rank(u) < rank(v); result n = max surviving id + 1. Fails with
 * GMSB_ERR_INVALID on a directed input (the reference throws std::invalid_argument, :14-16). */
GMSB_API int gmsb_orient(gmsb_graph_t g, const int32_t *ranking, gmsb_graph_t *dag);

/* ---- triangle counting --------------------------------------------------------------------------------------------- */
/* TriangleCount::{Seq,Par}::count_total                 gms/algorithms/set_based/triangle_count/parallel/total.h:8-24 */
GMSB_API int gmsb_tc_total(gmsb_graph_t g, uint64_t *out);

/* Which intersection kernel handles an oriented edge (u,v). AUTO picks per edge: the shared-memory bitmap kernel
 * when v is a hub, else merge-path or galloping by the length ratio of the two lists. */
typedef enum { GMSB_TC_AUTO = 0, GMSB_TC_MERGE = 1, GMSB_TC_GALLOP = 2, GMSB_TC_BITMAP = 3 } gmsb_tc_variant;

typedef struct {
    int32_t variant;         /* gmsb_tc_variant */
    int32_t part_index;      /* this process handles share part_index of part_count of the oriented edges:  */
    int32_t part_count;      /* those whose closing vertex it owns (vertices dealt from the top of the degree
                                order; the schedule is built for the share only); 0 or 1 = all                */
    int32_t reuse_plan;      /* 0: build the oriented DAG and the schedule for this call and drop them; 1: keep
                                both cached on the handle between calls; 2: keep the DAG (the FromCGraph analogue),
                                rebuild the kernel-specific schedule on every call                             */
    int32_t hub_bitmap_bits; /* bitmap kernel's shared-memory window in bits; 0 = default                     */
    int32_t gallop_ratio;    /* galloping when longer/shorter >= ratio; 0 = default                           */
    int64_t hub_min_work;    /* a vertex is a hub when its incoming wedge work >= this; 0 = default            */
    int32_t reserved[4];     /* [0..2] must be 0.  [3] = form of the schedule's two passes over the edges:
                                0 = chosen from part_count (element-wise from 4 parts on), 2 = walk the rows,
                                3 = element-wise over the edge slots.  Both forms build the same schedule.
                                Other values fail with GMSB_ERR_INVALID.                                      */
} gmsb_tc_options;

typedef struct {
    uint64_t triangles;        /* this part's count (sum over parts = total)                                   */
    uint64_t algorithmic_bytes;/* B_TC share: sum over this part's oriented edges of 4*(d+(u)+d+(v))            */
    uint64_t wedges_checked;   /* list elements actually probed (this part)                                    */
    int64_t oriented_edges;    /* |E+| of the whole graph                                                       */
    int64_t edges_bitmap, edges_merge, edges_gallop;   /* this part's edges by kernel                          */
    double ms_orient;          /* device ms: degree ranking + DAG build + schedule                              */
    double ms_count;           /* device ms: all counting kernels                                               */
    double ms_bitmap, ms_merge, ms_gallop;             /* per-kernel device ms (launched back to back)          */
    int32_t launches;          /* kernels launched by this call                                                 */
    int32_t max_dplus;
    uint64_t bytes_bitmap;     /* algorithmic bytes of the edges the bitmap kernel handles (this part)          */
    uint64_t bytes_light;      /* ... of the edges the merge + gallop kernels handle                            */
    uint64_t wedges_bitmap;    /* list elements the bitmap kernel probes (this part)                            */
    int64_t bitmap_items;      /* work items of the bitmap kernel (this part)                                   */
    int32_t bitmap_smem_bytes; /* dynamic shared memory per CTA of the bitmap kernel                            */
    int32_t reserved;
} gmsb_tc_stats;

GMSB_API int gmsb_tc_total_ex(gmsb_graph_t g, const gmsb_tc_options *opt, uint64_t *out, gmsb_tc_stats *stats);

/* TriangleCount::{Seq,Par}::vertex_count2 (= 2*t(u))    gms/algorithms/set_based/triangle_count/parallel/vertex.h:15-49 */
GMSB_API int gmsb_tc_vertex2(gmsb_graph_t g, int64_t *out_n);

/* ---- batched Set algebra (SortedSet::intersect_count / intersect / difference / union on neighbourhoods) -------- */
/* SortedSetBase::intersect_count                        gms/representations/sets/sorted_set.h:176-182
 * out[i] = |N(a[i]) ∩ N(b[i])| */
GMSB_API int gmsb_intersect_count_batch(gmsb_graph_t g, int64_t npairs, const int32_t *a, const int32_t *b, uint64_t *out);
/* SortedSetBase::intersect                              gms/representations/sets/sorted_set.h:160-166
 * two-pass: out_offsets[npairs+1] always written; out_elems may be NULL to size the result first. */
GMSB_API int gmsb_intersect_batch(gmsb_graph_t g, int64_t npairs, const int32_t *a, const int32_t *b, int64_t *out_offsets,
                         int32_t *out_elems, int64_t out_capacity);

/* SortedSetBase::difference(const Set&)                 gms/representations/sets/sorted_set.h:184-189
 * N(a[i]) \ N(b[i]), ascending; same two-pass protocol as gmsb_intersect_batch. */
GMSB_API int gmsb_difference_batch(gmsb_graph_t g, int64_t npairs, const int32_t *a, const int32_t *b, int64_t *out_offsets,
                          int32_t *out_elems, int64_t out_capacity);
/* SortedSetBase::union_with(const Set&)                 gms/representations/sets/sorted_set.h:104-109
 * N(a[i]) ∪ N(b[i]), ascending; same two-pass protocol. */
GMSB_API int gmsb_union_batch(gmsb_graph_t g, int64_t npairs, const int32_t *a, const int32_t *b, int64_t *out_offsets,
                     int32_t *out_elems, int64_t out_capacity);
/* SortedSetBase::union_count                            gms/representations/sets/sorted_set.h:140
 * out[i] = |N(a[i]) ∪ N(b[i])| */
GMSB_API int gmsb_union_count_batch(gmsb_graph_t g, int64_t npairs, const int32_t *a, const int32_t *b, uint64_t *out);

/* ---- device-resident sets: the Set concept as an object -------------------------------------------------------------- */
/* SortedSetBase<int32_t> / SortedSetRefBase<int32_t>        gms/representations/sets/sorted_set.h:22-270, sorted_set_ref.h:10-80
 * An ascending, duplicate-free int32 set in device memory.  Binary operations take set HANDLES and leave their result
 * on the device, so chains like Bron-Kerbosch's P ∩ N(v), X ∩ N(v), P \ {v} (maximal_clique_enum/sequential/tomita.h)
 * never return to the host.  include/gms_b200/cuda_sorted_set.hpp wraps these in a move-only class with the
 * reference's member names. */
typedef struct gmsb_set_s *gmsb_set_t;
typedef enum { GMSB_SET_INTERSECT = 0, GMSB_SET_UNION = 1, GMSB_SET_DIFFERENCE = 2 } gmsb_set_op_kind;
/* SortedSetBase(const SetElement*, size_t): sorts what it is given   sorted_set.h:64-66 */
GMSB_API int gmsb_set_from_host(const int32_t *elems, int64_t count, gmsb_set_t *out);
/* SortedSetBase::Range(bound) = {0 .. bound-1}                       sorted_set.h:246-251 */
GMSB_API int gmsb_set_range(int64_t bound, gmsb_set_t *out);
/* SetGraph::out_neigh(v) as a borrowed view of the graph's CSR (SortedSetRef); the graph must outlive the view.
 * Modifying operations on a view first turn it into an owning set. */
GMSB_API int gmsb_set_neighbourhood(gmsb_graph_t g, int32_t v, gmsb_set_t *out);
GMSB_API int gmsb_set_clone(gmsb_set_t a, gmsb_set_t *out);                          /* sorted_set.h:245 */
GMSB_API int gmsb_set_free(gmsb_set_t a);
GMSB_API int gmsb_set_cardinality(gmsb_set_t a, int64_t *n);                         /* sorted_set.h:253 */
GMSB_API int gmsb_set_to_host(gmsb_set_t a, int32_t *out);                           /* toArray, sorted_set.h:258-262 */
GMSB_API int gmsb_set_contains(gmsb_set_t a, int32_t x, int *flag);                  /* sorted_set.h:216-220 */
GMSB_API int gmsb_set_add(gmsb_set_t a, int32_t x);                                  /* add / union_inplace(elem) :222-231 */
GMSB_API int gmsb_set_remove(gmsb_set_t a, int32_t x);                               /* remove / difference_inplace(elem) :233-243 */
GMSB_API int gmsb_set_equal(gmsb_set_t a, gmsb_set_t b, int *flag);                  /* operator== :255 */
/* a op b as a new device set: intersect :160-166, union_with :104-109, difference :184-189 */
GMSB_API int gmsb_set_op(int op, gmsb_set_t a, gmsb_set_t b, gmsb_set_t *out);
/* a <- a op b: intersect_inplace :168-174, union_inplace :118-124, difference_inplace :198-204 */
GMSB_API int gmsb_set_op_inplace(int op, gmsb_set_t a, gmsb_set_t b);
/* |a op b|: intersect_count :176-182, union_count :140 */
GMSB_API int gmsb_set_op_count(int op, gmsb_set_t a, gmsb_set_t b, uint64_t *out);
/* one left set against a batch of right sets, one launch: out[i] = |a op bs[i]| / outs[i] = a op bs[i] (device sets) */
GMSB_API int gmsb_set_op_count_many(int op, gmsb_set_t a, int64_t count, const gmsb_set_t *bs, uint64_t *out);
GMSB_API int gmsb_set_op_many(int op, gmsb_set_t a, int64_t count, const gmsb_set_t *bs, gmsb_set_t *outs);
/* out[i] = |a op N(members[i])| for every member of the set `members` (ascending): the pivot scoring loop of Tomita's
 * Bron-Kerbosch (tomita.h:17-31, cand.intersect_count(graph.out_neigh(v))) and the pull step of the approximate
 * degeneracy order (degeneracy_approx_set.h:77) as one launch. */
GMSB_API int gmsb_set_op_count_neighbourhoods(int op, gmsb_set_t a, gmsb_graph_t g, gmsb_set_t members, uint64_t *out);

/* ---- vertex similarity ------------------------------------------------------------------------------------------------ */
/* GMS::VertexSim::Metric                                gms/algorithms/set_based/vertex_similarity/vertex_similarity.h:18 */
typedef enum {
    GMSB_SIM_JACCARD = 0, GMSB_SIM_OVERLAP = 1, GMSB_SIM_ADAMIC_ADAR = 2, GMSB_SIM_RESOURCE = 3,
    GMSB_SIM_COMM_NEIGH = 4, GMSB_SIM_TOTAL_NEIGH = 5, GMSB_SIM_PREF_ATT = 6
} gmsb_sim_metric;
/* vertex_similarity<Metric>(a, b, g) for a batch of pairs   vertex_similarity.h:202-221 */
GMSB_API int gmsb_pair_similarity(gmsb_graph_t g, int metric, int64_t npairs, const int32_t *a, const int32_t *b, double *out);
/* one score per undirected edge u<v in CSR order (BASELINE.json configs[3]); returns the edge count in *m_out */
GMSB_API int gmsb_edge_similarity(gmsb_graph_t g, int metric, double *out, int64_t *m_out);

/* ---- k-cliques ------------------------------------------------------------------------------------------------------------ */
/* KClique::Par::{NP,EP}_kclisting on an oriented DAG      gms/algorithms/non_set_based/k_clique_list/clique_counting.h:14-34
 * g may be a DAG from gmsb_orient, or an undirected graph (then it is degree-oriented internally; the count is
 * orientation-invariant). k==1 -> nodes, k==2 -> edges as parallelize.h:43-44.
 * Kernels for the d+ > 32 sub-problems, chosen from k and the out-degrees: lane-parallel for 5 <= k <= 10,
 * warp-cooperative otherwise. */
GMSB_API int gmsb_kclique_count(gmsb_graph_t g, int k, uint64_t *out);
/* multi-GPU form: this process counts share part_index of part_count of the per-vertex sub-problems (graph
 * replicated, dealt out round-robin in descending size); the shares add up to gmsb_kclique_count's result. */
GMSB_API int gmsb_kclique_count_ex(gmsb_graph_t g, int k, int part_index, int part_count, uint64_t *out);
/* CliqueCount<Set,SGraph,Set2> (returns k!*C_k)           gms/algorithms/set_based/k_clique_count/k_clique_count_set_based.h:20-31 */
GMSB_API int gmsb_kclique_count_ordered(gmsb_graph_t g, int k, uint64_t *out);

#ifdef __cplusplus
}
#endif
#endif /* GMSB_H_ */
