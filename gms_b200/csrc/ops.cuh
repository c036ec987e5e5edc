// ops.cuh — host-callable operators implemented across the .cu files (all take HOST output buffers).
#pragma once
#include "common.cuh"

namespace gmsb {

// generator.cu (host side)
void generate_rmat(int scale, int64_t m, float a, float b, float c, bool permute, vid_t *src, vid_t *dst);
void generate_uniform(int scale, int64_t m, vid_t *src, vid_t *dst);

// setops.cu
void intersect_count_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, uint64_t *out);
void intersect_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, int64_t *out_offsets, vid_t *out_elems,
                     int64_t cap);
void difference_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, int64_t *out_offsets, vid_t *out_elems,
                      int64_t cap);
void union_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, int64_t *out_offsets, vid_t *out_elems,
                 int64_t cap);
void union_count_batch(Graph &g, int64_t np, const vid_t *a, const vid_t *b, uint64_t *out);
void pair_similarity(Graph &g, int metric, int64_t np, const vid_t *a, const vid_t *b, double *out);
void edge_similarity(Graph &g, int metric, double *out, int64_t *m_out);

// tc_support.cu
void tc_vertex2(Graph &g, int64_t *out_n);
void edge_scores_from_support(Graph &g, int metric, const int64_t *base_dev, double *out_dev);
void tc_support(Graph &g, DevBuf<uint32_t> &sup, int part_index = 0, int part_count = 1);
void support_to_vertex2(Graph &g, const uint32_t *sup, unsigned long long *t2_dev);
void vertex2_unrank(Graph &g, const unsigned long long *t2_dev, int64_t *out_dev);
void edge_scores_range(Graph &g, int metric, const int64_t *base_dev, const uint32_t *sup, int64_t a_begin, int64_t a_end,
                       double *out_dev);
void edge_support(Graph &g, const int64_t *base_dev, uint32_t *out_dev);
void upper_edge_base(Graph &g, DevBuf<int64_t> &base, int64_t *m_out);      // setops.cu: scan of per-vertex counts of neighbours > vertex
void emit_upper_pairs(Graph &g, const int64_t *base_dev, vid_t *pa, vid_t *pb);
void pair_similarity_device(Graph &g, int metric, int64_t np, const vid_t *da, const vid_t *db, double *out_host);

// mgpu.cu — several GPUs inside one process
void mg_set_devices(int n, const int *ids);
int mg_device_count();
void mg_tc_total(Graph &g, uint64_t *out);
void mg_kclique_count(Graph &g, int k, uint64_t *out);
void mg_tc_vertex2(Graph &g, int64_t *out_n);
void mg_edge_similarity(Graph &g, int metric, double *out, int64_t *m_out);
void mg_release(Graph &g);

// kcore.cu
void degeneracy_rank(Graph &g, vid_t *out_rank);
void core_numbers(Graph &g, int32_t *out_core);

// truss.cu
void truss_numbers(Graph &g, int32_t *out, int64_t *m_out);
void degeneracy_order_approx(Graph &g, double epsilon, bool rank_format, vid_t *out_host);
void degeneracy_order_approx_ex(Graph &g, double epsilon, bool rank_format, int boundary, bool pull, uint64_t seed,
                                vid_t *out_host);

// kclique.cu
void kclique_count(Graph &g, int k, uint64_t *out, int part_index = 0, int part_count = 1);
void kclique_count_ordered(Graph &g, int k, uint64_t *out);

}  // namespace gmsb
