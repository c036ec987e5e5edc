// sets.cuh — device-resident sorted set (sets.cu) behind the gmsb_set_* entry points; its binary operations are in
// setops.cu.
#pragma once
#include "common.cuh"

namespace gmsb {

struct DevSet {
    DevBuf<vid_t> own;          // storage of an owning set; empty for a view borrowed from a graph's CSR
    const vid_t *p = nullptr;   // ascending, duplicate-free
    int64_t n = 0;
};

// an ascending list in device memory: a set's elements or a neighbourhood
struct Span {
    const vid_t *p;
    int64_t n;
};

DevSet *set_from_host(const vid_t *elems, int64_t count);
DevSet *set_from_device(const vid_t *src, int64_t count, bool sorted);
DevSet *set_range(int64_t bound);
DevSet *set_neighbourhood(Graph &g, vid_t v);
DevSet *set_clone(const DevSet &a);
void set_to_host(const DevSet &a, vid_t *out);
bool set_contains(const DevSet &a, vid_t x);
bool set_equal(const DevSet &a, const DevSet &b);
void set_add(DevSet &a, vid_t x);
void set_remove(DevSet &a, vid_t x);
// setops.cu; difference is left minus right
void set_op_count_many(gmsb_set_op_kind op, const DevSet &a, int64_t np, DevSet *const *bs, uint64_t *out);
void set_op_count_members(gmsb_set_op_kind op, const DevSet &a, Graph &g, const DevSet &members, uint64_t *out);
void set_op_many(gmsb_set_op_kind op, const DevSet &a, int64_t np, DevSet *const *bs, DevSet **outs);

}  // namespace gmsb
