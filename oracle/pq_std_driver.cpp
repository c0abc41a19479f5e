// The reference's priority queue as its MEX source describes it (priority_queue_interface_mex.cpp:19-31): a
// std::priority_queue of (id, value) entries ordered by value only, the smallest on top, ties left to libstdc++'s
// push_heap / pop_heap.  Output: oracle/libpq_std.so (git-ignored).
// TEST INFRASTRUCTURE: an implementation of the queue that shares no code with the oracle's heap restatement
// (pdmpc_oracle.c).  It stands in for the reference's own source (oracle/_ref/libpq_ref.so) where that is not built.
#include <cstdint>
#include <queue>
#include <utility>
#include <vector>

namespace {
using Entry = std::pair<int64_t, double>;  // (id, value)
struct Greater {
    bool operator()(const Entry &a, const Entry &b) const { return a.second > b.second; }
};
using Queue = std::priority_queue<Entry, std::vector<Entry>, Greater>;
}  // namespace

extern "C" {

void *pq_std_new(void) { return new Queue(); }

void pq_std_free(void *q) { delete static_cast<Queue *>(q); }

void pq_std_push(void *q, const double *ids, const double *vals, int64_t n) {
    for (int64_t i = 0; i < n; ++i) static_cast<Queue *>(q)->push(Entry(static_cast<int64_t>(ids[i]), vals[i]));
}

// -1 when empty (mex.cpp:87-94)
int64_t pq_std_pop(void *q, double *val) {
    Queue &pq = *static_cast<Queue *>(q);
    if (pq.empty()) {
        if (val) *val = -1.0;
        return -1;
    }
    const Entry top = pq.top();
    pq.pop();
    if (val) *val = top.second;
    return top.first;
}

int64_t pq_std_size(void *q) { return static_cast<int64_t>(static_cast<Queue *>(q)->size()); }
}
