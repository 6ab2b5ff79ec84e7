// rrt_best_oracle.cpp -- RRT::plan's second half, get_best_solution (rrt.rs:183-193) + RRTTree::get_path_to (:48-60), restated over a
// grown tree's arrays (states, parents, finals as tests/rrt_oracle.cpp exports them) with the oracle's norm2 -- TEST INFRASTRUCTURE,
// the CPU baseline of scripts/rrt_query_batch_bench.py.  tests/rrt_best_oracle.py compiles it together with oracle/porrt_oracle.cpp.
#include <cstdint>
#include <vector>

#include "../oracle/porrt_oracle.hpp"

#define API extern "C" __attribute__((visibility("default")))

using namespace orc;

// The final with the smallest (cost, path length), the first of equal pairs; a path is the chain of parents, root first, and its cost
// is summed root first from 0.0.  xy[2 V], parent[V] (-1 at the root), finals[F].  out = (final id or -1, path length); path_xy[2 V]
// receives the path.  Returns the cost (0.0 without a final).
API double orc_rrt_best_path(const double* xy, const int64_t* parent, int64_t V, const int64_t* finals, int64_t F, double* path_xy,
                             int64_t* out) {
  int64_t best = -1;
  double best_c = 0.0;
  std::vector<int64_t> chain, best_chain;
  for (int64_t k = 0; k < F; ++k) {
    chain.clear();
    for (int64_t v = finals[k]; v >= 0 && (int64_t)chain.size() <= V; v = parent[v]) chain.push_back(v);
    double c = 0.0;
    for (size_t j = chain.size() - 1; j > 0; --j)
      c += norm2(State{xy[2 * chain[j]], xy[2 * chain[j] + 1]}, State{xy[2 * chain[j - 1]], xy[2 * chain[j - 1] + 1]});
    if (best < 0 || c < best_c || (c == best_c && chain.size() < best_chain.size())) {
      best = finals[k]; best_c = c; best_chain = chain;
    }
  }
  out[0] = best;
  out[1] = (int64_t)best_chain.size();
  for (size_t i = 0; i < best_chain.size(); ++i) {
    const int64_t v = best_chain[best_chain.size() - 1 - i];
    path_xy[2 * i] = xy[2 * v]; path_xy[2 * i + 1] = xy[2 * v + 1];
  }
  return best_c;
}
