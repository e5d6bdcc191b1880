// Host-only table of what one evaluation of the logistic GLMM runs for every K = 1 .. kMaxK, taken from the
// planner's own functions (fused_eval_kernel, gram_mid_kernel, gram_big_plan, obs_tile_buffers, ...); launches
// nothing.  tests/test_host_api.py maps the parity cases through it to check that they reach every class.
//   nvcc -std=c++17 -gencode arch=compute_100a,code=sm_100a -o tools/build/dispatch tools/dispatch_table.cu
//
// One line per K, key=value fields ("-" where the field does not apply):
//   gram    order-2 Gram path: fused (k_fused_eval), mid (k_gram_mid), wide (k_gram_wide), big (k_gram_big)
//   id      instantiation of k_fused_eval / k_gram_mid, numbered by first K in each family: two K share an id
//           exactly when the planner returns the same kernel
//   plan    k_gram_big plan key n_groups/TN/straddle (straddle 1 when the plan has the straddle-tile job)
//   chunks  32-column chunks of k_obs_fused (K <= kOfMaxK; it runs the order-0 and order-1 evaluations also
//           where k_fused_eval runs order 2)
//   nbuf    k_obs tile buffers at Q = 1, 8, kMaxQ (K > kOfMaxK)
#include <cstdio>
#include <map>
#include "../linearresponsevariationalbayes.py_b200/csrc/fused.cuh"
#include "../linearresponsevariationalbayes.py_b200/csrc/gram_wide.cuh"
#include "../linearresponsevariationalbayes.py_b200/csrc/gram_big.cuh"
namespace lrvb { void set_error(const char*, ...) {} long long g_launches = 0; }
using namespace lrvb;

int main() {
  std::map<const void*, int> fu_ids, gm_ids;
  auto id_of = [](std::map<const void*, int>& ids, const void* fn) {
    auto it = ids.find(fn);
    if (it != ids.end()) return it->second;
    const int id = (int)ids.size();
    ids[fn] = id;
    return id;
  };
  int bad = 0;
  for (int K = 1; K <= kMaxK; ++K) {
    char gram[8] = "-", id[8] = "-", plan[24] = "-", chunks[8] = "-", nbuf[16] = "-";
    if (K <= kFuMaxK) {
      const void* fn = (const void*)fused_eval_kernel(K);
      if (!fn) { printf("K=%d: no k_fused_eval instantiation\n", K); ++bad; }
      snprintf(gram, sizeof gram, "fused");
      snprintf(id, sizeof id, "%d", id_of(fu_ids, fn));
    } else if (K <= kGmMaxK) {
      const void* fn = (const void*)gram_mid_kernel(K).fn;
      if (!fn) { printf("K=%d: no k_gram_mid instantiation\n", K); ++bad; }
      snprintf(gram, sizeof gram, "mid");
      snprintf(id, sizeof id, "%d", id_of(gm_ids, fn));
    } else if (gram_wide_eligible(K)) {
      snprintf(gram, sizeof gram, "wide");
    } else {
      const GbPlan pl = gram_big_plan(K);
      int straddle = 0;
      for (const GbJob& j : pl.jobs) straddle |= j.kind == 1;
      snprintf(gram, sizeof gram, "big");
      snprintf(plan, sizeof plan, "%d/%d/%d", pl.n_groups, pl.TN, straddle);
    }
    if (K <= kOfMaxK)
      snprintf(chunks, sizeof chunks, "%d", obs_fused_chunks(K));
    else
      snprintf(nbuf, sizeof nbuf, "%d,%d,%d", obs_tile_buffers(K, 1), obs_tile_buffers(K, 8), obs_tile_buffers(K, kMaxQ));
    printf("K=%d gram=%s id=%s plan=%s chunks=%s nbuf=%s\n", K, gram, id, plan, chunks, nbuf);
  }
  printf("kMaxK=%d kMaxQ=%d kFuUnroll=%d kOfUnroll=%d fused_ids=%zu mid_ids=%zu\n", kMaxK, kMaxQ, kFuUnroll,
         kOfUnroll, fu_ids.size(), gm_ids.size());
  return bad != 0;
}
