// Argument check of ur3e_batch_rollout (include/ur3e_b200.h); plain C++ so that tests/hostcheck can compile it without a GPU.
#pragma once
#include <string>

namespace ur3e {

// m rollouts of T env-steps; which inputs are given (actions, source ids, qpos0, qvel0, the warm start); `out` given and `any` of its
// outputs given.  Returns "" when valid, else the reason the call is rejected.
inline std::string rollout_check(long long m, long long T, bool actions, bool src_ids, bool qpos0, bool qvel0, bool ws0, bool out, bool any) {
  if (m < 1 || m > 2147483647LL) return "m=" + std::to_string(m) + " rollouts (1 .. 2^31 - 1: the tier lists hold int32 indices)";
  if (T < 1) return "T=" + std::to_string(T) + " env-steps (at least 1)";
  if (!actions) return "actions is null";
  if (qpos0 != qvel0) return qpos0 ? "qpos0 is given without qvel0" : "qvel0 is given without qpos0";
  if (ws0 && !qpos0) return "qacc_warmstart0 is given without qpos0 and qvel0";
  if (src_ids && qpos0) return "both sources are given (src_env_ids and qpos0 / qvel0)";
  if (!src_ids && !qpos0) return "no source is given (src_env_ids or qpos0 / qvel0)";
  if (!out) return "out is null";
  if (!any) return "all outputs are null";
  return "";
}

}  // namespace ur3e
