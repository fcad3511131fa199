// TEST-ONLY: compiles the rollout's argument check (ur3e_b200/csrc/rollout.h) as plain C++ so that it can be checked without a GPU.
// Not part of the package, never loaded by ur3e_b200.  Bound by tests/hostcheck/rollout.py.
#include <string>

#include "../../ur3e_b200/csrc/rollout.h"

using namespace ur3e;

static std::string g_err;   // the reason the latest call was rejected

extern "C" const char* hro_error() { return g_err.c_str(); }

// rollout_check itself: 0 when the call is accepted, -1 when rejected (hro_error gives the reason)
extern "C" int hro_rollout_check(long long m, long long T, int actions, int src_ids, int qpos0, int qvel0, int ws0, int out, int any) {
  g_err = rollout_check(m, T, actions != 0, src_ids != 0, qpos0 != 0, qvel0 != 0, ws0 != 0, out != 0, any != 0);
  return g_err.empty() ? 0 : -1;
}
