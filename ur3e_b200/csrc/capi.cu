// C ABI (include/ur3e_b200.h): thin, exception-free wrappers over the model loader and the typed batches.
#include <cstdio>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/ur3e_b200.h"
#include "batch_base.h"
#include "dev_model.h"

using namespace ur3e;

struct ur3e_model { HostModel h; };
struct ur3e_batch { std::unique_ptr<BatchBase> impl; };

extern "C" {

const char* ur3e_last_error(void) { return g_err.c_str(); }

ur3e_model* ur3e_model_load(const char* xml_path) {
  try {
    if (!xml_path) { set_err("null path"); return nullptr; }
    auto m = std::make_unique<ur3e_model>();
    m->h = load_mjcf(xml_path);
    return m.release();
  } catch (const std::exception& e) { set_err(e.what()); return nullptr; }
}
void ur3e_model_destroy(ur3e_model* m) { delete m; }

int ur3e_model_info(const ur3e_model* m, ur3e_model_dims* o) {
  if (!m || !o) return set_err("null argument");
  const HostModel& h = m->h;
  o->nq = h.nq; o->nv = h.nv; o->nu = h.nu; o->nbody = h.nbody; o->njnt = h.njnt; o->ngeom = h.ngeom; o->nsite = h.nsite; o->neq = h.neq;
  o->ntendon = h.ntendon; o->npair = h.npair; o->nkey = h.nkey; o->timestep = h.timestep;
  return 0;
}
int ur3e_model_name2id(const ur3e_model* m, int objtype, const char* name) { return (m && name) ? m->h.name2id(objtype, name) : -1; }
const char* ur3e_model_id2name(const ur3e_model* m, int objtype, int id) {
  if (!m) return nullptr;
  auto it = m->h.names.find(objtype);
  if (it == m->h.names.end() || id < 0 || id >= (int)it->second.size()) return nullptr;
  return it->second[id].c_str();
}
int ur3e_model_array(const ur3e_model* m, const char* field, const void** ptr, int64_t* shape2, int* ndim, int* is_int) {
  if (!m || !field || !ptr) return set_err("null argument");
  auto it = m->h.arr.find(field);
  if (it == m->h.arr.end()) return set_err(std::string("unknown model array '") + field + "'");
  const HostArray& a = it->second;
  *ptr = a.is_int ? (const void*)a.i.data() : (const void*)a.d.data();
  if (ndim) *ndim = (int)a.shape.size();
  if (shape2) { shape2[0] = a.shape.size() > 0 ? a.shape[0] : 0; shape2[1] = a.shape.size() > 1 ? a.shape[1] : 1; }
  if (is_int) *is_int = a.is_int ? 1 : 0;
  return 0;
}
int ur3e_model_num_warnings(const ur3e_model* m) { return m ? (int)m->h.warnings.size() : 0; }
const char* ur3e_model_warning(const ur3e_model* m, int i) { return (m && i >= 0 && i < (int)m->h.warnings.size()) ? m->h.warnings[i].c_str() : nullptr; }

ur3e_batch* ur3e_batch_create(const ur3e_model* m, const ur3e_env_config* cfg, int64_t n_envs, int device, int dtype) {
  try {
    if (!m || !cfg || n_envs <= 0) { set_err("bad argument"); return nullptr; }
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) { set_err("no CUDA device: ur3e_b200 has no CPU path"); return nullptr; }
    if (device < 0 || device >= count) { set_err("device index out of range"); return nullptr; }
    const HostModel& h = m->h;
    auto b = std::make_unique<ur3e_batch>();
    bool f64 = dtype == UR3E_F64;
    if (dtype != UR3E_F32 && dtype != UR3E_F64) { set_err("dtype must be UR3E_F32 or UR3E_F64"); return nullptr; }
    // size classes (engine.cuh Dims*): raw arm 8/6, arm+gripper 23/14, arm+gripper+mug 25/20
    if (h.nbody <= 8 && h.nv <= 6 && h.nu <= 6 && h.npair == 0) b->impl = f64 ? make_batch_f64_raw(h, *cfg, n_envs, device) : make_batch_f32_raw(h, *cfg, n_envs, device);
    else if (h.nbody <= 23 && h.nv <= 14 && h.nq <= 14) b->impl = f64 ? make_batch_f64_grip(h, *cfg, n_envs, device) : make_batch_f32_grip(h, *cfg, n_envs, device);
    else if (h.nbody <= 25 && h.nv <= 20 && h.nq <= 21) b->impl = f64 ? make_batch_f64_main(h, *cfg, n_envs, device) : make_batch_f32_main(h, *cfg, n_envs, device);
    else { set_err("model does not fit any compiled kernel size class"); return nullptr; }
    if (!b->impl) return nullptr;
    return b.release();
  } catch (const std::exception& e) { set_err(e.what()); return nullptr; }
}
void ur3e_batch_destroy(ur3e_batch* b) { delete b; }

#define GUARD(b) if (!(b) || !(b)->impl) return set_err("null batch")
int ur3e_batch_reset(ur3e_batch* b, const uint8_t* mask_dev, uint64_t seed, void* obs_out_dev, void* stream) { GUARD(b); return b->impl->reset(mask_dev, seed, obs_out_dev, (cudaStream_t)stream); }
int ur3e_batch_step(ur3e_batch* b, const void* a, void* o, void* r, uint8_t* te, uint8_t* tr, void* fo, void* stream) { GUARD(b); return b->impl->step(a, o, r, te, tr, fo, (cudaStream_t)stream); }
int ur3e_batch_step_host(ur3e_batch* b, const void* a, void* o, void* r, uint8_t* te, uint8_t* tr) { GUARD(b); return b->impl->step_host(a, o, r, te, tr); }
int ur3e_batch_get_state(ur3e_batch* b, void* qp, void* qv, void* ws, void* stream) { GUARD(b); return b->impl->get_state(qp, qv, ws, (cudaStream_t)stream); }
int ur3e_batch_set_state(ur3e_batch* b, const void* qp, const void* qv, const void* ws, void* stream) { GUARD(b); return b->impl->set_state(qp, qv, ws, (cudaStream_t)stream); }
int ur3e_batch_set_sensor_buffer(ur3e_batch* b, void* buf) { GUARD(b); return b->impl->set_sensor_buffer(buf); }
int ur3e_batch_stats(ur3e_batch* b, double* out, int reset, void* stream) { GUARD(b); if (!out) return set_err("null stats buffer"); return b->impl->stats(out, reset, (cudaStream_t)stream); }
int64_t ur3e_batch_launch_count(const ur3e_batch* b) { return (b && b->impl) ? b->impl->launches : -1; }
int ur3e_batch_kernel_info(const ur3e_batch* b, int32_t* arena_bytes, int32_t* wpb, int32_t* blocks_per_sm, int32_t* regs) {
  GUARD(b);
  if (arena_bytes) *arena_bytes = b->impl->arena_bytes; if (wpb) *wpb = b->impl->wpb; if (blocks_per_sm) *blocks_per_sm = b->impl->blocks_per_sm; if (regs) *regs = b->impl->regs;
  return 0;
}
int ur3e_batch_tier_info(const ur3e_batch* b, int64_t* o) {
  GUARD(b); if (!o) return set_err("null argument");
  int64_t l = 0, f = 0; b->impl->tier_steps(&l, &f);
  o[0] = b->impl->lite_arena_bytes; o[1] = b->impl->lite_wpb; o[2] = b->impl->lite_blocks_per_sm; o[3] = b->impl->lite_regs; o[4] = l; o[5] = f; o[6] = b->impl->last_overflow(); o[7] = 0;
  return 0;
}
int ur3e_batch_mid_tier_info(const ur3e_batch* b, int32_t* arena_bytes, int32_t* wpb, int32_t* regs) {
  GUARD(b);
  if (arena_bytes) *arena_bytes = b->impl->mid_arena_bytes; if (wpb) *wpb = b->impl->mid_wpb; if (regs) *regs = b->impl->mid_regs;
  return 0;
}
int ur3e_batch_kernel_timing(ur3e_batch* b, int enable) { GUARD(b); return b->impl->kernel_timing(enable); }
int ur3e_batch_kernel_times(ur3e_batch* b, double* out6) { GUARD(b); if (!out6) return set_err("null argument"); return b->impl->kernel_times(out6); }
int ur3e_batch_state_bytes(const ur3e_batch* b) { return (b && b->impl) ? b->impl->state_bytes : -1; }
int ur3e_batch_query_create(ur3e_batch* b, const int32_t* objtype, const int32_t* objid, int32_t k) {
  GUARD(b);
  try { return b->impl->query_create(objtype, objid, k); } catch (const std::exception& e) { return set_err(e.what()); }
}
int ur3e_batch_query(ur3e_batch* b, int query_id, void* pos, void* mat, void* vel, int flg_local, void* stream) {
  GUARD(b); return b->impl->query(query_id, pos, mat, vel, flg_local, (cudaStream_t)stream);
}
int ur3e_batch_query_jac(ur3e_batch* b, int query_id, void* jacp, void* jacr, void* M, void* qfrc_bias, void* stream) {
  GUARD(b); return b->impl->query_jac(query_id, jacp, jacr, M, qfrc_bias, (cudaStream_t)stream);
}
int ur3e_batch_max_contacts(const ur3e_batch* b) { GUARD(b); return b->impl->max_contacts(); }
int ur3e_batch_forward(ur3e_batch* b, const void* ctrl, const ur3e_forward_out* out, void* stream) {
  GUARD(b); return b->impl->forward(ctrl, out, (cudaStream_t)stream);
}

}  // extern "C"
