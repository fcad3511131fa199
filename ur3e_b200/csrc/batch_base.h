// Type-erased batch interface + per-(dtype, size class) factories (each factory lives in its own
// translation unit so the six kernel instantiations compile in parallel).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <memory>
#include <string>

#include "../../include/ur3e_b200.h"
#include "host_model.h"

namespace ur3e {

inline thread_local std::string g_err;
inline int set_err(const std::string& e, int code = -1) { g_err = e; return code; }
#define CUDA_OK(expr)                                                                                       \
  do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return ::ur3e::set_err(std::string(#expr) + ": " + cudaGetErrorString(e_), -2); } while (0)


struct BatchBase {
  virtual ~BatchBase() {}
  virtual int reset(const uint8_t* mask, uint64_t seed, void* obs, cudaStream_t s) = 0;
  virtual int step(const void* act, void* obs, void* rew, uint8_t* term, uint8_t* trunc, void* fobs, cudaStream_t s) = 0;
  virtual int step_host(const void* act, void* obs, void* rew, uint8_t* term, uint8_t* trunc) = 0;
  virtual int get_state(void* qpos, void* qvel, void* ws, cudaStream_t s) = 0;
  virtual int set_state(const void* qpos, const void* qvel, const void* ws, cudaStream_t s) = 0;
  virtual int stats(double* out, int reset, cudaStream_t s) = 0;
  virtual int set_sensor_buffer(void* buf) = 0;
  // optional CUDA-event timing of every step-kernel launch (bench.py's roofline: the duration of the dominant kernel alone)
  virtual int kernel_timing(int enable) = 0;
  virtual int kernel_times(double* out6) = 0;   // {ms, launches} x {lite tier, grasp / generic tier on the caller's stream, generic tier on the side stream}; synchronises
  // kinematics queries (query.cuh): the batch owns the compiled object tables; query_create returns the query's id
  virtual int query_create(const int32_t* objtype, const int32_t* objid, int k) = 0;
  virtual int query(int id, void* pos, void* mat, void* vel, int local, cudaStream_t s) = 0;
  // Jacobians of a query's objects, mass matrix and bias forces (query.cuh query_jac_env); id = -1: no objects
  virtual int query_jac(int id, void* jacp, void* jacr, void* M, void* bias, cudaStream_t s) = 0;
  // one mj_forward per environment at the stored state: contacts, contact forces, qacc, sensordata (query_fwd.cuh forward_query_env)
  virtual int max_contacts() const = 0;
  virtual int forward(const void* ctrl, const ur3e_forward_out* out, cudaStream_t s) = 0;
  // offscreen rendering (render.cuh): the batch owns its renderers and their pose scratch; render_create returns the renderer's id
  virtual int render_create(const ur3e_camera* cam, const int32_t* geom_ids, int k, const float* rgba, int width, int height) = 0;
  virtual int render(int id, const int32_t* env_ids, long long m, uint8_t* rgb, void* depth, int32_t* seg, cudaStream_t s) = 0;
  // T tiered steps of m scratch copies of records (src ids) or of fresh records (qpos0 / qvel0 / ws0); the batch is not modified
  virtual int rollout(const int32_t* src, const void* qpos0, const void* qvel0, const void* ws0, long long m, int T, const void* act,
                      const ur3e_rollout_out* out, cudaStream_t s) = 0;
  int64_t launches = 0;
  virtual void tier_steps(int64_t* lite, int64_t* full) const { *lite = 0; *full = 0; }
  virtual int64_t last_overflow() const { return 0; }
  int arena_bytes = 0, blocks_per_sm = 0, regs = 0, device = 0, state_bytes = 0, wpb = 0;
  int lite_arena_bytes = 0, lite_blocks_per_sm = 0, lite_regs = 0, lite_wpb = 0;   // zero when the model has no lite size class
  int mid_arena_bytes = 0, mid_regs = 0, mid_wpb = 0;                              // zero when the model has no grasp-tier size class
  long long n = 0;
};


// returns nullptr (and sets the error) on failure
std::unique_ptr<BatchBase> make_batch_f32_raw(const HostModel&, const ur3e_env_config&, long long n, int device);
std::unique_ptr<BatchBase> make_batch_f64_raw(const HostModel&, const ur3e_env_config&, long long n, int device);
std::unique_ptr<BatchBase> make_batch_f32_grip(const HostModel&, const ur3e_env_config&, long long n, int device);
std::unique_ptr<BatchBase> make_batch_f64_grip(const HostModel&, const ur3e_env_config&, long long n, int device);
std::unique_ptr<BatchBase> make_batch_f32_main(const HostModel&, const ur3e_env_config&, long long n, int device);
std::unique_ptr<BatchBase> make_batch_f64_main(const HostModel&, const ur3e_env_config&, long long n, int device);

}  // namespace ur3e
