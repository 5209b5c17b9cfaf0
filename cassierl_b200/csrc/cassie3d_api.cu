// C-ABI of the batched 3-D step path (include/cassie3d.h).  Host glue only: the arithmetic is tree_engine.cuh.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <dlfcn.h>

#include "../../include/cassie3d.h"
#include "mjcf_flatten.h"
#include "rollout_args.h"
#include "tree_kernels.cuh"

using namespace cassie;
using namespace cassie::tree;

static thread_local std::string g3_last_error;
static int fail3(const std::string& msg) {
  g3_last_error = msg;
  return -1;
}
#define CU3_OK(expr)                                                                             \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) return fail3(std::string(#expr) + ": " + cudaGetErrorString(_e));     \
  } while (0)

static std::string default_xml3() {
  if (const char* e = getenv("CASSIE3D_XML")) return e;
  Dl_info info;
  if (dladdr((void*)&default_xml3, &info) && info.dli_fname) {
    std::string p = info.dli_fname;  // <pkg>/lib/libcassie2d.so -> <pkg>/model/cassie3d_stiff.xml
    size_t s = p.rfind('/');
    if (s != std::string::npos) {
      p = p.substr(0, s);
      size_t s2 = p.rfind('/');
      if (s2 != std::string::npos) return p.substr(0, s2) + "/model/cassie3d_stiff.xml";
    }
  }
  return "cassie3d_stiff.xml";
}

struct Cassie3dBatch {
  int n = 0, device = 0, precision = 32, lanes = 32;
  TreeModel<double> model;
  TreeModel<float> m32;
  TreeModel<double> m64;
  TreeBatchView<float> v32;
  TreeBatchView<double> v64;
  std::vector<void*> allocs;
  std::vector<double> reset_q, reset_qd;
  void* d_reset_q = nullptr;
  void* d_reset_qd = nullptr;
  void* d_action = nullptr;   // host-variant staging
  uint8_t* d_done = nullptr;
  void* d_obs = nullptr;      // host-variant staging of EnvStepHost
  void* d_reward = nullptr;
  int32_t* ep_len = nullptr;  // [n] policy steps since the env's last reset (EnvStep)
  int32_t* policy_step = nullptr;   // [n] Philox step counter of Rollout: zero at Create, advanced by Rollout only
  void* d_act_env = nullptr;  // [n][nu] the mapped, clipped action of Rollout's current policy step
  std::vector<double> kp, kd; // PD gains of the env's kActPd action space, per motor
  cudaStream_t own_stream = nullptr;
  size_t rs() const { return precision == 64 ? 8 : 4; }
};

namespace {
struct DeviceGuard {
  int prev = 0;
  explicit DeviceGuard(int dev) { cudaGetDevice(&prev); cudaSetDevice(dev); }
  ~DeviceGuard() { cudaSetDevice(prev); }
};

int dmalloc(Cassie3dBatch* h, void** p, size_t bytes) {
  CU3_OK(cudaMalloc(p, bytes));
  h->allocs.push_back(*p);
  CU3_OK(cudaMemset(*p, 0, bytes));
  return 0;
}

template <typename T>
int setup(Cassie3dBatch* h, TreeBatchView<T>& v) {
  const size_t n = (size_t)h->n;
  const TreeModel<double>& m = h->model;
  cast_tree_model(&h->m32, h->model);
  cast_tree_model(&h->m64, h->model);
  v.n = h->n;
  if (dmalloc(h, (void**)&v.qpos, sizeof(T) * n * m.nq) || dmalloc(h, (void**)&v.qvel, sizeof(T) * n * m.nv) ||
      dmalloc(h, (void**)&v.warm, sizeof(T) * n * m.nv) || dmalloc(h, (void**)&v.stats, sizeof(int32_t) * 4 * n) ||
      dmalloc(h, (void**)&v.resets, sizeof(int32_t) * n) ||
      dmalloc(h, (void**)&v.order, sizeof(int32_t) * n) || dmalloc(h, (void**)&v.bins, sizeof(int32_t) * 2 * kTreeBins) ||
      dmalloc(h, (void**)&v.resume, sizeof(int32_t) * n) || dmalloc(h, &h->d_reset_q, sizeof(T) * m.nq) ||
      dmalloc(h, &h->d_reset_qd, sizeof(T) * m.nv) || dmalloc(h, &h->d_action, sizeof(T) * n * m.nu) ||
      dmalloc(h, (void**)&h->d_done, n) || dmalloc(h, &h->d_obs, sizeof(T) * n * kObsDim3d) ||
      dmalloc(h, &h->d_reward, sizeof(T) * n) || dmalloc(h, (void**)&h->ep_len, sizeof(int32_t) * n) ||
      dmalloc(h, (void**)&h->policy_step, sizeof(int32_t) * n) || dmalloc(h, &h->d_act_env, sizeof(T) * n * m.nu))
    return -1;
  return 0;
}

template <typename T>
int upload_reset(Cassie3dBatch* h) {
  std::vector<T> q(h->reset_q.begin(), h->reset_q.end()), v(h->reset_qd.begin(), h->reset_qd.end());
  CU3_OK(cudaMemcpy(h->d_reset_q, q.data(), sizeof(T) * q.size(), cudaMemcpyHostToDevice));
  CU3_OK(cudaMemcpy(h->d_reset_qd, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
  return 0;
}

template <typename T> const TreeModel<T>& model_of(Cassie3dBatch* h);
template <> const TreeModel<float>& model_of<float>(Cassie3dBatch* h) { return h->m32; }
template <> const TreeModel<double>& model_of<double>(Cassie3dBatch* h) { return h->m64; }
template <typename T> TreeBatchView<T>& view(Cassie3dBatch* h);
template <> TreeBatchView<float>& view<float>(Cassie3dBatch* h) { return h->v32; }
template <> TreeBatchView<double>& view<double>(Cassie3dBatch* h) { return h->v64; }

template <typename T>
int step(Cassie3dBatch* h, const void* action, int n_sub, double z_done, int auto_reset, uint8_t* done, cudaStream_t s) {
  TreeStepArgs a;
  a.action = action; a.n_sub = n_sub; a.z_done = z_done; a.auto_reset = auto_reset; a.done = done;
  a.reset_q = h->d_reset_q; a.reset_qd = h->d_reset_qd;
  CU3_OK(TreeLaunch<T>::step(model_of<T>(h), view<T>(h), a, h->lanes, s));
  return 0;
}

template <typename T>
int env_step(Cassie3dBatch* h, int mode, const void* action, int n_sub, int max_path_length, int flags, void* obs, void* reward,
             uint8_t* done, cudaStream_t s) {
  TreeStepArgs a;
  a.action = action; a.n_sub = n_sub; a.z_done = 0; a.auto_reset = 0; a.done = done;
  a.reset_q = h->d_reset_q; a.reset_qd = h->d_reset_qd;
  TreeEnvParams<T> ep;
  for (int i = 0; i < kMaxAct; i++) {
    ep.kp[i] = i < h->model.nu ? (T)h->kp[i] : (T)0;
    ep.kd[i] = i < h->model.nu ? (T)h->kd[i] : (T)0;
  }
  ep.mode = mode; ep.flags = flags; ep.max_path_length = max_path_length;
  ep.obs = (T*)obs; ep.reward = (T*)reward; ep.ep_len = h->ep_len;
  CU3_OK(TreeLaunch<T>::env_step(model_of<T>(h), view<T>(h), a, ep, h->lanes, s));
  return 0;
}

template <typename T>
int rollout(Cassie3dBatch* h, int mode, const PolicyShape3d& shape, const void* params, int T_steps, int n_sub,
            int max_path_length, int normalize, unsigned long long seed, unsigned int env0, void* obs, void* act, void* mean,
            void* reward, uint8_t* done, cudaStream_t s) {
  const size_t n = (size_t)h->n, nu = (size_t)h->model.nu;
  TreeStepArgs a;
  a.action = nullptr; a.n_sub = n_sub; a.z_done = 0; a.auto_reset = 1; a.done = nullptr;
  a.reset_q = h->d_reset_q; a.reset_qd = h->d_reset_qd;
  TreeEnvParams<T> ep;
  for (int i = 0; i < kMaxAct; i++) {
    ep.kp[i] = i < h->model.nu ? (T)h->kp[i] : (T)0;
    ep.kd[i] = i < h->model.nu ? (T)h->kd[i] : (T)0;
  }
  ep.mode = mode; ep.flags = kEnvAutoReset; ep.max_path_length = max_path_length;
  ep.obs = nullptr; ep.reward = nullptr; ep.ep_len = h->ep_len;
  TreeRolloutParams<T> ro;
  double lo[kMaxAct] = {0}, hi[kMaxAct] = {0};
  action_box(h->model, mode, lo, hi);
  for (int i = 0; i < kMaxAct; i++) { ro.lo[i] = (T)lo[i]; ro.hi[i] = (T)hi[i]; }
  ro.params = (const T*)params; ro.shape = shape; ro.normalize = normalize; ro.seed = seed; ro.env0 = env0;
  ro.policy_step = h->policy_step; ro.act_env = (T*)h->d_act_env;
  for (int k = 0; k < T_steps; k++) {   // one launch pass per policy step, no host synchronisation in between
    ro.obs = (T*)obs + (size_t)k * n * kObsDim3d;
    ro.act = (T*)act + (size_t)k * n * nu;
    ro.mean = (T*)mean + (size_t)k * n * nu;
    ro.rew = (T*)reward + (size_t)k * n;
    ro.done = done + (size_t)k * n;
    CU3_OK(TreeLaunch<T>::rollout_step(model_of<T>(h), view<T>(h), a, ep, ro, h->lanes, s));
  }
  return 0;
}

template <typename T>
int observe(Cassie3dBatch* h, void* obs, cudaStream_t s) {
  CU3_OK(TreeLaunch<T>::observe(model_of<T>(h), view<T>(h), (T*)obs, s));
  return 0;
}

int check_env_step(Cassie3dBatch* h, int mode, const void* action, int n_substeps, int flags) {
  if (!h) return fail3("null handle");
  if (mode != CASSIE3D_MODE_TORQUE && mode != CASSIE3D_MODE_PD) return fail3("mode must be CASSIE3D_MODE_TORQUE or CASSIE3D_MODE_PD");
  if (!action) return fail3("EnvStep needs an action");
  if (n_substeps < 1) return fail3("n_substeps must be at least 1");
  if (flags & ~(CASSIE3D_AUTO_RESET | CASSIE3D_TERMINAL_OBS)) return fail3("unknown flag bits");
  return 0;
}
}  // namespace

static_assert((int)CASSIE3D_MODE_TORQUE == (int)kActTorque && (int)CASSIE3D_MODE_PD == (int)kActPd, "action modes");
static_assert((int)CASSIE3D_AUTO_RESET == (int)kEnvAutoReset && (int)CASSIE3D_TERMINAL_OBS == (int)kEnvTerminalObs, "env flags");
static_assert((int)CASSIE3D_OBS_DIM == kObsDim3d, "observation size");
static_assert((int)CASSIE3D_POLICY_PARAMS == kPolicyParams3d, "policy parameter count");
static_assert((int)CASSIE3D_POLICY_MAX_LAYERS == kPolicyMaxLayers3d && (int)CASSIE3D_POLICY_MAX_WIDTH == kPolicyMaxWidth3d,
              "policy shape limits");
static_assert(kMaxFeat3d == 2 * kObsDim3d + 4, "baseline features of the 3-D observation");

#define DISPATCH3(h, expr32, expr64) ((h)->precision == 64 ? (expr64) : (expr32))

extern "C" {

const char* Cassie3dGetLastError(void) { return g3_last_error.c_str(); }

Cassie3dBatch* Cassie3dBatchCreate(const char* xml_path, int n_envs, int device, int precision) {
  g3_last_error.clear();
  if (n_envs <= 0) { fail3("n_envs must be positive"); return nullptr; }
  if (precision != 32 && precision != 64) { fail3("precision must be 32 or 64"); return nullptr; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { fail3("no CUDA device: libcassie2d has no CPU fallback"); return nullptr; }
  if (device < 0 || device >= ndev) { fail3("bad device index"); return nullptr; }
  Cassie3dBatch* h = new Cassie3dBatch();
  h->n = n_envs; h->device = device; h->precision = precision;
  if (const char* e = getenv("CASSIE3D_LANES")) {
    const int l = atoi(e);
    if (l == 8 || l == 16 || l == 32) h->lanes = l;
  }
  std::string err;
  if (!flatten_tree_file(xml_path ? xml_path : default_xml3(), &h->model, &err)) { fail3("model: " + err); delete h; return nullptr; }
  DeviceGuard g(device);
  const int rc = precision == 64 ? setup<double>(h, h->v64) : setup<float>(h, h->v32);
  if (rc) { Cassie3dBatchDestroy(h); return nullptr; }
  // default reset state: the planar constructor pose (Cassie2d.cpp:56-58) on the 3-D joints, abduction = yaw = 0;
  // joints are matched by their MuJoCo order per leg: abduction, yaw, hip, knee, ankle, toe, achilles rod
  const TreeModel<double>& m = h->model;
  h->reset_q.assign(m.nq, 0.0);
  h->reset_qd.assign(m.nv, 0.0);
  for (int i = 0; i < 7; i++) h->reset_q[i] = m.qpos0[i];
  for (int d = 6; d < m.nv; d++) h->reset_q[m.user_dof[d] + 1] = m.qpos0[d + 1];
  if (m.nq == 21) {
    const double leg[7] = {0.0, 0.0, 0.68111815, -1.40730357, 1.62972042, -1.77611107, -0.61968407};
    h->reset_q[2] = 0.939;
    for (int i = 0; i < 7; i++) { h->reset_q[7 + i] = leg[i]; h->reset_q[14 + i] = leg[i]; }
  }
  if (DISPATCH3(h, upload_reset<float>(h), upload_reset<double>(h))) { Cassie3dBatchDestroy(h); return nullptr; }
  h->kp.assign(m.nu, kDefaultKp);
  h->kd.assign(m.nu, kDefaultKd);
  if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) { fail3("cudaStreamCreate"); Cassie3dBatchDestroy(h); return nullptr; }
  if (Cassie3dBatchResetAll(h, nullptr, nullptr)) { Cassie3dBatchDestroy(h); return nullptr; }
  cudaDeviceSynchronize();
  return h;
}

void Cassie3dBatchDestroy(Cassie3dBatch* h) {
  if (!h) return;
  DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  for (void* p : h->allocs) cudaFree(p);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

int Cassie3dBatchSizes(Cassie3dBatch* h, int32_t* out) {
  if (!h || !out) return fail3("null argument");
  out[0] = h->model.nq; out[1] = h->model.nv; out[2] = h->model.nu; out[3] = tree::kMaxRows; out[4] = tree::kMaxCon;
  out[5] = (int32_t)(h->precision == 64 ? sizeof(Scratch<double, tree::kFastRows, tree::kFastCon>) : sizeof(Scratch<float, tree::kFastRows, tree::kFastCon>));
  return 0;
}

int Cassie3dBatchSetLanes(Cassie3dBatch* h, int lanes) {
  if (!h) return fail3("null handle");
  if (lanes != 8 && lanes != 16 && lanes != 32) return fail3("lanes must be 8, 16 or 32");
  h->lanes = lanes;
  return 0;
}

int Cassie3dBatchSetResetState(Cassie3dBatch* h, const double* qpos, const double* qvel) {
  if (!h || !qpos || !qvel) return fail3("null argument");
  DeviceGuard g(h->device);
  h->reset_q.assign(qpos, qpos + h->model.nq);
  h->reset_qd.assign(qvel, qvel + h->model.nv);
  cudaDeviceSynchronize();
  return DISPATCH3(h, upload_reset<float>(h), upload_reset<double>(h));
}

int Cassie3dBatchGetResetState(Cassie3dBatch* h, double* qpos, double* qvel) {
  if (!h || !qpos || !qvel) return fail3("null argument");
  memcpy(qpos, h->reset_q.data(), sizeof(double) * h->reset_q.size());
  memcpy(qvel, h->reset_qd.data(), sizeof(double) * h->reset_qd.size());
  return 0;
}

int Cassie3dBatchResetAll(Cassie3dBatch* h, const uint8_t* mask, void* stream) {
  if (!h) return fail3("null handle");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (h->precision == 64)
    CU3_OK(TreeLaunch<double>::set_all(h->v64, h->model.nq, h->model.nv, (const double*)h->d_reset_q, (const double*)h->d_reset_qd, mask, s));
  else
    CU3_OK(TreeLaunch<float>::set_all(h->v32, h->model.nq, h->model.nv, (const float*)h->d_reset_q, (const float*)h->d_reset_qd, mask, s));
  if (mask) {
    k_tree_zero_len<<<(h->n + 127) / 128, 128, 0, s>>>(h->n, mask, h->ep_len);
    count_launch();
    CU3_OK(cudaGetLastError());
  } else
    CU3_OK(cudaMemsetAsync(h->ep_len, 0, sizeof(int32_t) * (size_t)h->n, s));
  return 0;
}

static void* qpos_of(Cassie3dBatch* h) { return h->precision == 64 ? (void*)h->v64.qpos : (void*)h->v32.qpos; }
static void* qvel_of(Cassie3dBatch* h) { return h->precision == 64 ? (void*)h->v64.qvel : (void*)h->v32.qvel; }
static void* warm_of(Cassie3dBatch* h) { return h->precision == 64 ? (void*)h->v64.warm : (void*)h->v32.warm; }
static int32_t* stats_of(Cassie3dBatch* h) { return h->precision == 64 ? h->v64.stats : h->v32.stats; }
static int32_t* resets_of(Cassie3dBatch* h) { return h->precision == 64 ? h->v64.resets : h->v32.resets; }

int Cassie3dBatchSetState(Cassie3dBatch* h, const void* qpos, const void* qvel, void* stream) {
  if (!h || !qpos || !qvel) return fail3("null argument");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)h->n;
  CU3_OK(cudaMemcpyAsync(qpos_of(h), qpos, h->rs() * n * h->model.nq, cudaMemcpyDeviceToDevice, s));
  CU3_OK(cudaMemcpyAsync(qvel_of(h), qvel, h->rs() * n * h->model.nv, cudaMemcpyDeviceToDevice, s));
  CU3_OK(cudaMemsetAsync(warm_of(h), 0, h->rs() * n * h->model.nv, s));
  CU3_OK(cudaMemsetAsync(h->ep_len, 0, sizeof(int32_t) * n, s));
  return 0;
}

int Cassie3dBatchGetState(Cassie3dBatch* h, void* qpos, void* qvel, void* stream) {
  if (!h || !qpos || !qvel) return fail3("null argument");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = (size_t)h->n;
  CU3_OK(cudaMemcpyAsync(qpos, qpos_of(h), h->rs() * n * h->model.nq, cudaMemcpyDeviceToDevice, s));
  CU3_OK(cudaMemcpyAsync(qvel, qvel_of(h), h->rs() * n * h->model.nv, cudaMemcpyDeviceToDevice, s));
  return 0;
}

int Cassie3dBatchGetWarmStart(Cassie3dBatch* h, void* w, void* stream) {
  if (!h || !w) return fail3("null argument");
  DeviceGuard g(h->device);
  CU3_OK(cudaMemcpyAsync(w, warm_of(h), h->rs() * (size_t)h->n * h->model.nv, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int Cassie3dBatchSetWarmStart(Cassie3dBatch* h, const void* w, void* stream) {
  if (!h || !w) return fail3("null argument");
  DeviceGuard g(h->device);
  CU3_OK(cudaMemcpyAsync(warm_of(h), w, h->rs() * (size_t)h->n * h->model.nv, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int Cassie3dBatchStep(Cassie3dBatch* h, const void* action, int n_substeps, double z_done, int auto_reset, uint8_t* done,
                      void* stream) {
  if (!h) return fail3("null handle");
  if (n_substeps < 0) return fail3("n_substeps must not be negative");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  return DISPATCH3(h, step<float>(h, action, n_substeps, z_done, auto_reset, done, s),
                   step<double>(h, action, n_substeps, z_done, auto_reset, done, s));
}

int Cassie3dBatchStepHost(Cassie3dBatch* h, const void* action, int n_substeps, double z_done, int auto_reset,
                          void* qpos_out, void* qvel_out, uint8_t* done_out) {
  if (!h) return fail3("null handle");
  DeviceGuard g(h->device);
  cudaStream_t s = h->own_stream;
  const size_t n = (size_t)h->n;
  if (action) CU3_OK(cudaMemcpyAsync(h->d_action, action, h->rs() * n * h->model.nu, cudaMemcpyHostToDevice, s));
  if (DISPATCH3(h, step<float>(h, action ? h->d_action : nullptr, n_substeps, z_done, auto_reset, h->d_done, s),
                step<double>(h, action ? h->d_action : nullptr, n_substeps, z_done, auto_reset, h->d_done, s)))
    return -1;
  if (qpos_out) CU3_OK(cudaMemcpyAsync(qpos_out, qpos_of(h), h->rs() * n * h->model.nq, cudaMemcpyDeviceToHost, s));
  if (qvel_out) CU3_OK(cudaMemcpyAsync(qvel_out, qvel_of(h), h->rs() * n * h->model.nv, cudaMemcpyDeviceToHost, s));
  if (done_out) CU3_OK(cudaMemcpyAsync(done_out, h->d_done, n, cudaMemcpyDeviceToHost, s));
  CU3_OK(cudaStreamSynchronize(s));
  return 0;
}

int Cassie3dBatchGetStats(Cassie3dBatch* h, int32_t* stats, void* stream) {
  if (!h || !stats) return fail3("null argument");
  DeviceGuard g(h->device);
  CU3_OK(cudaMemcpyAsync(stats, stats_of(h), sizeof(int32_t) * 4 * (size_t)h->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int Cassie3dBatchGetResets(Cassie3dBatch* h, int32_t* resets, void* stream) {
  if (!h || !resets) return fail3("null argument");
  DeviceGuard g(h->device);
  CU3_OK(cudaMemcpyAsync(resets, resets_of(h), sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

int Cassie3dBatchSetPdGains(Cassie3dBatch* h, const double* kp, const double* kd) {
  if (!h || !kp || !kd) return fail3("null argument");
  h->kp.assign(kp, kp + h->model.nu);
  h->kd.assign(kd, kd + h->model.nu);
  return 0;
}

int Cassie3dBatchEnvStep(Cassie3dBatch* h, int mode, const void* action, int n_substeps, int max_path_length, int flags,
                         void* obs, void* reward, uint8_t* done, void* stream) {
  if (check_env_step(h, mode, action, n_substeps, flags)) return -1;
  if (!obs || !reward || !done) return fail3("null argument");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  return DISPATCH3(h, env_step<float>(h, mode, action, n_substeps, max_path_length, flags, obs, reward, done, s),
                   env_step<double>(h, mode, action, n_substeps, max_path_length, flags, obs, reward, done, s));
}

int Cassie3dBatchEnvStepHost(Cassie3dBatch* h, int mode, const void* action, int n_substeps, int max_path_length, int flags,
                             void* obs_out, void* reward_out, uint8_t* done_out) {
  if (check_env_step(h, mode, action, n_substeps, flags)) return -1;
  DeviceGuard g(h->device);
  cudaStream_t s = h->own_stream;
  const size_t n = (size_t)h->n;
  CU3_OK(cudaMemcpyAsync(h->d_action, action, h->rs() * n * h->model.nu, cudaMemcpyHostToDevice, s));
  if (DISPATCH3(h, env_step<float>(h, mode, h->d_action, n_substeps, max_path_length, flags, h->d_obs, h->d_reward, h->d_done, s),
                env_step<double>(h, mode, h->d_action, n_substeps, max_path_length, flags, h->d_obs, h->d_reward, h->d_done, s)))
    return -1;
  if (obs_out) CU3_OK(cudaMemcpyAsync(obs_out, h->d_obs, h->rs() * n * kObsDim3d, cudaMemcpyDeviceToHost, s));
  if (reward_out) CU3_OK(cudaMemcpyAsync(reward_out, h->d_reward, h->rs() * n, cudaMemcpyDeviceToHost, s));
  if (done_out) CU3_OK(cudaMemcpyAsync(done_out, h->d_done, n, cudaMemcpyDeviceToHost, s));
  CU3_OK(cudaStreamSynchronize(s));
  return 0;
}

int Cassie3dBatchEnvReset(Cassie3dBatch* h, const uint8_t* mask, void* obs, void* stream) {
  if (Cassie3dBatchResetAll(h, mask, stream)) return -1;
  return obs ? Cassie3dBatchObserve(h, obs, stream) : 0;
}

int Cassie3dBatchObserve(Cassie3dBatch* h, void* obs, void* stream) {
  if (!h || !obs) return fail3("null argument");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  return DISPATCH3(h, observe<float>(h, obs, s), observe<double>(h, obs, s));
}

int Cassie3dBatchRolloutMlp(Cassie3dBatch* h, int mode, int n_hidden, const int32_t* hidden_sizes, const void* params_dev,
                            int n_params, int n_policy_steps, int n_substeps, int max_path_length, int normalize,
                            unsigned long long seed, unsigned int first_global_env, void* obs_dev, void* action_dev,
                            void* mean_dev, void* reward_dev, uint8_t* done_dev, void* stream) {
  if (!h || !hidden_sizes || !params_dev || !obs_dev || !action_dev || !mean_dev || !reward_dev || !done_dev)
    return fail3("null argument");
  if (mode != CASSIE3D_MODE_TORQUE && mode != CASSIE3D_MODE_PD) return fail3("mode must be CASSIE3D_MODE_TORQUE or CASSIE3D_MODE_PD");
  if (n_policy_steps < 0) return fail3("n_policy_steps must not be negative");
  if (n_substeps < 1) return fail3("n_substeps must be at least 1");
  if (max_path_length <= 0) return fail3("max_path_length must be positive");
  if (n_hidden < 1 || n_hidden > kPolicyMaxLayers3d)
    return fail3("n_hidden is " + std::to_string(n_hidden) + ", the policy takes 1 to " + std::to_string(kPolicyMaxLayers3d) + " hidden layers");
  PolicyShape3d shape = {n_hidden, {0, 0, 0, 0}};
  for (int l = 0; l < n_hidden; l++) {
    if (hidden_sizes[l] < 1 || hidden_sizes[l] > kPolicyMaxWidth3d)
      return fail3("hidden_sizes[" + std::to_string(l) + "] is " + std::to_string(hidden_sizes[l]) + ", a hidden layer has 1 to " +
                   std::to_string(kPolicyMaxWidth3d) + " units");
    shape.width[l] = hidden_sizes[l];
  }
  const int want = policy_params3d(shape);
  if (n_params != want)
    return fail3("policy parameter vector has " + std::to_string(n_params) + " entries, expected " + std::to_string(want));
  if (h->model.nu != kPolicyAct3d) return fail3("the policy has " + std::to_string(kPolicyAct3d) + " actions, the model " + std::to_string(h->model.nu) + " motors");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  return DISPATCH3(h, rollout<float>(h, mode, shape, params_dev, n_policy_steps, n_substeps, max_path_length, normalize, seed,
                                     first_global_env, obs_dev, action_dev, mean_dev, reward_dev, done_dev, s),
                   rollout<double>(h, mode, shape, params_dev, n_policy_steps, n_substeps, max_path_length, normalize, seed,
                                   first_global_env, obs_dev, action_dev, mean_dev, reward_dev, done_dev, s));
}

int Cassie3dBatchRollout(Cassie3dBatch* h, int mode, const void* params_dev, int n_params, int n_policy_steps,
                         int n_substeps, int max_path_length, int normalize, unsigned long long seed,
                         unsigned int first_global_env, void* obs_dev, void* action_dev, void* mean_dev,
                         void* reward_dev, uint8_t* done_dev, void* stream) {
  static const int32_t kDefault[2] = {kPolicyHidden3d, kPolicyHidden3d};
  return Cassie3dBatchRolloutMlp(h, mode, 2, kDefault, params_dev, n_params, n_policy_steps, n_substeps, max_path_length,
                                 normalize, seed, first_global_env, obs_dev, action_dev, mean_dev, reward_dev, done_dev, stream);
}

int Cassie3dBatchActionBox(Cassie3dBatch* h, int mode, double* lo, double* hi) {
  if (!h || !lo || !hi) return fail3("null argument");
  if (mode != CASSIE3D_MODE_TORQUE && mode != CASSIE3D_MODE_PD) return fail3("mode must be CASSIE3D_MODE_TORQUE or CASSIE3D_MODE_PD");
  action_box(h->model, mode, lo, hi);
  return 0;
}

int Cassie3dBatchDiscountedReturns(Cassie3dBatch* h, const void* reward_dev, const uint8_t* done_dev, const void* tail_dev,
                                   double gamma, int n_policy_steps, void* returns_dev, void* stream) {
  if (!h || !reward_dev || !done_dev || !returns_dev) return fail3("null argument");
  if (n_policy_steps < 0) return fail3("n_policy_steps must not be negative");
  DeviceGuard g(h->device);
  cudaStream_t s = (cudaStream_t)stream;
  if (h->precision == 64) CU3_OK(launch_discounted_returns<double>(reward_dev, done_dev, tail_dev, gamma, n_policy_steps, h->n, returns_dev, s));
  else CU3_OK(launch_discounted_returns<float>(reward_dev, done_dev, tail_dev, gamma, n_policy_steps, h->n, returns_dev, s));
  return 0;
}

int Cassie3dBatchBaselineMoments(Cassie3dBatch* h, const void* obs_dev, const void* returns_dev, const uint8_t* done_dev,
                                 const int32_t* path_start_dev, int n_policy_steps, int32_t* path_index_dev,
                                 double* moments_dev, void* stream) {
  if (!h || !obs_dev || !returns_dev || !done_dev || !path_index_dev || !moments_dev) return fail3("null argument");
  if (n_policy_steps < 0) return fail3("n_policy_steps must not be negative");
  DeviceGuard g(h->device);
  BaselineArgs a{};
  a.obs = obs_dev; a.ret = returns_dev; a.done = done_dev; a.start = path_start_dev; a.idx = path_index_dev; a.moments = moments_dev;
  a.odim = kObsDim3d; a.T_steps = n_policy_steps; a.n = h->n;
  cudaStream_t s = (cudaStream_t)stream;
  if (h->precision == 64) CU3_OK((launch_baseline_moments<double, kMaxFeat3d, kMomentsPerThread3d>(a, s)));
  else CU3_OK((launch_baseline_moments<float, kMaxFeat3d, kMomentsPerThread3d>(a, s)));
  return 0;
}

int Cassie3dBatchAdvantages(Cassie3dBatch* h, const void* obs_dev, const void* reward_dev, const uint8_t* done_dev,
                            const int32_t* path_index_dev, const void* coeffs_dev, double gamma, double gae_lambda,
                            int n_policy_steps, void* advantages_dev, void* values_dev, void* stream) {
  if (!h || !obs_dev || !reward_dev || !done_dev || !path_index_dev || !coeffs_dev || !advantages_dev) return fail3("null argument");
  if (n_policy_steps < 0) return fail3("n_policy_steps must not be negative");
  DeviceGuard g(h->device);
  BaselineArgs a{};
  a.obs = obs_dev; a.rew = reward_dev; a.done = done_dev; a.idx = const_cast<int32_t*>(path_index_dev); a.coeffs = coeffs_dev;
  a.adv = advantages_dev; a.value = values_dev; a.odim = kObsDim3d; a.T_steps = n_policy_steps; a.n = h->n;
  a.gamma = gamma; a.lambda = gae_lambda;
  cudaStream_t s = (cudaStream_t)stream;
  if (h->precision == 64) CU3_OK((launch_advantages<double, kMaxFeat3d>(a, s)));
  else CU3_OK((launch_advantages<float, kMaxFeat3d>(a, s)));
  return 0;
}

int Cassie3dBatchGetEpisodeLengths(Cassie3dBatch* h, int32_t* ep_len, void* stream) {
  if (!h || !ep_len) return fail3("null argument");
  DeviceGuard g(h->device);
  CU3_OK(cudaMemcpyAsync(ep_len, h->ep_len, sizeof(int32_t) * (size_t)h->n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

}  // extern "C"
