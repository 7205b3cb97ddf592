// agphys.cu — kernels + C ABI (include/agphys.h) of the B200-native batched physics step.
//
// Build (product):  nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
// Build (kernel-logic harness, tests only):  g++ -x c++ -DAG_CPU_EMU ...   (never loaded by the package)
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include "../../include/agphys.h"
#include "ag_device.cuh"
#include "ag_solver.cuh"
#include "ag_feeding.cuh"
#include "ag_bathing.cuh"
#include "ag_ik.cuh"
#include "ag_cloth.cuh"
#include "ag_dressing.cuh"
#include "ag_render.cuh"
#include "ag_scratch.cuh"

#ifndef AG_CPU_EMU
#include <cuda_runtime.h>
#define AG_GLOBAL __global__
#else
#define AG_GLOBAL
typedef void* cudaStream_t;
enum cudaMemcpyKind { cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2 };
#endif

static thread_local std::string g_err;
static int fail(const std::string& m) { g_err = m; return -1; }

// ------------------------------------------------------------------ kernel wrappers
#ifndef AG_CPU_EMU
#define AG_KERNEL(name, body)                                                   \
  __global__ void __launch_bounds__(128) name(SimDev S, KP p) {                 \
    int tid = blockIdx.x * blockDim.x + threadIdx.x;                            \
    if (tid < p.n) body(tid, S, p);                                             \
  }
#else
#define AG_KERNEL(name, body) \
  static void name(SimDev S, KP p) { for (int tid = 0; tid < p.n; tid++) body(tid, S, p); }
#endif

#ifndef AG_CPU_EMU
#define AG_KERNEL_B(name, body, minblocks)                                      \
  __global__ void __launch_bounds__(128, minblocks) name(SimDev S, KP p) {      \
    int tid = blockIdx.x * blockDim.x + threadIdx.x;                            \
    if (tid < p.n) body(tid, S, p);                                             \
  }
#else
#define AG_KERNEL_B(name, body, minblocks) AG_KERNEL(name, body)
#endif
AG_KERNEL(k_fk, fk_body)
AG_KERNEL(k_aabb, aabb_body)
AG_KERNEL(k_linkaabb, linkaabb_body)
AG_KERNEL(k_pairs, pairs_body)
AG_KERNEL(k_csort, csort_body)
AG_KERNEL_B(k_narrow, narrow_body, 3)
AG_KERNEL(k_sort, sort_body)
AG_KERNEL(k_dyn, dyn_body)
AG_KERNEL(k_rows, rows_body)
AG_KERNEL(k_crows, crows_body)
// k_pgs: one warp per CTA = four envs, eight lanes each; per-env shared memory = velocity deltas + impulses +
// a two-deep ring of 2 KB row-stream chunks filled by TMA bulk copies (see ag_solver.cuh).
// k_order: heaviest-first env order for k_pgs (64-bucket counting sort, one CTA).
#ifndef AG_CPU_EMU
__global__ void __launch_bounds__(32) k_pgs(SimDev S, KP p) {
  extern __shared__ __align__(128) float pgs_smem[];
  pgs_warp(S, pgs_smem, p.i0, blockIdx.x * 4);
}
__global__ void __launch_bounds__(1024) k_order(SimDev S, KP) {
  __shared__ int hist[64];
  if (threadIdx.x < 64) hist[threadIdx.x] = 0;
  __syncthreads();
  for (int e = threadIdx.x; e < S.N; e += blockDim.x) atomicAdd(&hist[pgs_work_bucket(S, e)], 1);
  __syncthreads();
  if (threadIdx.x == 0) { int acc = 0; for (int b = 0; b < 64; b++) { int c = hist[b]; hist[b] = acc; acc += c; } }
  __syncthreads();
  for (int e = threadIdx.x; e < S.N; e += blockDim.x) S.pgs_order[atomicAdd(&hist[pgs_work_bucket(S, e)], 1)] = e;
}
#else
static void k_pgs(SimDev S, KP p) {
  std::vector<float> buf((size_t)rs_env_floats(S) + 8);
  float* base = (float*)(((uintptr_t)buf.data() + 15) & ~(uintptr_t)15);
  static const bool emul = getenv("AG_EMU_PLAIN_PGS") == nullptr;     // default: the restatement of the device loop
  for (int tid = 0; tid < p.n; tid++) { if (emul) pgs_env_emul(tid, S, base); else pgs_body_host(tid, S, base); }
}
static void k_order(SimDev S, KP) {
  int hist[64] = {0};
  for (int e = 0; e < S.N; e++) hist[pgs_work_bucket(S, e)]++;
  int acc = 0; for (int b = 0; b < 64; b++) { int c = hist[b]; hist[b] = acc; acc += c; }
  for (int e = 0; e < S.N; e++) S.pgs_order[hist[pgs_work_bucket(S, e)]++] = e;
}
#endif
AG_KERNEL(k_integrate, integrate_body)
AG_KERNEL(k_gather, gather_body)
AG_KERNEL(k_scatter, scatter_body)
AG_KERNEL(k_linkstate, linkstate_body)
AG_KERNEL(k_contact_query, contact_query_body)
AG_KERNEL(k_closest, closest_body)
AG_KERNEL(k_feed_pre, feeding_pre_body)
AG_KERNEL(k_feed_food, feeding_food_body)
AG_KERNEL(k_feed_post, feeding_post_body)
AG_KERNEL(k_ik, ik_body)
AG_KERNEL(k_bath_pre, bathing_pre_body)
AG_KERNEL(k_bath_dist, bathing_dist_body)
AG_KERNEL(k_bath_post, bathing_post_body)
AG_KERNEL(k_dress_pre, dressing_pre_body)
AG_KERNEL(k_dress_post, dressing_post_body)
AG_KERNEL(k_scratch_pre, scratch_pre_body)
AG_KERNEL(k_scratch_post, scratch_post_body)
AG_KERNEL(k_render, render_body)
AG_KERNEL(k_cloth_snap, cloth_snap_body)
AG_KERNEL(k_cloth_follow, cloth_follow_body)

// ------------------------------------------------------------------ host object
// The fused env steps (action -> PD targets -> frame_skip substeps -> obs / reward / done / info in one call): one record per task.
enum FusedTask { FT_FEEDING, FT_BATHING, FT_DRESSING, FT_SCRATCH, FT_COUNT };
static const char* const fused_name[FT_COUNT] = {"feeding", "bathing", "dressing", "scratch"};
struct AgSim;
typedef int (*StepEnqueue)(AgSim*, const float*, float*, float*, float*, float*);
// CUDA-graph replay of a fused step, keyed by its device pointers
struct StepGraph { void* exec = nullptr; const void* key[5] = {}; uint64_t launches = 0; bool valid = false; };
struct FusedStep {
  int obs_dim = 0;
  StepEnqueue enqueue = nullptr;                // enqueues the task's kernels on the sim's stream
  float *d_action = nullptr, *d_obs = nullptr, *d_reward = nullptr, *d_done = nullptr, *d_info = nullptr;   // the task's own device I/O
  float *h_in = nullptr, *h_out = nullptr;      // pinned staging of the host-buffer step: [N][7] and [N][obs_dim + 6]
  StepGraph graph;
  bool ready = false;                           // the task's init has run
};

struct AgSim {
  SimDev S;
  AgConfig cfg;
  int device;
  cudaStream_t stream;
  uint64_t launches;
  std::vector<void*> allocs;
  // host copies of template info needed by the API
  std::vector<int> body_link0, body_nlinks, body_kind, link_body;
  int nl, nb;
  // staging
  float* d_stage; size_t stage_floats;
  std::vector<float> h_stage;
  int* d_mask; int* d_links; int* d_icount;
  // the fused env steps' per-task state
  FeedDev F; FeedDev* F_dev;
  BathDev B; BathDev* B_dev;
  DressPost DP; DressPost* DP_dev;
  ScratchDev SD; ScratchDev* SD_dev;
  FusedStep fused[FT_COUNT];
  bool use_graph; int graph_failures;       // CUDA-graph replay of the fused steps
  // cloth (Dressing): one k_cloth launch per stepSimulation = `C.K` rigid substeps
  ClothDev C; ClothDev* C_dev; bool cloth; int cloth_sub, cloth_npt, cloth_qs;
  size_t render_pix; int render_n; int* d_render_ids; unsigned char* d_render_rgba; float* d_render_depth; void* d_render_dev;
  // profiling
  bool profiling;
  std::vector<std::string> knames;
  std::vector<int> ev_slot;
  std::vector<void*> ev_begin, ev_end;
};

#ifndef AG_CPU_EMU
#define CK(x) do { cudaError_t err__ = (x); if (err__ != cudaSuccess) { g_err = std::string(#x) + ": " + cudaGetErrorString(err__); return -1; } } while (0)
#define CKP(x) do { cudaError_t err__ = (x); if (err__ != cudaSuccess) { g_err = std::string(#x) + ": " + cudaGetErrorString(err__); return nullptr; } } while (0)
#endif

static void* dev_alloc(AgSim* s, size_t bytes) {
  void* p = nullptr;
  if (bytes == 0) bytes = 16;
#ifndef AG_CPU_EMU
  if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
  // zero on the sim's OWN stream: it is a non-blocking stream, so a cudaMemset on the legacy default stream would not be
  // ordered against the copies / kernels that use the buffer next (a staging buffer grown inside an API call was
  // sometimes zeroed AFTER the host data had been copied into it)
  if (s->stream) cudaMemsetAsync(p, 0, bytes, s->stream); else { cudaMemset(p, 0, bytes); cudaDeviceSynchronize(); }
#else
  p = calloc(1, bytes);
#endif
  s->allocs.push_back(p);
  return p;
}
static int h2d(AgSim* s, void* d, const void* h, size_t bytes) {
#ifndef AG_CPU_EMU
  CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s->stream));
  CK(cudaStreamSynchronize(s->stream));
#else
  (void)s; memcpy(d, h, bytes);
#endif
  return 0;
}
static int d2h(AgSim* s, void* h, const void* d, size_t bytes) {
#ifndef AG_CPU_EMU
  CK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
#else
  (void)s; memcpy(h, d, bytes);
#endif
  return 0;
}
static int dev_zero(AgSim* s, void* d, size_t bytes) {
#ifndef AG_CPU_EMU
  CK(cudaMemsetAsync(d, 0, bytes, s->stream));
#else
  (void)s; memset(d, 0, bytes);
#endif
  return 0;
}
// a copy enqueued on the sim's stream; unlike h2d / d2h it does not wait for it
static int copy_async(AgSim* s, void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
#ifndef AG_CPU_EMU
  CK(cudaMemcpyAsync(dst, src, bytes, kind, s->stream));
#else
  (void)s; (void)kind; memcpy(dst, src, bytes);
#endif
  return 0;
}
static int pinned_alloc(float** p, size_t floats) {
#ifndef AG_CPU_EMU
  CK(cudaMallocHost((void**)p, sizeof(float) * floats));
#else
  if (!(*p = (float*)malloc(sizeof(float) * floats))) return fail("host allocation failed");
#endif
  return 0;
}
static void pinned_free(float* p) {
#ifndef AG_CPU_EMU
  if (p) cudaFreeHost(p);
#else
  free(p);
#endif
}
static void drop_graph(StepGraph& G) {
#ifndef AG_CPU_EMU
  if (G.valid) cudaGraphExecDestroy((cudaGraphExec_t)G.exec);
#endif
  G.valid = false;
}
// a change to state the fused steps share (a SimDev / ClothDev field a captured kernel holds by value) makes every captured step stale
static void drop_graphs(AgSim* s) { for (FusedStep& R : s->fused) drop_graph(R.graph); }
template <typename T>
static const T* upload(AgSim* s, const std::vector<T>& v) {
  T* d = (T*)dev_alloc(s, v.size() * sizeof(T));
  if (d && !v.empty()) h2d(s, d, v.data(), v.size() * sizeof(T));
  return d;
}
template <typename T>
static T* dalloc(AgSim* s, size_t n) { return (T*)dev_alloc(s, n * sizeof(T)); }

// per-kernel device timing (bench.py roofline): CUDA events recorded on the sim's own stream around
// every launch while profiling is enabled; resolved lazily by ag_profile_get.
#define AG_MAX_KNAMES 32
static int prof_slot(AgSim* s, const char* name);
static void prof_mark(AgSim* s, int slot, bool begin);
#ifndef AG_CPU_EMU
#define LAUNCH(sim, kern, nthreads, kp)                                                     \
  do {                                                                                      \
    KP kp__ = (kp); kp__.n = (int)(nthreads);                                               \
    if (kp__.n > 0) {                                                                       \
      int ps__ = (sim)->profiling ? prof_slot((sim), #kern) : -1;                           \
      if (ps__ >= 0) prof_mark((sim), ps__, true);                                          \
      kern<<<(kp__.n + 127) / 128, 128, 0, (sim)->stream>>>((sim)->S, kp__);                \
      if (ps__ >= 0) prof_mark((sim), ps__, false);                                         \
      (sim)->launches++;                                                                    \
    }                                                                                       \
  } while (0)
#else
#define LAUNCH(sim, kern, nthreads, kp) \
  do { KP kp__ = (kp); kp__.n = (int)(nthreads); if (kp__.n > 0) { kern((sim)->S, kp__); (sim)->launches++; } } while (0)
#endif

static int prof_slot(AgSim* s, const char* name) {
  for (size_t i = 0; i < s->knames.size(); i++) if (s->knames[i] == name) return (int)i;
  if (s->knames.size() >= AG_MAX_KNAMES) return -1;
  s->knames.push_back(name);
  return (int)s->knames.size() - 1;
}
static void prof_mark(AgSim* s, int slot, bool begin) {
#ifndef AG_CPU_EMU
  cudaEvent_t ev;
  if (cudaEventCreate(&ev) != cudaSuccess) return;
  cudaEventRecord(ev, s->stream);
  if (begin) { s->ev_slot.push_back(slot); s->ev_begin.push_back((void*)ev); } else s->ev_end.push_back((void*)ev);
#else
  (void)s; (void)slot; (void)begin;
#endif
}

static KP kp0() { KP p; memset(&p, 0, sizeof(p)); return p; }

// Every entry point runs against the sim's own GPU and leaves the caller's current device untouched (a learner may keep
// torch on cuda:0 while a sim lives on cuda:1; allocations, launches and graph replays must not land on the wrong one).
struct DevGuard {
  int prev;
  explicit DevGuard(int device) : prev(-1) {
#ifndef AG_CPU_EMU
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != device) cudaSetDevice(device); else prev = -1;
#else
    (void)device;
#endif
  }
  ~DevGuard() {
#ifndef AG_CPU_EMU
    if (prev >= 0) cudaSetDevice(prev);
#endif
  }
};

// ------------------------------------------------------------------ quaternion helpers on the host (double)
struct HQ { double x, y, z, w; };
static HQ hq_mul(HQ a, HQ b) {
  return HQ{a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y, a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x,
            a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w, a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
static void hq_mat(HQ q, double R[9]) {
  double x = q.x, y = q.y, z = q.z, w = q.w;
  R[0] = 1 - 2 * (y * y + z * z); R[1] = 2 * (x * y - z * w); R[2] = 2 * (x * z + y * w);
  R[3] = 2 * (x * y + z * w); R[4] = 1 - 2 * (x * x + z * z); R[5] = 2 * (y * z - x * w);
  R[6] = 2 * (x * z - y * w); R[7] = 2 * (y * z + x * w); R[8] = 1 - 2 * (x * x + y * y);
}

extern "C" {

const char* ag_last_error(void) { return g_err.c_str(); }

void ag_default_config(AgConfig* c) {
  c->dt = 0.02; c->num_substeps = 1; c->num_solver_iters = 50; c->erp = 0.2; c->contact_erp = 0.08;
  c->linear_slop = 1e-5; c->residual_threshold = 1e-7; c->contact_threshold = 0.02;
  c->linear_damping = 0.04; c->angular_damping = 0.04; c->max_coord_velocity = 100; c->hull_margin = 0.001;
  c->cone_friction = 1; c->gyroscopic = 1; c->max_contacts = 128;
  c->warmstart_contact = 0.0; c->warmstart_joint = 0.0;
}

AgSim* ag_create(const AgSceneDesc* d, const AgConfig* cfg, int n_envs, int device) {
  if (!d || !cfg || n_envs <= 0) { g_err = "ag_create: bad arguments"; return nullptr; }
  DevGuard guard__(device);
  AgSim* s = new AgSim();
  memset(&s->S, 0, sizeof(SimDev));
  memset(&s->F, 0, sizeof(FeedDev));
  s->cfg = *cfg; s->device = device; s->launches = 0; s->cloth = false; s->cloth_sub = 0; s->C_dev = nullptr; s->DP_dev = nullptr; s->SD_dev = nullptr; s->render_pix = 0; s->render_n = 0; s->d_render_ids = nullptr; s->d_render_rgba = nullptr; s->d_render_depth = nullptr; s->d_render_dev = nullptr; s->use_graph = true; s->graph_failures = 0; s->B_dev = nullptr; s->stream = nullptr; s->F_dev = nullptr; s->profiling = false;
  s->d_stage = nullptr; s->stage_floats = 0;
#ifndef AG_CPU_EMU
  { int ndev = 0; if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) { g_err = "no such CUDA device (is a CUDA device present? there is no CPU fallback)"; delete s; return nullptr; } }
  if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess) { g_err = "cudaStreamCreate failed"; delete s; return nullptr; }
#endif
  SimDev& S = s->S;
  const int N = n_envs;
  S.N = N;
  int sub = cfg->num_substeps > 0 ? cfg->num_substeps : 1;
  S.dt = (float)(cfg->dt / sub); S.iters = cfg->num_solver_iters; S.erp = (float)cfg->erp; S.contact_erp = (float)cfg->contact_erp;
  S.slop = (float)cfg->linear_slop; S.resid_thr = (float)cfg->residual_threshold; S.contact_thr = (float)cfg->contact_threshold;
  S.lin_damp = (float)cfg->linear_damping; S.ang_damp = (float)cfg->angular_damping; S.vmax = (float)cfg->max_coord_velocity;
  S.cone = cfg->cone_friction; S.gyro = cfg->gyroscopic; S.maxc = cfg->max_contacts > 0 ? cfg->max_contacts : 128;
  const int nb = d->n_bodies, nl = d->n_links, nc = d->n_colliders;
  S.nb = nb; S.nl = nl; S.nc = nc; S.npair = d->n_pairs; S.ncon = d->n_constraints;
  s->nb = nb; s->nl = nl;
  s->body_link0.assign(d->body_link0, d->body_link0 + nb);
  s->body_nlinks.assign(d->body_nlinks, d->body_nlinks + nb);
  s->link_body.assign(d->link_body, d->link_body + nl);

  // ---- classify bodies, live joints, dyn links
  std::vector<double> subtree(nl, 0.0);
  for (int k = nl - 1; k >= 0; k--) { subtree[k] += d->link_mass[k]; if (d->link_parent[k] >= 0) subtree[d->link_parent[k]] += subtree[k]; }
  std::vector<int> live(nl, 0), link_dl(nl, -1), body_kind(nb, BK_STATIC), body_idx(nb, -1);
  std::vector<int> free_body, art_body, art_dl0, art_nd, dl_link, dl_parent, dl_type, dl_art, dl_part0, dl_nparts;
  std::vector<float> dl_mass, dl_mc, dl_J, dl_damping, pt_mass, pt_com, pt_I;
  for (int b = 0; b < nb; b++) {
    int l0 = d->body_link0[b], nlk = d->body_nlinks[b];
    int nlive = 0;
    for (int k = l0 + 1; k < l0 + nlk; k++) {
      int jt = d->link_jtype[k];
      if ((jt == AG_JOINT_REVOLUTE || jt == AG_JOINT_PRISMATIC) && subtree[k] > 0) { live[k] = 1; nlive++; }
    }
    if (d->link_jtype[l0] == AG_JOINT_FREE_BASE && d->link_mass[l0] > 0) {
      if (nlive > 0) { g_err = "floating-base articulated bodies are not supported yet"; ag_destroy(s); return nullptr; }
      body_kind[b] = BK_FREE; body_idx[b] = (int)free_body.size(); free_body.push_back(b);
    } else if (nlive > 0) {
      body_kind[b] = BK_ART; body_idx[b] = (int)art_body.size();
      art_body.push_back(b); art_dl0.push_back((int)dl_link.size()); art_nd.push_back(nlive);
      // relative transform of each link w.r.t. the dyn link that carries it (through fixed joints only)
      std::vector<HQ> rq(nlk); std::vector<double> rp(3 * nlk, 0.0);
      for (int k = l0; k < l0 + nlk; k++) {
        int i = k - l0;
        if (k == l0) { link_dl[k] = -1; rq[i] = HQ{0, 0, 0, 1}; continue; }
        int par = d->link_parent[k];
        if (live[k]) {
          int dd = (int)dl_link.size();
          link_dl[k] = dd; rq[i] = HQ{0, 0, 0, 1}; rp[3 * i] = rp[3 * i + 1] = rp[3 * i + 2] = 0;
          dl_link.push_back(k); dl_parent.push_back(link_dl[par]); dl_type.push_back(d->link_jtype[k]); dl_art.push_back(body_idx[b]);
          dl_damping.push_back((float)d->link_damping[k]);
        } else {
          link_dl[k] = link_dl[par];
          // T_rel(k) = T_rel(par) * T_joint(k)   (fixed joint or locked joint at q=0; locked joints carry no mass)
          int pi = par - l0;
          double R[9]; hq_mat(rq[pi], R);
          for (int a = 0; a < 3; a++) rp[3 * i + a] = rp[3 * pi + a] + R[3 * a] * d->link_jpos[3 * k] + R[3 * a + 1] * d->link_jpos[3 * k + 1] + R[3 * a + 2] * d->link_jpos[3 * k + 2];
          rq[i] = hq_mul(rq[pi], HQ{d->link_jquat[4 * k], d->link_jquat[4 * k + 1], d->link_jquat[4 * k + 2], d->link_jquat[4 * k + 3]});
        }
      }
      // merged inertias + parts
      int d0 = art_dl0.back();
      for (int dd = d0; dd < d0 + nlive; dd++) {
        double m = 0, mc[3] = {0, 0, 0}, J[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        dl_part0.push_back((int)pt_mass.size());
        int np = 0;
        for (int k = l0 + 1; k < l0 + nlk; k++) {
          if (link_dl[k] != dd || d->link_mass[k] <= 0) continue;
          int i = k - l0;
          double R[9]; hq_mat(rq[i], R);
          double c[3];
          for (int a = 0; a < 3; a++) c[a] = rp[3 * i + a] + R[3 * a] * d->link_com[3 * k] + R[3 * a + 1] * d->link_com[3 * k + 1] + R[3 * a + 2] * d->link_com[3 * k + 2];
          HQ qi = hq_mul(rq[i], HQ{d->link_iquat[4 * k], d->link_iquat[4 * k + 1], d->link_iquat[4 * k + 2], d->link_iquat[4 * k + 3]});
          double Ri[9]; hq_mat(qi, Ri);
          double Ic[9];
          for (int a = 0; a < 3; a++) for (int bb = 0; bb < 3; bb++) {
            double t = 0; for (int q = 0; q < 3; q++) t += Ri[3 * a + q] * d->link_inertia[3 * k + q] * Ri[3 * bb + q];
            Ic[3 * a + bb] = t;
          }
          double mk = d->link_mass[k];
          m += mk;
          double cc = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
          for (int a = 0; a < 3; a++) { mc[a] += mk * c[a]; for (int bb = 0; bb < 3; bb++) J[3 * a + bb] += Ic[3 * a + bb] + mk * ((a == bb ? cc : 0.0) - c[a] * c[bb]); }
          pt_mass.push_back((float)mk);
          for (int a = 0; a < 3; a++) pt_com.push_back((float)c[a]);
          pt_I.push_back((float)Ic[0]); pt_I.push_back((float)Ic[4]); pt_I.push_back((float)Ic[8]);
          pt_I.push_back((float)Ic[1]); pt_I.push_back((float)Ic[2]); pt_I.push_back((float)Ic[5]);
          np++;
        }
        dl_nparts.push_back(np);
        dl_mass.push_back((float)m);
        for (int a = 0; a < 3; a++) dl_mc.push_back((float)mc[a]);
        dl_J.push_back((float)J[0]); dl_J.push_back((float)J[4]); dl_J.push_back((float)J[8]);
        dl_J.push_back((float)J[1]); dl_J.push_back((float)J[2]); dl_J.push_back((float)J[5]);
      }
    }
  }
  S.nf = (int)free_body.size(); S.nart = (int)art_body.size(); S.ND = (int)dl_link.size(); S.nparts = (int)pt_mass.size();
  for (int nd_a : art_nd) if (nd_a > AG_MAXND) { g_err = "too many DoFs in one articulated body (AG_MAXND)"; ag_destroy(s); return nullptr; }
  if (S.ND > 32) { g_err = "too many articulated DoFs per env (32)"; ag_destroy(s); return nullptr; }
  s->body_kind = body_kind;
  // movable lists
  std::vector<int> link_col0(nl, 0), link_ncol(nl, 0);
  for (int c = nc - 1; c >= 0; c--) { link_col0[d->col_link[c]] = c; link_ncol[d->col_link[c]]++; }
  std::vector<int> movcol, movlink, allcol, alllink;
  for (int k = 0; k < nl; k++) {
    int b = d->link_body[k];
    bool mov = (body_kind[b] == BK_FREE) || (body_kind[b] == BK_ART && link_dl[k] >= 0);
    if (link_ncol[k] > 0) { alllink.push_back(k); if (mov) movlink.push_back(k); }
    for (int c = link_col0[k]; c < link_col0[k] + link_ncol[k]; c++) { allcol.push_back(c); if (mov) movcol.push_back(c); }
  }
  S.nmovcol = (int)movcol.size(); S.nmovlink = (int)movlink.size(); S.nalllink = (int)alllink.size();
  S.ngr = 6 * S.ncon;

  // ---- upload template
  auto f32 = [](const double* p, size_t n) { std::vector<float> v(n); for (size_t i = 0; i < n; i++) v[i] = (float)p[i]; return v; };
  auto i32 = [](const int32_t* p, size_t n) { return std::vector<int>(p, p + n); };
  S.body_link0 = upload(s, i32(d->body_link0, nb)); S.body_nlinks = upload(s, i32(d->body_nlinks, nb));
  S.body_kind = upload(s, body_kind); S.body_idx = upload(s, body_idx);
  S.body_gravity = upload(s, f32(d->body_gravity, 3 * nb));
  S.link_body = upload(s, i32(d->link_body, nl)); S.link_parent = upload(s, i32(d->link_parent, nl));
  S.link_jtype = upload(s, i32(d->link_jtype, nl)); S.link_dl = upload(s, link_dl);
  S.link_haslimit = upload(s, i32(d->link_haslimit, nl)); S.link_col0 = upload(s, link_col0); S.link_ncol = upload(s, link_ncol);
  S.link_axis = upload(s, f32(d->link_axis, 3 * nl)); S.link_jpos = upload(s, f32(d->link_jpos, 3 * nl));
  S.link_jquat = upload(s, f32(d->link_jquat, 4 * nl)); S.link_com = upload(s, f32(d->link_com, 3 * nl));
  S.link_iquat = upload(s, f32(d->link_iquat, 4 * nl)); S.link_inertia = upload(s, f32(d->link_inertia, 3 * nl));
  S.link_mass = upload(s, f32(d->link_mass, nl)); S.link_lower = upload(s, f32(d->link_lower, nl)); S.link_upper = upload(s, f32(d->link_upper, nl));
  S.col_link = upload(s, i32(d->col_link, nc)); S.col_type = upload(s, i32(d->col_type, nc));
  S.col_v0 = upload(s, i32(d->col_v0, nc)); S.col_nv = upload(s, i32(d->col_nv, nc));
  S.col_p0 = upload(s, i32(d->col_p0, nc)); S.col_np = upload(s, i32(d->col_np, nc));
  S.col_radius = upload(s, f32(d->col_radius, nc)); S.col_thresh = upload(s, f32(d->col_thresh, nc));
  S.max_thresh = 0.f; for (int c = 0; c < nc; c++) S.max_thresh = std::max(S.max_thresh, (float)d->col_thresh[c]);
  { std::vector<float> lt(nl, 0.f); for (int c = 0; c < nc; c++) lt[d->col_link[c]] = std::max(lt[d->col_link[c]], (float)d->col_thresh[c]); S.link_thresh = upload(s, lt); } S.col_center = upload(s, f32(d->col_center, 3 * nc)); S.col_half = upload(s, f32(d->col_half, 3 * nc));
  {
    std::vector<float> vq; std::vector<int> g0(nc);
    for (int c = 0; c < nc; c++) {
      g0[c] = (int)(vq.size() / 12);
      int v0 = d->col_v0[c], nv = d->col_nv[c];
      for (int g = 0; g < (nv + 3) / 4; g++)
        for (int comp = 0; comp < 3; comp++)
          for (int k = 0; k < 4; k++) { int i = 4 * g + k; vq.push_back((float)d->verts[3 * (size_t)(v0 + (i < nv ? i : 0)) + comp]); }
    }
    if (vq.empty()) vq.resize(12, 0.f);
    S.vertq = upload(s, vq); S.col_g0 = upload(s, g0);
  }
  S.verts = upload(s, f32(d->verts, 3 * (size_t)d->n_verts)); S.planes = upload(s, f32(d->planes, 4 * (size_t)d->n_planes));
  S.pair_link = upload(s, i32(d->pair_link, 2 * (size_t)d->n_pairs));
  {
    // Broadphase work items.  A thread of k_pairs used to take a whole link pair, and the pair spoon (64 hulls) x bowl (70 hulls) is
    // 4 480 collider box tests in one thread while the other 1 300 pairs are a handful each: the kernel ended with that pair.  Pairs are
    // cut into slices of link a's colliders so that a work item is at most ~64 box tests.
    std::vector<int> sl;
    for (int p = 0; p < d->n_pairs; p++) {
      int la = d->pair_link[2 * p], lb = d->pair_link[2 * p + 1];
      int nca = link_ncol[la], ncb = link_ncol[lb];
      if (nca == 0 || ncb == 0) continue;
      int chunk = std::max(1, 64 / ncb);
      for (int c = 0; c < nca; c += chunk) { sl.push_back(la); sl.push_back(lb); sl.push_back(link_col0[la] + c); sl.push_back(std::min(chunk, nca - c)); }
    }
    S.nslice = (int)(sl.size() / 4);
    if (sl.empty()) sl.resize(4, 0);
    S.pair_slice = upload(s, sl);
  }
  S.movcol = upload(s, movcol); S.movlink = upload(s, movlink); S.allcol = upload(s, allcol); S.alllink = upload(s, alllink);
  s->S.nmovcol = (int)movcol.size();
  S.con_link = upload(s, i32(d->con_link, 2 * (size_t)S.ncon)); S.con_pivot = upload(s, f32(d->con_pivot, 6 * (size_t)S.ncon));
  S.con_quat = upload(s, f32(d->con_quat, 8 * (size_t)S.ncon)); S.con_maxforce = upload(s, f32(d->con_maxforce, S.ncon));
  S.free_body = upload(s, free_body);
  { std::vector<float> im(free_body.size()); for (size_t f = 0; f < free_body.size(); f++) im[f] = (float)(1.0 / d->link_mass[d->body_link0[free_body[f]]]); S.free_invm = upload(s, im); }
  S.art_body = upload(s, art_body); S.art_dl0 = upload(s, art_dl0); S.art_nd = upload(s, art_nd);
  {
    std::vector<int> art_voff; int acc = 0;
    for (int nd_a : art_nd) { art_voff.push_back(acc); acc += (nd_a + 7) & ~7; }
    S.art_voff = upload(s, art_voff); S.NDp = acc;
  }
  S.dl_link = upload(s, dl_link); S.dl_parent = upload(s, dl_parent); S.dl_type = upload(s, dl_type); S.dl_art = upload(s, dl_art);
  S.dl_part0 = upload(s, dl_part0); S.dl_nparts = upload(s, dl_nparts);
  S.dl_mass = upload(s, dl_mass); S.dl_mc = upload(s, dl_mc); S.dl_J = upload(s, dl_J); S.dl_damping = upload(s, dl_damping);
  S.pt_mass = upload(s, pt_mass); S.pt_com = upload(s, pt_com); S.pt_I = upload(s, pt_I);
  // ---- per-env state
  S.hard_limit = dalloc<int>(s, nl);
  S.motor_mode = dalloc<int>(s, nl); S.motor_kp = dalloc<float>(s, nl); S.motor_kd = dalloc<float>(s, nl); S.motor_maxf = dalloc<float>(s, nl);
  S.motor_target = dalloc<float>(s, (size_t)nl * N); S.motor_applied = dalloc<float>(s, (size_t)nl * N);
  S.base_pos = dalloc<float>(s, (size_t)nb * 3 * N); S.base_quat = dalloc<float>(s, (size_t)nb * 4 * N);
  S.base_lin = dalloc<float>(s, (size_t)nb * 3 * N); S.base_ang = dalloc<float>(s, (size_t)nb * 3 * N);
  S.jq = dalloc<float>(s, (size_t)nl * N); S.jqd = dalloc<float>(s, (size_t)nl * N);
  S.friction = dalloc<float>(s, (size_t)nl * N); S.body_mode = dalloc<int>(s, (size_t)nb * N);
  S.lpos = dalloc<float>(s, (size_t)nl * 3 * N); S.lquat = dalloc<float>(s, (size_t)nl * 4 * N);
  S.cmin = dalloc<float>(s, (size_t)nc * 3 * N); S.cmax = dalloc<float>(s, (size_t)nc * 3 * N);
  S.lmin = dalloc<float>(s, (size_t)nl * 3 * N); S.lmax = dalloc<float>(s, (size_t)nl * 3 * N);
  S.c_count = dalloc<int>(s, N); S.overflow = dalloc<int>(s, N); S.iters_used = dalloc<int>(s, N); S.pgs_cycles = dalloc<int>(s, N); S.pgs_trips = dalloc<int>(s, N);
  S.pgs_order = dalloc<int>(s, N);
  S.maxcand = 4 * S.maxc; S.cand_count = dalloc<int>(s, N); S.cand = dalloc<unsigned>(s, (size_t)S.maxcand * N); S.cand_s = dalloc<unsigned>(s, (size_t)S.maxcand * N);
  if ((size_t)nc * nc >= (1u << 24)) { g_err = "too many colliders (pair id must fit 24 bits)"; ag_destroy(s); return nullptr; }
  S.maxraw = 4 * S.maxc;
  S.c_key = dalloc<unsigned>(s, (size_t)S.maxraw * N); S.s_key = dalloc<unsigned>(s, (size_t)S.maxc * N);
  S.c_data = dalloc<float>(s, (size_t)S.maxraw * AG_CFR * N); S.s_data = dalloc<float>(s, (size_t)S.maxc * AG_CF * N);
  S.s_ref = dalloc<int>(s, (size_t)S.maxc * 4 * N);
  S.fcom = dalloc<float>(s, (size_t)S.nf * 3 * N); S.fIinv = dalloc<float>(s, (size_t)S.nf * 6 * N);
  S.jax = dalloc<float>(s, (size_t)S.ND * 3 * N); S.jor = dalloc<float>(s, (size_t)S.ND * 3 * N);
  S.Minv = dalloc<float>(s, (size_t)S.ND * S.ND * N);
  S.dv = dalloc<float>(s, (size_t)(S.ND + 6 * S.nf) * N);
  S.dr_lam = dalloc<float>(s, (size_t)3 * S.ND * N);
  // row stream: dof rows pair up (two lane blocks for an articulation of > 8 dofs), 3 records per fixed constraint, and
  // per contact a normal row (half a record when it pairs up) + a friction record of two lane blocks; 30 % slack for
  // chunk padding and articulated sides.  An env that needs more is flagged (ag_overflow_count).
  {
    size_t fl = (size_t)(3 * S.ND / 2 + 2) * rs_rec_floats(2) + (size_t)3 * S.ncon * rs_rec_floats(3) + (size_t)S.maxc * 2 * rs_rec_floats(2);
    fl = fl + fl * 3 / 10 + 1024;
    S.rs_cap = (int)((fl + 1023) / 1024 * 1024);
  }
  if (rs_nv(S) + 8 >= 65536 || rs_nlam(S) >= 65536) { g_err = "solver index space exceeds 16 bits: lower max_contacts"; ag_destroy(s); return nullptr; }
  S.rs_data = dalloc<float>(s, (size_t)S.rs_cap * N); S.rs_nfloats = dalloc<int>(s, N);
  S.gr_lam = dalloc<float>(s, (size_t)S.ngr * N); S.row_off = dalloc<int>(s, (size_t)(3 * S.ND + S.ngr) * N); S.row_pair = dalloc<int>(s, (size_t)(3 * S.ND + S.ngr) * N);
  s->d_mask = dalloc<int>(s, N); s->d_links = dalloc<int>(s, 1024); s->d_icount = dalloc<int>(s, N);
  if (!S.gr_lam || !S.rs_data || !S.rs_nfloats || !S.row_pair || !S.s_data) { g_err = "device allocation failed"; ag_destroy(s); return nullptr; }
#ifndef AG_CPU_EMU
  {
    { const char* gg = getenv("AG_GRAPH"); if (gg && atoi(gg) == 0) s->use_graph = false; }
    size_t smem = (size_t)rs_cta_floats(S) * sizeof(float) + 32;
    if (smem > 227 * 1024) { g_err = "PGS shared-memory footprint exceeds 227 KB per CTA: lower max_contacts"; ag_destroy(s); return nullptr; }
    if (cudaFuncSetAttribute(k_pgs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { g_err = "cudaFuncSetAttribute(k_pgs) failed"; ag_destroy(s); return nullptr; }
  }
#endif
  // defaults: friction from the template, all bodies active, identity quaternions
  {
    std::vector<float> fr((size_t)nl * N);
    for (int k = 0; k < nl; k++) for (int e = 0; e < N; e++) fr[(size_t)k * N + e] = (float)d->link_friction[k];
    h2d(s, S.friction, fr.data(), fr.size() * sizeof(float));
    std::vector<int> md((size_t)nb * N, 1);
    h2d(s, S.body_mode, md.data(), md.size() * sizeof(int));
    std::vector<float> q((size_t)nb * 4 * N, 0.f);
    for (int b = 0; b < nb; b++) for (int e = 0; e < N; e++) q[((size_t)b * 4 + 3) * N + e] = 1.f;
    h2d(s, S.base_quat, q.data(), q.size() * sizeof(float));
  }
  return s;
}

void ag_destroy(AgSim* s) {
  if (!s) return;
  DevGuard guard__(s->device);
#ifndef AG_CPU_EMU
  if (s->stream) cudaStreamSynchronize(s->stream);
  for (void* p : s->allocs) cudaFree(p);
  if (s->stream) cudaStreamDestroy(s->stream);
#else
  for (void* p : s->allocs) free(p);
#endif
  for (FusedStep& R : s->fused) { pinned_free(R.h_in); pinned_free(R.h_out); drop_graph(R.graph); }
  delete s;
}

int ag_num_envs(const AgSim* s) {
  DevGuard guard__(s->device); return s->S.N; }
void* ag_stream(AgSim* s) {
  DevGuard guard__(s->device); return (void*)s->stream; }
uint64_t ag_kernel_launches(const AgSim* s) {
  DevGuard guard__(s->device); return s->launches; }

int ag_profile_enable(AgSim* s, int on) {
  DevGuard guard__(s->device);
  s->profiling = on != 0;
  return 0;
}
// Resolves the recorded events: per kernel name total milliseconds and launch count since the last call.
int ag_profile_get(AgSim* s, int max_names, char* names, int name_stride, float* total_ms, int32_t* counts) {
  DevGuard guard__(s->device);
  int n = (int)s->knames.size();
  if (n > max_names) n = max_names;
  for (int i = 0; i < n; i++) { total_ms[i] = 0.f; counts[i] = 0; snprintf(names + (size_t)i * name_stride, name_stride, "%s", s->knames[i].c_str()); }
#ifndef AG_CPU_EMU
  CK(cudaStreamSynchronize(s->stream));
  size_t m = std::min(s->ev_begin.size(), s->ev_end.size());
  for (size_t i = 0; i < m; i++) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, (cudaEvent_t)s->ev_begin[i], (cudaEvent_t)s->ev_end[i]);
    int sl = s->ev_slot[i];
    if (sl < n) { total_ms[sl] += ms; counts[sl] += 1; }
  }
  for (void* e : s->ev_begin) cudaEventDestroy((cudaEvent_t)e);
  for (void* e : s->ev_end) cudaEventDestroy((cudaEvent_t)e);
#endif
  s->ev_begin.clear(); s->ev_end.clear(); s->ev_slot.clear();
  return n;
}

// ---- staging helpers: host env-major [N][K] <-> device SoA via gather/scatter kernels
static float* stage(AgSim* s, size_t floats) {
  if (floats > s->stage_floats) {
    s->d_stage = dalloc<float>(s, floats);
    s->stage_floats = floats;
  }
  return s->d_stage;
}
static int set_mask(AgSim* s, const int32_t* mask) {
  if (!mask) return 0;
  return h2d(s, s->d_mask, mask, sizeof(int) * s->S.N);
}
// scatter host [N][K] rows into a device SoA array with `comp` components per item:
// dst[(item*comp + c)*N + e] = src[e*K + j*comp + c] for item = items[j]
static int check_items(const AgSim* s, const float* arr, int nitems, const int* items) {
  // the item-indexed arrays are per body (base_*) or per link (everything else)
  int limit = (arr == s->S.base_pos || arr == s->S.base_quat || arr == s->S.base_lin || arr == s->S.base_ang) ? s->nb : s->nl;
  if (nitems < 0 || (nitems > 0 && !items)) return fail("bad item list");
  for (int j = 0; j < nitems; j++) if (items[j] < 0 || items[j] >= limit) return fail(limit == s->nb ? "bad body" : "bad link");
  return 0;
}
static int scatter_host(AgSim* s, float* dst, int comp, int nitems, const int* items, const float* src, const int32_t* mask) {
  const int N = s->S.N;
  if (check_items(s, dst, nitems, items)) return -1;
  size_t K = (size_t)nitems * comp;
  float* st = stage(s, K * N);
  if (!st) return fail("staging alloc failed");
  if (h2d(s, st, src, K * N * sizeof(float))) return -1;
  if (nitems > 1024) return fail("too many items");
  if (h2d(s, s->d_links, items, sizeof(int) * nitems)) return -1;
  if (set_mask(s, mask)) return -1;
  KP p = kp0(); p.i0 = comp; p.i1 = nitems; p.p0 = st; p.p1 = dst; p.p2 = s->d_links; p.p3 = mask ? s->d_mask : nullptr;
  LAUNCH(s, k_scatter, (size_t)N * K, p);
  return 0;
}
static int gather_host(AgSim* s, const float* srcdev, int comp, int nitems, const int* items, float* dst) {
  const int N = s->S.N;
  if (check_items(s, srcdev, nitems, items)) return -1;
  size_t K = (size_t)nitems * comp;
  float* st = stage(s, K * N);
  if (!st) return fail("staging alloc failed");
  if (nitems > 1024) return fail("too many items");
  if (h2d(s, s->d_links, items, sizeof(int) * nitems)) return -1;
  KP p = kp0(); p.i0 = comp; p.i1 = nitems; p.p0 = srcdev; p.p1 = st; p.p2 = s->d_links;
  LAUNCH(s, k_gather, (size_t)N * K, p);
  return d2h(s, dst, st, K * N * sizeof(float));
}

int ag_set_base_pose(AgSim* s, int body, const float* pos, const float* quat, const int32_t* mask) {
  DevGuard guard__(s->device);
  if (body < 0 || body >= s->nb) return fail("bad body");
  if (pos && scatter_host(s, s->S.base_pos, 3, 1, &body, pos, mask)) return -1;
  if (quat && scatter_host(s, s->S.base_quat, 4, 1, &body, quat, mask)) return -1;
  return 0;
}
int ag_set_base_velocity(AgSim* s, int body, const float* lin, const float* ang, const int32_t* mask) {
  DevGuard guard__(s->device);
  if (body < 0 || body >= s->nb) return fail("bad body");
  if (lin && scatter_host(s, s->S.base_lin, 3, 1, &body, lin, mask)) return -1;
  if (ang && scatter_host(s, s->S.base_ang, 3, 1, &body, ang, mask)) return -1;
  return 0;
}
int ag_set_joint_state(AgSim* s, int n, const int32_t* links, const float* q, const float* qd, const int32_t* mask) {
  DevGuard guard__(s->device);
  if (q && scatter_host(s, s->S.jq, 1, n, links, q, mask)) return -1;
  if (qd && scatter_host(s, s->S.jqd, 1, n, links, qd, mask)) return -1;
  return 0;
}
int ag_set_link_friction(AgSim* s, int link, const float* mu, const int32_t* mask) {
  DevGuard guard__(s->device);
  return scatter_host(s, s->S.friction, 1, 1, &link, mu, mask);
}
int ag_set_body_active(AgSim* s, int body, const int32_t* active) {
  DevGuard guard__(s->device);
  if (body < 0 || body >= s->nb) return fail("bad body");
  return h2d(s, s->S.body_mode + (size_t)body * s->S.N, active, sizeof(int) * s->S.N);
}

int ag_set_hard_limits(AgSim* s, int n, const int32_t* links, int on) {
  DevGuard guard__(s->device);
  std::vector<int> h(s->nl);
  if (d2h(s, h.data(), s->S.hard_limit, sizeof(int) * s->nl)) return -1;
  for (int j = 0; j < n; j++) { if (links[j] < 0 || links[j] >= s->nl) return fail("bad link"); h[links[j]] = on ? 1 : 0; }
  return h2d(s, s->S.hard_limit, h.data(), sizeof(int) * s->nl);
}

static void run_fk_all(AgSim* s) {
  KP p = kp0(); p.i0 = 1;
  LAUNCH(s, k_fk, (size_t)s->S.nb * s->S.N, p);
  KP a = kp0(); a.p0 = s->S.allcol; a.i0 = s->S.nc;
  LAUNCH(s, k_aabb, (size_t)s->S.nc * s->S.N, a);
  KP l = kp0(); l.p0 = s->S.alllink; l.i0 = s->S.nalllink;
  LAUNCH(s, k_linkaabb, (size_t)s->S.nalllink * s->S.N, l);
}

int ag_set_body_gravity(AgSim* s, int body, const double g[3]) {
  DevGuard guard__(s->device);
  if (body < 0 || body >= s->nb) return fail("bad body");
  float gf[3] = {(float)g[0], (float)g[1], (float)g[2]};
  return h2d(s, (float*)s->S.body_gravity + 3 * body, gf, sizeof(gf));        // a template table shared by the envs; kernels read it at launch
}
int ag_get_link_aabb(AgSim* s, int n, const int32_t* links, float* aabb_min, float* aabb_max) {
  DevGuard guard__(s->device);
  run_fk_all(s);
  if (gather_host(s, s->S.lmin, 3, n, links, aabb_min)) return -1;
  return gather_host(s, s->S.lmax, 3, n, links, aabb_max);
}
int ag_forward_kinematics(AgSim* s) {
  DevGuard guard__(s->device); run_fk_all(s); return 0; }

int ag_set_motor_host(AgSim* s, int n, const int32_t* links, int mode, const float* target, const float* kp, const float* kd, const float* maxf) {
  DevGuard guard__(s->device);
  std::vector<int> mm(s->nl); std::vector<float> a(s->nl), b(s->nl), c(s->nl);
  if (d2h(s, mm.data(), s->S.motor_mode, sizeof(int) * s->nl) || d2h(s, a.data(), s->S.motor_kp, sizeof(float) * s->nl) ||
      d2h(s, b.data(), s->S.motor_kd, sizeof(float) * s->nl) || d2h(s, c.data(), s->S.motor_maxf, sizeof(float) * s->nl)) return -1;
  for (int j = 0; j < n; j++) {
    int k = links[j]; if (k < 0 || k >= s->nl) return fail("bad link");
    mm[k] = mode; if (kp) a[k] = kp[j]; b[k] = kd ? kd[j] : 1.0f; if (maxf) c[k] = maxf[j];
  }
  if (h2d(s, s->S.motor_mode, mm.data(), sizeof(int) * s->nl) || h2d(s, s->S.motor_kp, a.data(), sizeof(float) * s->nl) ||
      h2d(s, s->S.motor_kd, b.data(), sizeof(float) * s->nl) || h2d(s, s->S.motor_maxf, c.data(), sizeof(float) * s->nl)) return -1;
  if (target) return scatter_host(s, s->S.motor_target, 1, n, links, target, nullptr);
  return 0;
}
int ag_set_motor_force_scale(AgSim* s, int n, const int32_t* links, const float* scale) {
  DevGuard guard__(s->device);
  if (!s->S.motor_fscale) {
    const size_t cnt = (size_t)s->nl * s->S.N;
    s->S.motor_fscale = dalloc<float>(s, cnt);
    if (!s->S.motor_fscale) return fail("device allocation failed");
    std::vector<float> ones(cnt, 1.0f);
    if (h2d(s, s->S.motor_fscale, ones.data(), cnt * sizeof(float))) return -1;
    drop_graphs(s);                                       // captured kernels hold the SimDev of before (null pointer)
  }
  return scatter_host(s, s->S.motor_fscale, 1, n, links, scale, nullptr);
}
int ag_set_motor_targets_dev(AgSim* s, int n, const int32_t* links, const float* target_dev) {
  DevGuard guard__(s->device);
  if (n > 1024) return fail("too many items");
  if (check_items(s, s->S.motor_target, n, links)) return -1;
  if (h2d(s, s->d_links, links, sizeof(int) * n)) return -1;
  KP p = kp0(); p.i0 = 1; p.i1 = n; p.p0 = target_dev; p.p1 = s->S.motor_target; p.p2 = s->d_links; p.p3 = nullptr;
  LAUNCH(s, k_scatter, (size_t)s->S.N * n, p);
  return 0;
}

int ag_set_motor_targets_host(AgSim* s, int n, const int32_t* links, const float* target) {
  DevGuard guard__(s->device);
  return scatter_host(s, s->S.motor_target, 1, n, links, target, nullptr);
}

static void cloth_launch(AgSim* s);
static void substep(AgSim* s) {
  SimDev& S = s->S;
  const int N = S.N;
  KP z = kp0();
  LAUNCH(s, k_fk, (size_t)S.nb * N, z);
  if (s->cloth) {                                      // the cloth collides with the link poses at the START of the substep
    KP cs = kp0(); cs.p0 = s->C_dev; cs.i0 = s->cloth_sub;
    LAUNCH(s, k_cloth_snap, (size_t)s->C.ncl * N, cs);
  }
  KP a = kp0(); a.p0 = S.movcol; a.i0 = S.nmovcol;
  LAUNCH(s, k_aabb, (size_t)S.nmovcol * N, a);
  KP l = kp0(); l.p0 = S.movlink; l.i0 = S.nmovlink;
  LAUNCH(s, k_linkaabb, (size_t)S.nmovlink * N, l);
  dev_zero(s, S.c_count, sizeof(int) * N);
  dev_zero(s, S.cand_count, sizeof(int) * N);
  int Npad = (N + 31) / 32 * 32;
  KP c = kp0(); c.i0 = Npad;
  LAUNCH(s, k_pairs, (size_t)S.nslice * Npad, c);
  LAUNCH(s, k_csort, (size_t)S.maxcand * N, z);
  LAUNCH(s, k_narrow, (size_t)S.maxcand * N, z);
  LAUNCH(s, k_sort, (size_t)S.maxraw * N, z);
  LAUNCH(s, k_dyn, (size_t)(S.nf + S.nart) * N, z);
  LAUNCH(s, k_rows, N, z);
  LAUNCH(s, k_crows, (size_t)(S.maxc + 3 * S.ND + S.ngr) * N, z);
#ifndef AG_CPU_EMU
  {
    int ps = s->profiling ? prof_slot(s, "k_order") : -1;
    if (ps >= 0) prof_mark(s, ps, true);
    k_order<<<1, 1024, 0, s->stream>>>(S, z);
    if (ps >= 0) prof_mark(s, ps, false);
    KP kp = z; kp.n = N;
    size_t smem = (size_t)rs_cta_floats(S) * sizeof(float) + 32;
    ps = s->profiling ? prof_slot(s, "k_pgs") : -1;
    if (ps >= 0) prof_mark(s, ps, true);
    k_pgs<<<(N + 3) / 4, 32, smem, s->stream>>>(S, kp);
    if (ps >= 0) prof_mark(s, ps, false);
    s->launches += 2;
  }
#else
  k_order(S, z);
  LAUNCH(s, k_pgs, N, z);
  LAUNCH(s, k_integrate, N, z);                      // (fused into k_pgs on the device)
#endif
  if (s->cloth && ++s->cloth_sub == s->C.K) { s->cloth_sub = 0; cloth_launch(s); }
}

int ag_step(AgSim* s, int n_steps) {
  DevGuard guard__(s->device);
  int sub = s->cfg.num_substeps > 0 ? s->cfg.num_substeps : 1;
  for (int i = 0; i < n_steps * sub; i++) substep(s);
  KP z = kp0();
  LAUNCH(s, k_fk, (size_t)s->S.nb * s->S.N, z);
#ifndef AG_CPU_EMU
  CK(cudaGetLastError());
#endif
  return 0;
}

int ag_get_joint_states(AgSim* s, int n, const int32_t* links, float* q, float* qd, float* tau) {
  DevGuard guard__(s->device);
  if (q && gather_host(s, s->S.jq, 1, n, links, q)) return -1;
  if (qd && gather_host(s, s->S.jqd, 1, n, links, qd)) return -1;
  if (tau && gather_host(s, s->S.motor_applied, 1, n, links, tau)) return -1;
  return 0;
}

int ag_get_link_states(AgSim* s, int n, const int32_t* links, float* pos, float* quat, float* com_pos, float* com_quat, float* lin_vel, float* ang_vel) {
  DevGuard guard__(s->device);
  const int N = s->S.N;
  if (n > 1024) return fail("too many items");
  for (int j = 0; j < n; j++) if (links[j] < 0 || links[j] >= s->nl) return fail("bad link");
  // out record per (env, link): 20 floats: pos3 quat4 cpos3 cquat4 lin3 ang3
  float* st = stage(s, (size_t)N * n * 20);
  if (!st) return fail("staging alloc failed");
  if (h2d(s, s->d_links, links, sizeof(int) * n)) return -1;
  KP p = kp0(); p.i1 = n; p.p1 = st; p.p2 = s->d_links;
  LAUNCH(s, k_linkstate, (size_t)N * n, p);
  s->h_stage.resize((size_t)N * n * 20);
  if (d2h(s, s->h_stage.data(), st, sizeof(float) * s->h_stage.size())) return -1;
  for (size_t i = 0; i < (size_t)N * n; i++) {
    const float* r = &s->h_stage[i * 20];
    if (pos) memcpy(pos + 3 * i, r, 12);
    if (quat) memcpy(quat + 4 * i, r + 3, 16);
    if (com_pos) memcpy(com_pos + 3 * i, r + 7, 12);
    if (com_quat) memcpy(com_quat + 4 * i, r + 10, 16);
    if (lin_vel) memcpy(lin_vel + 3 * i, r + 14, 12);
    if (ang_vel) memcpy(ang_vel + 3 * i, r + 17, 12);
  }
  return 0;
}

static int contact_query(AgSim* s, int body_a, int body_b, int link_a, int link_b, int max_pts, AgContact* out, int32_t* count, float* fsum) {
  const int N = s->S.N;
  if (body_a < 0 || body_a >= s->nb || body_b >= s->nb) return fail("bad body");
  if (max_pts < 0) return fail("bad max_pts");
  if (link_a >= s->body_nlinks[body_a] - 1 || (body_b >= 0 && link_b >= s->body_nlinks[body_b] - 1)) return fail("bad link");
  size_t rec = sizeof(AgContact) / sizeof(float);
  float* st = stage(s, (size_t)N * max_pts * rec + (size_t)N);
  if (!st) return fail("staging alloc failed");
  KP p = kp0();
  p.i0 = body_a; p.i1 = body_b; p.i2 = link_a < -1 ? -2 : (link_a < 0 ? s->body_link0[body_a] : s->body_link0[body_a] + 1 + link_a);
  p.i3 = (body_b < 0 || link_b < -1) ? -2 : (link_b < 0 ? s->body_link0[body_b] : s->body_link0[body_b] + 1 + link_b);
  p.f0 = (float)max_pts; p.p1 = st; p.p2 = s->d_icount; p.p3 = st + (size_t)N * max_pts * rec;
  LAUNCH(s, k_contact_query, N, p);
  if (out && max_pts > 0 && d2h(s, out, st, (size_t)N * max_pts * sizeof(AgContact))) return -1;
  if (count && d2h(s, count, s->d_icount, sizeof(int) * N)) return -1;
  if (fsum && d2h(s, fsum, st + (size_t)N * max_pts * rec, sizeof(float) * N)) return -1;
  return 0;
}
int ag_get_contacts(AgSim* s, int body_a, int body_b, int link_a, int link_b, int max_pts, AgContact* out, int32_t* count) {
  DevGuard guard__(s->device);
  return contact_query(s, body_a, body_b, link_a, link_b, max_pts, out, count, nullptr);
}
int ag_contact_force_sum(AgSim* s, int body_a, int body_b, int link_a, int link_b, float* out) {
  DevGuard guard__(s->device);
  return contact_query(s, body_a, body_b, link_a, link_b, 0, nullptr, nullptr, out);
}
int ag_closest_points(AgSim* s, int body_a, int body_b, float distance, int max_pts, AgContact* out, int32_t* count) {
  DevGuard guard__(s->device);
  const int N = s->S.N;
  if (body_a < 0 || body_a >= s->nb || body_b < 0 || body_b >= s->nb) return fail("bad body");
  run_fk_all(s);
  size_t rec = sizeof(AgContact) / sizeof(float);
  float* st = stage(s, (size_t)N * std::max(1, max_pts) * rec);
  if (!st) return fail("staging alloc failed");
  KP p = kp0(); p.i0 = body_a; p.i1 = body_b; p.i2 = max_pts; p.f0 = distance; p.p1 = st; p.p2 = s->d_icount;
  LAUNCH(s, k_closest, N, p);
  if (out && max_pts > 0 && d2h(s, out, st, (size_t)N * max_pts * sizeof(AgContact))) return -1;
  if (count && d2h(s, count, s->d_icount, sizeof(int) * N)) return -1;
  return 0;
}

int ag_ik_solve(AgSim* s, int n_joints, const int32_t* joint_links, int ee_link, const float* target_pos, const float* target_quat,
                int max_restarts, int iters, float threshold, uint64_t seed, const int32_t* env_mask, float* q_out, float* err_out) {
  DevGuard guard__(s->device);
  const int N = s->S.N;
  if (n_joints < 1 || n_joints > AG_IK_MAXJ) return fail("ag_ik_solve: 1..8 joints");
  if (ee_link < 0 || ee_link >= s->nl) return fail("bad link");
  std::vector<int> parent(s->nl), jtype(s->nl);
  std::vector<float> lo(s->nl), hi(s->nl);
  d2h(s, parent.data(), s->S.link_parent, sizeof(int) * s->nl); d2h(s, jtype.data(), s->S.link_jtype, sizeof(int) * s->nl);
  d2h(s, lo.data(), s->S.link_lower, sizeof(float) * s->nl); d2h(s, hi.data(), s->S.link_upper, sizeof(float) * s->nl);
  IkDev K; memset(&K, 0, sizeof(K));
  K.body = s->link_body[ee_link]; K.ee_link = ee_link; K.n_joints = n_joints; K.max_restarts = max_restarts; K.iters = iters;
  K.threshold = threshold; K.damping = 0.05f; K.step_clip = 0.2f; K.seed = seed;
  std::vector<int> chain;
  for (int k = ee_link; k >= 0 && k != s->body_link0[K.body]; k = parent[k]) chain.push_back(k);
  if ((int)chain.size() > AG_IK_MAXCHAIN) return fail("ag_ik_solve: chain too long");
  std::reverse(chain.begin(), chain.end());
  K.n_chain = (int)chain.size();
  for (int i = 0; i < K.n_chain; i++) { K.chain[i] = chain[i]; K.chain_joint[i] = -1; }
  for (int j = 0; j < n_joints; j++) {
    int k = joint_links[j], at = -1;
    for (int i = 0; i < K.n_chain; i++) if (chain[i] == k) at = i;
    if (at < 0 || (jtype[k] != 1 && jtype[k] != 2)) return fail("ag_ik_solve: joint is not a movable joint on the path to the end effector");
    K.chain_joint[at] = j; K.lower[j] = lo[k]; K.upper[j] = hi[k]; K.col_jtype[j] = jtype[k];
  }
  size_t nfl = ((size_t)N * (3 + 4 + n_joints + 1) + 3) & ~(size_t)3;     // IkDev holds a 64-bit seed: keep it 16-byte aligned
  float* st = stage(s, nfl + (sizeof(IkDev) + 3) / 4);
  if (!st) return fail("staging alloc failed");
  float *d_tp = st, *d_tq = st + (size_t)N * 3, *d_q = d_tq + (size_t)N * 4, *d_err = d_q + (size_t)N * n_joints;
  IkDev* d_K = (IkDev*)(st + nfl);
  if (h2d(s, d_tp, target_pos, sizeof(float) * 3 * N) || h2d(s, d_tq, target_quat, sizeof(float) * 4 * N) || h2d(s, d_K, &K, sizeof(IkDev))) return -1;
  if (set_mask(s, env_mask)) return -1;
  KP p = kp0(); p.p0 = d_K; p.p1 = d_tp; p.p2 = d_tq; p.p3 = d_q; p.p4 = d_err; p.p5 = env_mask ? s->d_mask : nullptr;
  LAUNCH(s, k_ik, N, p);
  if (d2h(s, q_out, d_q, sizeof(float) * n_joints * N) || d2h(s, err_out, d_err, sizeof(float) * N)) return -1;
  return 0;
}

size_t ag_state_size(const AgSim* s) {
  DevGuard guard__(s->device); return (size_t)s->nb * 13 + (size_t)s->nl * 2; }
int ag_state_get(AgSim* s, float* out) {
  DevGuard guard__(s->device);
  const int N = s->S.N; size_t sz = ag_state_size(s);
  std::vector<float> bp((size_t)s->nb * 3 * N), bq((size_t)s->nb * 4 * N), bl((size_t)s->nb * 3 * N), ba((size_t)s->nb * 3 * N), q((size_t)s->nl * N), qd((size_t)s->nl * N);
  if (d2h(s, bp.data(), s->S.base_pos, bp.size() * 4) || d2h(s, bq.data(), s->S.base_quat, bq.size() * 4) ||
      d2h(s, bl.data(), s->S.base_lin, bl.size() * 4) || d2h(s, ba.data(), s->S.base_ang, ba.size() * 4) ||
      d2h(s, q.data(), s->S.jq, q.size() * 4) || d2h(s, qd.data(), s->S.jqd, qd.size() * 4)) return -1;
  for (int e = 0; e < N; e++) {
    float* o = out + sz * e;
    for (int b = 0; b < s->nb; b++) {
      for (int a = 0; a < 3; a++) { o[a] = bp[((size_t)b * 3 + a) * N + e]; o[7 + a] = bl[((size_t)b * 3 + a) * N + e]; o[10 + a] = ba[((size_t)b * 3 + a) * N + e]; }
      for (int a = 0; a < 4; a++) o[3 + a] = bq[((size_t)b * 4 + a) * N + e];
      o += 13;
    }
    for (int k = 0; k < s->nl; k++) { o[0] = q[(size_t)k * N + e]; o[1] = qd[(size_t)k * N + e]; o += 2; }
  }
  return 0;
}
int ag_state_set(AgSim* s, const float* in) {
  DevGuard guard__(s->device);
  const int N = s->S.N; size_t sz = ag_state_size(s);
  std::vector<float> bp((size_t)s->nb * 3 * N), bq((size_t)s->nb * 4 * N), bl((size_t)s->nb * 3 * N), ba((size_t)s->nb * 3 * N), q((size_t)s->nl * N), qd((size_t)s->nl * N);
  for (int e = 0; e < N; e++) {
    const float* o = in + sz * e;
    for (int b = 0; b < s->nb; b++) {
      for (int a = 0; a < 3; a++) { bp[((size_t)b * 3 + a) * N + e] = o[a]; bl[((size_t)b * 3 + a) * N + e] = o[7 + a]; ba[((size_t)b * 3 + a) * N + e] = o[10 + a]; }
      for (int a = 0; a < 4; a++) bq[((size_t)b * 4 + a) * N + e] = o[3 + a];
      o += 13;
    }
    for (int k = 0; k < s->nl; k++) { q[(size_t)k * N + e] = o[0]; qd[(size_t)k * N + e] = o[1]; o += 2; }
  }
  if (h2d(s, s->S.base_pos, bp.data(), bp.size() * 4) || h2d(s, s->S.base_quat, bq.data(), bq.size() * 4) ||
      h2d(s, s->S.base_lin, bl.data(), bl.size() * 4) || h2d(s, s->S.base_ang, ba.data(), ba.size() * 4) ||
      h2d(s, s->S.jq, q.data(), q.size() * 4) || h2d(s, s->S.jqd, qd.data(), qd.size() * 4)) return -1;
  run_fk_all(s);
  return 0;
}

int ag_get_pgs_cycles(AgSim* s, int32_t* cycles) {
  DevGuard guard__(s->device); return d2h(s, cycles, s->S.pgs_cycles, sizeof(int) * s->S.N); }
int ag_get_pgs_trips(AgSim* s, int32_t* trips, int32_t* stream_floats) {
  DevGuard guard__(s->device);
  if (trips && d2h(s, trips, s->S.pgs_trips, sizeof(int) * s->S.N)) return -1;
  if (stream_floats && d2h(s, stream_floats, s->S.rs_nfloats, sizeof(int) * s->S.N)) return -1;
  return 0;
}

int ag_get_solver_stats(AgSim* s, int32_t* contacts, int32_t* iters) {
  DevGuard guard__(s->device);
  if (contacts && d2h(s, contacts, s->S.c_count, sizeof(int) * s->S.N)) return -1;
  if (iters && d2h(s, iters, s->S.iters_used, sizeof(int) * s->S.N)) return -1;
  return 0;
}

int ag_overflow_count(AgSim* s) {
  DevGuard guard__(s->device);
  std::vector<int> o(s->S.N);
  if (d2h(s, o.data(), s->S.overflow, sizeof(int) * s->S.N)) return -1;
  int n = 0; for (int v : o) n += v != 0;
  if (n && dev_zero(s, s->S.overflow, sizeof(int) * s->S.N)) return -1;     // the flags are sticky until read
  return n;
}

// ------------------------------------------------------------------ fused env steps: the driver the four tasks share
// Each task's init fills its FusedStep (fused_alloc) and its enqueue function launches the task's kernels; stepping,
// graph replay and the host-buffer staging are the same for every task.
//
// One env step is ~90 small launches (14 kernels + 3 memsets per substep); captured once per set of device
// pointers and replayed with a single cudaGraphLaunch.  Falls back to direct launches while profiling
// (per-kernel events), when AG_GRAPH=0, or if capture fails.
static int run_step(AgSim* s, FusedStep& R, const float* action, float* obs, float* reward, float* done, float* info) {
#ifndef AG_CPU_EMU
  if (s->use_graph && !s->profiling) {
    // The graph is captured against the task's OWN action buffer: a learner hands in a freshly allocated action tensor
    // every step, and a graph keyed on that address would be re-captured (~90 launches + instantiate) each time.
    if (action != R.d_action) { CK(cudaMemcpyAsync(R.d_action, action, sizeof(float) * 7 * s->S.N, cudaMemcpyDeviceToDevice, s->stream)); action = R.d_action; }
    StepGraph& G = R.graph;
    const void* key[5] = {action, obs, reward, done, info};
    if (G.valid && memcmp(G.key, key, sizeof(key)) != 0) drop_graph(G);
    if (!G.valid) {
      uint64_t l0 = s->launches;
      cudaGraph_t graph = nullptr; cudaGraphExec_t exec = nullptr;
      if (cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        int rc = R.enqueue(s, action, obs, reward, done, info);
        cudaError_t ce = cudaStreamEndCapture(s->stream, &graph);
        if (rc == 0 && ce == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
          G.exec = exec; memcpy(G.key, key, sizeof(key)); G.launches = s->launches - l0; G.valid = true; s->graph_failures = 0;
        }
        if (graph) cudaGraphDestroy(graph);
      }
      s->launches = l0;
      if (!G.valid) { cudaGetLastError(); if (++s->graph_failures >= 3) s->use_graph = false; }   // a transient failure: try again next step
    }
    if (G.valid) {
      CK(cudaGraphLaunch((cudaGraphExec_t)G.exec, s->stream));
      s->launches += G.launches;
      return 0;
    }
  }
#endif
  return R.enqueue(s, action, obs, reward, done, info);
}
// Allocates task t's step I/O on its first init; a later init (an episode reset) keeps the buffers.
static int fused_alloc(AgSim* s, FusedTask t, int obs_dim, StepEnqueue enqueue) {
  FusedStep& R = s->fused[t];
  R.obs_dim = obs_dim; R.enqueue = enqueue;
  if (R.h_out) return 0;
  const size_t N = s->S.N;
  R.d_action = dalloc<float>(s, N * 7); R.d_obs = dalloc<float>(s, N * obs_dim);
  R.d_reward = dalloc<float>(s, N); R.d_done = dalloc<float>(s, N); R.d_info = dalloc<float>(s, N * 4);
  if (!R.d_action || !R.d_obs || !R.d_reward || !R.d_done || !R.d_info) return fail("device allocation failed");
  if (!R.h_in && pinned_alloc(&R.h_in, N * 7)) return -1;
  return pinned_alloc(&R.h_out, N * (obs_dim + 6));
}
static int need_init(AgSim* s, FusedTask t) {
  return s->fused[t].ready ? 0 : fail(std::string("ag_") + fused_name[t] + "_init not called");
}
// device-buffer step: enqueued on the sim's stream, returns without waiting for it
static int fused_step_dev(AgSim* s, FusedTask t, const float* action, float* obs, float* reward, float* done, float* info) {
  if (need_init(s, t)) return -1;
  if (s->cloth && s->cloth_sub != 0)
    return fail(std::string("ag_") + fused_name[t] + "_step: a stepSimulation is half done (ag_step with a partial substep count?)");
  int rc = run_step(s, s->fused[t], action, obs, reward, done, info);
#ifndef AG_CPU_EMU
  CK(cudaGetLastError());
#endif
  return rc;
}
// host-buffer step in two halves: `begin` stages the actions (pinned) and enqueues H2D, the fused step and the D2H
// read-back on the sim's stream and returns; `end` waits for that stream and hands the results out (`info` may be NULL).
// Several sims (sub-batches of one batch, each on its own stream) overlap this way.
static int fused_step_host_begin(AgSim* s, FusedTask t, const float* action) {
  if (need_init(s, t)) return -1;
  FusedStep& R = s->fused[t];
  const size_t N = s->S.N, D = R.obs_dim;
  float* o = R.h_out;
  memcpy(R.h_in, action, sizeof(float) * N * 7);
  if (copy_async(s, R.d_action, R.h_in, sizeof(float) * N * 7, cudaMemcpyHostToDevice)) return -1;
  if (fused_step_dev(s, t, R.d_action, R.d_obs, R.d_reward, R.d_done, R.d_info)) return -1;
  if (copy_async(s, o, R.d_obs, sizeof(float) * N * D, cudaMemcpyDeviceToHost) ||
      copy_async(s, o + N * D, R.d_reward, sizeof(float) * N, cudaMemcpyDeviceToHost) ||
      copy_async(s, o + N * (D + 1), R.d_done, sizeof(float) * N, cudaMemcpyDeviceToHost) ||
      copy_async(s, o + N * (D + 2), R.d_info, sizeof(float) * N * 4, cudaMemcpyDeviceToHost)) return -1;
  return 0;
}
static int fused_step_host_end(AgSim* s, FusedTask t, float* obs, float* reward, float* done, float* info) {
  if (need_init(s, t)) return -1;
  const FusedStep& R = s->fused[t];
  const size_t N = s->S.N, D = R.obs_dim;
#ifndef AG_CPU_EMU
  CK(cudaStreamSynchronize(s->stream));
  CK(cudaGetLastError());
#endif
  memcpy(obs, R.h_out, sizeof(float) * N * D);
  memcpy(reward, R.h_out + N * D, sizeof(float) * N);
  memcpy(done, R.h_out + N * (D + 1), sizeof(float) * N);
  if (info) memcpy(info, R.h_out + N * (D + 2), sizeof(float) * N * 4);
  return 0;
}
static int fused_step_host(AgSim* s, FusedTask t, const float* action, float* obs, float* reward, float* done, float* info) {
  if (fused_step_host_begin(s, t, action)) return -1;
  return fused_step_host_end(s, t, obs, reward, done, info);
}
// tremor of `nj` joints of the person: per env on/off, rest angles and amplitudes [N][nj] -> the task's [N], [nj][N], [nj][N]
// device arrays.  NULL `on` switches tremor off.
static int set_tremor(AgSim* s, FusedTask t, int nj, int* d_on, float* d_rest, float* d_amp, const int32_t* on, const float* rest, const float* amplitude) {
  if (need_init(s, t)) return -1;
  const int N = s->S.N;
  std::vector<int> o(N, 0); std::vector<float> r((size_t)nj * N, 0.f), a((size_t)nj * N, 0.f);
  if (on) for (int e = 0; e < N; e++) {
    o[e] = on[e];
    for (int j = 0; j < nj; j++) { r[(size_t)j * N + e] = rest ? rest[(size_t)e * nj + j] : 0.f; a[(size_t)j * N + e] = amplitude ? amplitude[(size_t)e * nj + j] : 0.f; }
  }
  if (h2d(s, d_on, o.data(), sizeof(int) * N) || h2d(s, d_rest, r.data(), sizeof(float) * nj * N)) return -1;
  return h2d(s, d_amp, a.data(), sizeof(float) * nj * N);
}

// ------------------------------------------------------------------ cloth (K8, ag_cloth.cuh)
static size_t cloth_smem_bytes(const AgSim* s) {
  size_t f = (size_t)4 * s->cloth_npt * AG_CLOTH_T + AG_CLOTH_LKS * AG_CLOTH_MAXCL + 12 * (size_t)s->C.maxcc + 40 + 192;
  if (s->cloth_qs) f += (size_t)4 * s->cloth_npt * AG_CLOTH_T;
  return f * sizeof(float);
}
static void cloth_launch(AgSim* s) {
#ifndef AG_CPU_EMU
  size_t smem = cloth_smem_bytes(s);
  int ps = s->profiling ? prof_slot(s, "k_cloth") : -1;
  if (ps >= 0) prof_mark(s, ps, true);
  if (s->cloth_npt == 4) { if (s->cloth_qs) k_cloth<4, true><<<s->S.N, AG_CLOTH_T, smem, s->stream>>>(s->S, s->C); else k_cloth<4, false><<<s->S.N, AG_CLOTH_T, smem, s->stream>>>(s->S, s->C); }
  else { if (s->cloth_qs) k_cloth<8, true><<<s->S.N, AG_CLOTH_T, smem, s->stream>>>(s->S, s->C); else k_cloth<8, false><<<s->S.N, AG_CLOTH_T, smem, s->stream>>>(s->S, s->C); }
  if (ps >= 0) prof_mark(s, ps, false);
#else
  for (int e = 0; e < s->S.N; e++) cloth_env_host(s->S, s->C, e);
#endif
  s->launches++;
}

int ag_cloth_init(AgSim* s, const AgClothDesc* d) {
  DevGuard guard__(s->device);
  if (s->cloth) return fail("ag_cloth_init: the sim already has a cloth");
  if (!d || d->n_nodes <= 0 || d->n_nodes > 65535) return fail("ag_cloth_init: 1..65535 nodes");
  if (d->n_nodes > 8 * AG_CLOTH_T) return fail("ag_cloth_init: more than 8192 nodes");
  if (d->n_colours < 1 || d->n_colours > AG_CLOTH_MAXCOL) return fail("ag_cloth_init: 1..16 link colours");
  if (d->n_anchors < 0 || d->n_anchors > AG_CLOTH_MAXANCH) return fail("ag_cloth_init: at most 8 anchors");
  if (d->n_col_links < 0 || d->n_col_links > AG_CLOTH_MAXCL) return fail("ag_cloth_init: at most 96 collider links");
  const int N = s->S.N, nn = d->n_nodes;
  ClothDev& C = s->C;
  memset(&C, 0, sizeof(C));
  C.nn = nn; C.nlinks = d->n_links; C.ncol = d->n_colours; C.nanch = d->n_anchors; C.ncl = d->n_col_links;
  s->cloth_npt = nn <= 4 * AG_CLOTH_T ? 4 : 8;
  C.nnp = (nn + 31) / 32 * 32;
  C.maxcc = d->max_contacts > 0 ? d->max_contacts : 1024;
  C.K = s->cfg.num_substeps > 0 ? s->cfg.num_substeps : 1;
  C.piters = d->piterations; C.export_contacts = 1;
  C.dt = s->S.dt; C.im = (float)d->inv_mass; C.kLSTh = (float)(0.5 * d->kLST); C.kDP = (float)d->kDP; C.kDG = (float)d->kDG; C.kLF = (float)d->kLF;
  C.kDF = (float)d->kDF; C.kCHR = (float)d->kCHR; C.kKHR = (float)d->kKHR; C.kAHR = (float)d->kAHR; C.margin = (float)d->margin; C.density = (float)d->air_density;
  C.gx = (float)d->gravity[0]; C.gy = (float)d->gravity[1]; C.gz = (float)d->gravity[2];
  for (int c = 0; c <= d->n_colours; c++) C.col_off[c] = d->colour_off[c];
  if (C.col_off[0] != 0 || C.col_off[d->n_colours] != d->n_links) return fail("ag_cloth_init: colour offsets do not cover the link list");
  std::vector<unsigned> lij(d->n_links); std::vector<float> lr(d->n_links);
  {
    std::vector<int> seen(nn, -1);                     // links of one colour must not share a node (the kernel relaxes them concurrently)
    for (int c = 0; c < d->n_colours; c++)
      for (int l = C.col_off[c]; l < C.col_off[c + 1]; l++) {
        int a = d->links[2 * l], b = d->links[2 * l + 1];
        if (a < 0 || b < 0 || a >= nn || b >= nn || a == b) return fail("ag_cloth_init: bad link");
        if (seen[a] == c || seen[b] == c) return fail("ag_cloth_init: two links of one colour share a node");
        seen[a] = seen[b] = c;
        lij[l] = (unsigned)a | ((unsigned)b << 16); lr[l] = (float)d->link_rest2[l];
      }
  }
  std::vector<unsigned> nfp(d->n_nf);
  for (int f = 0; f < d->n_nf; f++) nfp[f] = (unsigned)d->nf_pair[2 * f] | ((unsigned)d->nf_pair[2 * f + 1] << 16);
  std::vector<float> area(nn), bs((size_t)4 * d->n_col_links);
  for (int i = 0; i < nn; i++) area[i] = (float)d->node_area[i];
  for (size_t i = 0; i < bs.size(); i++) bs[i] = (float)d->col_link_bsphere[i];
  for (int a = 0; a < d->n_anchors; a++) {
    if (d->anchor_node[a] < 0 || d->anchor_node[a] >= nn) return fail("ag_cloth_init: bad anchor node");
    C.anch_node[a] = d->anchor_node[a];
    for (int k = 0; k < 3; k++) C.anch_local[a][k] = (float)d->anchor_local[3 * a + k];
  }
  for (int L = 0; L < d->n_col_links; L++) if (d->col_links[L] < 0 || d->col_links[L] >= s->nl) return fail("ag_cloth_init: bad collider link");
  C.link_ij = upload(s, lij); C.link_rest2 = upload(s, lr);
  {
    std::vector<ClothLinkRec> tab;                    // every colour starts at a multiple of 32 entries
    for (int c = 0; c < d->n_colours; c++) {
      tab.resize((tab.size() + 31) / 32 * 32, ClothLinkRec{0u, 0.f});
      C.tab_off[c] = (int)tab.size();
      for (int l = C.col_off[c]; l < C.col_off[c + 1]; l++) tab.push_back(ClothLinkRec{lij[l], lr[l]});
      C.tab_end[c] = (int)tab.size();
    }
    C.link_tab = upload(s, tab);
    bool fits = true;
    for (int c = 0; c < d->n_colours; c++) fits &= C.col_off[c + 1] - C.col_off[c] <= AG_CLOTH_T;
    C.link_dense = nullptr;
    if (fits) {                                       // one row of AG_CLOTH_T entries per colour (+ one spare row: the fetch runs a pass ahead)
      std::vector<ClothLinkRec> dense((size_t)(d->n_colours + 1) * AG_CLOTH_T, ClothLinkRec{0xffffffffu, 0.f});
      for (int c = 0; c < d->n_colours; c++)
        for (int l = C.col_off[c]; l < C.col_off[c + 1]; l++) dense[(size_t)c * AG_CLOTH_T + (l - C.col_off[c])] = ClothLinkRec{lij[l], lr[l]};
      C.link_dense = upload(s, dense);
    }
  }
  C.nf_off = upload(s, std::vector<int>(d->nf_off, d->nf_off + nn + 1)); C.nf_pair = upload(s, nfp);
  C.node_area = upload(s, area);
  C.cl_link = upload(s, std::vector<int>(d->col_links, d->col_links + d->n_col_links)); C.cl_bs = upload(s, bs);
  C.cl_static = upload(s, std::vector<int>(d->col_link_static, d->col_link_static + d->n_col_links));
  C.x = dalloc<float>(s, (size_t)N * 3 * C.nnp); C.v = dalloc<float>(s, (size_t)N * 3 * C.nnp);
  C.anchor_pos = dalloc<float>(s, (size_t)3 * N);
  C.snap = dalloc<float>(s, (size_t)C.K * std::max(C.ncl, 1) * 7 * N);
  C.cc_count = dalloc<int>(s, N); C.cc_data = dalloc<float>(s, (size_t)N * C.maxcc * AG_CLOTH_CCF); C.overflow = s->S.overflow;   // the same sticky per-env flags as the rigid budgets (ag_overflow_count)
  s->C_dev = dalloc<ClothDev>(s, 1);
  if (!C.cc_data || !C.overflow || !s->C_dev || !C.snap || !C.v) return fail("ag_cloth_init: device allocation failed");
  if (h2d(s, s->C_dev, &C, sizeof(ClothDev))) return -1;
  { const char* qs = getenv("AG_CLOTH_QS"); s->cloth_qs = qs ? atoi(qs) != 0 : 1; }
  if (s->cloth_qs && cloth_smem_bytes(s) > 227 * 1024) s->cloth_qs = 0;          // the second node array does not fit next to a big contact pool: q / v in registers
#ifndef AG_CPU_EMU
  size_t smem = cloth_smem_bytes(s);
  if (smem > 227 * 1024) return fail("ag_cloth_init: cloth + contact budget exceed 227 KB of shared memory");
  if (s->cloth_npt == 4) { CK(cudaFuncSetAttribute(k_cloth<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); CK(cudaFuncSetAttribute(k_cloth<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); }
  else { CK(cudaFuncSetAttribute(k_cloth<8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); CK(cudaFuncSetAttribute(k_cloth<8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)); }
#endif
  drop_graphs(s);                                     // a captured step has no cloth launch
  s->cloth = true; s->cloth_sub = 0;
  return 0;
}
static int cloth_refresh(AgSim* s) { return h2d(s, s->C_dev, &s->C, sizeof(ClothDev)); }

int ag_cloth_set_state(AgSim* s, const float* x, const float* v, const int32_t* mask) {
  DevGuard guard__(s->device);
  if (!s->cloth) return fail("ag_cloth_init not called");
  const int N = s->S.N, nn = s->C.nn, nnp = s->C.nnp;
  std::vector<float> buf((size_t)N * 3 * nnp);
  for (int which = 0; which < 2; which++) {
    const float* src = which ? v : x; float* dst = which ? s->C.v : s->C.x;
    if (!src) continue;
    if (mask && d2h(s, buf.data(), dst, buf.size() * sizeof(float))) return -1;
    if (!mask) std::fill(buf.begin(), buf.end(), 0.f);
    for (int e = 0; e < N; e++) if (!mask || mask[e])
      for (int i = 0; i < nn; i++) for (int c = 0; c < 3; c++) buf[((size_t)e * 3 + c) * nnp + i] = src[((size_t)e * nn + i) * 3 + c];
    if (h2d(s, dst, buf.data(), buf.size() * sizeof(float))) return -1;
  }
  return 0;
}
int ag_cloth_get_state(AgSim* s, float* x, float* v) {
  DevGuard guard__(s->device);
  if (!s->cloth) return fail("ag_cloth_init not called");
  const int N = s->S.N, nn = s->C.nn, nnp = s->C.nnp;
  std::vector<float> buf((size_t)N * 3 * nnp);
  for (int which = 0; which < 2; which++) {
    float* dst = which ? v : x; const float* src = which ? s->C.v : s->C.x;
    if (!dst) continue;
    if (d2h(s, buf.data(), src, buf.size() * sizeof(float))) return -1;
    for (int e = 0; e < N; e++) for (int i = 0; i < nn; i++) for (int c = 0; c < 3; c++) dst[((size_t)e * nn + i) * 3 + c] = buf[((size_t)e * 3 + c) * nnp + i];
  }
  return 0;
}
int ag_cloth_set_anchor(AgSim* s, const float* pos, const int32_t* mask) {
  DevGuard guard__(s->device);
  if (!s->cloth) return fail("ag_cloth_init not called");
  const int N = s->S.N;
  std::vector<float> buf((size_t)3 * N);
  if (d2h(s, buf.data(), s->C.anchor_pos, buf.size() * sizeof(float))) return -1;
  for (int e = 0; e < N; e++) if (!mask || mask[e]) for (int c = 0; c < 3; c++) buf[(size_t)c * N + e] = pos[(size_t)e * 3 + c];
  return h2d(s, s->C.anchor_pos, buf.data(), buf.size() * sizeof(float));
}
int ag_cloth_anchor_follow(AgSim* s, int link) {
  DevGuard guard__(s->device);
  if (!s->cloth) return fail("ag_cloth_init not called");
  if (link < 0 || link >= s->nl) return fail("bad link");
  KP p = kp0(); p.p0 = s->C_dev; p.i0 = link;
  LAUNCH(s, k_cloth_follow, s->S.N, p);
  return 0;
}
int ag_cloth_set_gravity(AgSim* s, const double g[3]) {
  DevGuard guard__(s->device);
  if (!s->cloth) return fail("ag_cloth_init not called");
  s->C.gx = (float)g[0]; s->C.gy = (float)g[1]; s->C.gz = (float)g[2];
  drop_graphs(s);                                       // k_cloth takes ClothDev by value: a captured step holds the old gravity
  return cloth_refresh(s);
}
int ag_cloth_get_contacts(AgSim* s, int max_pts, int32_t* count, int32_t* node, float* pos, float* force, int32_t* link) {
  DevGuard guard__(s->device);
  if (!s->cloth) return fail("ag_cloth_init not called");
  if (max_pts < 0) return fail("max_pts < 0");
  const int N = s->S.N, M = s->C.maxcc;
  std::vector<int> cnt(N); std::vector<float> data((size_t)N * M * AG_CLOTH_CCF);
  if (d2h(s, cnt.data(), s->C.cc_count, sizeof(int) * N) || d2h(s, data.data(), s->C.cc_data, data.size() * sizeof(float))) return -1;
  for (int e = 0; e < N; e++) {
    if (count) count[e] = cnt[e];
    for (int k = 0; k < std::min(cnt[e], max_pts); k++) {
      const float* r = &data[((size_t)e * M + k) * AG_CLOTH_CCF];
      size_t o = (size_t)e * max_pts + k;
      int32_t id; memcpy(&id, r, 4); if (node) node[o] = id;
      memcpy(&id, r + 7, 4); if (link) link[o] = id;
      for (int c = 0; c < 3; c++) { if (pos) pos[3 * o + c] = r[1 + c]; if (force) force[3 * o + c] = r[4 + c]; }
    }
  }
  return 0;
}
int ag_cloth_device_state(AgSim* s, float** x_dev, float** v_dev, int32_t* nnp) {
  if (!s->cloth) return fail("ag_cloth_init not called");
  if (x_dev) *x_dev = s->C.x;
  if (v_dev) *v_dev = s->C.v;
  if (nnp) *nnp = s->C.nnp;
  return 0;
}

// ------------------------------------------------------------------ fused DressingEnv path
int ag_dressing_reset_episode(AgSim* s, const int32_t* env_mask) {
  DevGuard guard__(s->device);
  if (need_init(s, FT_DRESSING)) return -1;
  const int N = s->S.N;
  std::vector<int> it(N); std::vector<float> ts(N);
  if (d2h(s, it.data(), s->DP.D.iteration, sizeof(int) * N) || d2h(s, ts.data(), s->DP.D.task_success, sizeof(float) * N)) return -1;
  for (int e = 0; e < N; e++) if (!env_mask || env_mask[e]) { it[e] = 0; ts[e] = 0.f; }
  if (h2d(s, s->DP.D.iteration, it.data(), sizeof(int) * N) || h2d(s, s->DP.D.task_success, ts.data(), sizeof(float) * N)) return -1;
  return 0;
}
static int dressing_step_enqueue(AgSim* s, const float* action_dev, float* obs, float* reward, float* done, float* info) {
  const int N = s->S.N;
  KP p = kp0(); p.p0 = action_dev; p.p1 = s->DP_dev;
  LAUNCH(s, k_dress_pre, N, p);
  const int sub = s->cfg.num_substeps > 0 ? s->cfg.num_substeps : 1;
  KP z = kp0();
  for (int f = 0; f < s->DP.D.P.frame_skip; f++) {
    for (int i = 0; i < sub; i++) substep(s);                        // the last one launches k_cloth
    LAUNCH(s, k_fk, (size_t)s->S.nb * N, z);
    KP c = kp0(); c.p0 = s->C_dev; c.i0 = s->DP.D.P.ee_link;         // update_targets (dressing.py:210)
    LAUNCH(s, k_cloth_follow, N, c);
  }
  KP q = kp0(); q.p0 = action_dev; q.p1 = s->DP_dev; q.p2 = obs; q.p3 = reward; q.p4 = done; q.p5 = info;
  LAUNCH(s, k_dress_post, N, q);
  return 0;
}
int ag_dressing_init(AgSim* s, const AgDressingParams* p, const int32_t* gender_is_male) {
  DevGuard guard__(s->device);
  if (!s->cloth) return fail("ag_dressing_init: ag_cloth_init first");
  const int N = s->S.N;
  for (int j = 0; j < 7; j++) if (p->arm_links[j] < 0 || p->arm_links[j] >= s->nl) return fail("ag_dressing_init: bad arm link");
  for (int j = 0; j < 3; j++) if (p->tri1[j] < 0 || p->tri1[j] >= s->C.nn || p->tri2[j] < 0 || p->tri2[j] >= s->C.nn) return fail("ag_dressing_init: bad sleeve node");
  if (p->ee_link < 0 || p->ee_link >= s->nl) return fail("ag_dressing_init: bad end effector link");
  DressDev& D = s->DP.D;
  D.P = *p;
  drop_graph(s->fused[FT_DRESSING].graph);
  if (!s->fused[FT_DRESSING].ready) {
    D.male = dalloc<int>(s, N); D.iteration = dalloc<int>(s, N); D.task_success = dalloc<float>(s, N); D.action = dalloc<float>(s, (size_t)N * 7);
    D.tremor_on = dalloc<int>(s, N); D.tremor_rest = dalloc<float>(s, (size_t)N * 10); D.tremor_amp = dalloc<float>(s, (size_t)N * 10);
    s->DP_dev = dalloc<DressPost>(s, 1);
    if (!s->DP_dev) return fail("device allocation failed");
  }
  else if (dev_zero(s, D.tremor_on, sizeof(int) * N)) return -1;
  if (fused_alloc(s, FT_DRESSING, 24, dressing_step_enqueue)) return -1;
  for (int j = 0; j < 10; j++) if (p->human_arm_m[j] < 0 || p->human_arm_m[j] >= s->nl || p->human_arm_f[j] < 0 || p->human_arm_f[j] >= s->nl) return fail("ag_dressing_init: bad human arm link");
  s->DP.C = s->C_dev;
  if (h2d(s, D.male, gender_is_male, sizeof(int) * N)) return -1;
  if (h2d(s, s->DP_dev, &s->DP, sizeof(DressPost))) return -1;
  s->fused[FT_DRESSING].ready = true;
  return ag_dressing_reset_episode(s, nullptr);
}
int ag_dressing_set_tremor(AgSim* s, const int32_t* on, const float* rest, const float* amplitude) {
  DevGuard guard__(s->device);
  return set_tremor(s, FT_DRESSING, 10, s->DP.D.tremor_on, s->DP.D.tremor_rest, s->DP.D.tremor_amp, on, rest, amplitude);
}
int ag_dressing_step_dev(AgSim* s, const float* action_dev, float* obs_dev, float* reward_dev, float* done_dev, float* info_dev) {
  DevGuard guard__(s->device); return fused_step_dev(s, FT_DRESSING, action_dev, obs_dev, reward_dev, done_dev, info_dev); }
int ag_dressing_step_host(AgSim* s, const float* action, float* obs, float* reward, float* done, float* info) {
  DevGuard guard__(s->device); return fused_step_host(s, FT_DRESSING, action, obs, reward, done, info); }

// ------------------------------------------------------------------ camera images (K9, ag_render.cuh)
int ag_render(AgSim* s, const AgCamera* cam, int n, const int32_t* env_ids, uint8_t* rgba, float* depth) {
  DevGuard guard__(s->device);
  if (!cam || n <= 0 || !env_ids || !rgba) return fail("ag_render: bad arguments");
  if (cam->width <= 0 || cam->height <= 0 || cam->width * (long long)cam->height * n > (1ll << 30)) return fail("ag_render: bad image size");
  for (int i = 0; i < n; i++) if (env_ids[i] < 0 || env_ids[i] >= s->S.N) return fail("ag_render: bad env id");
  // link poses and link AABBs of the current state (all bodies)
  run_fk_all(s);
  RenderDev R = RenderDev();
  R.cam = *cam;
  f3 eye(cam->eye[0], cam->eye[1], cam->eye[2]), tgt(cam->target[0], cam->target[1], cam->target[2]), upv(cam->up[0], cam->up[1], cam->up[2]);
  f3 f = tgt - eye; float fl = norm(f); if (!(fl > 0.f)) return fail("ag_render: eye == target");
  f = f * (1.f / fl);
  f3 r = cross(f, upv); float rl = norm(r); if (!(rl > 0.f)) return fail("ag_render: up is parallel to the view direction");
  r = r * (1.f / rl);
  R.fwd = f; R.right = r; R.up = cross(r, f);
  R.tan_half = tanf(0.5f * cam->fov_deg * 3.14159265358979323846f / 180.f);
  const size_t npix = (size_t)cam->width * cam->height * n;
  if (npix > s->render_pix || n > s->render_n) {            // grow-only scratch (an episode renders a frame per step)
    s->render_pix = std::max(npix, s->render_pix); s->render_n = std::max(n, s->render_n);
    s->d_render_ids = dalloc<int>(s, s->render_n); s->d_render_rgba = (unsigned char*)dev_alloc(s, s->render_pix * 4);
    s->d_render_depth = dalloc<float>(s, s->render_pix);
    if (!s->d_render_dev) s->d_render_dev = dev_alloc(s, sizeof(RenderDev));
  }
  int* d_ids = s->d_render_ids; unsigned char* d_rgba = s->d_render_rgba; float* d_depth = s->d_render_depth;
  RenderDev* d_R = (RenderDev*)s->d_render_dev;
  if (!d_ids || !d_rgba || !d_depth || !d_R) return fail("device allocation failed");
  R.env_ids = d_ids; R.rgba = d_rgba; R.depth = d_depth;
  if (h2d(s, d_ids, env_ids, sizeof(int) * n) || h2d(s, d_R, &R, sizeof(RenderDev))) return -1;
  KP p = kp0(); p.p0 = d_R;
  LAUNCH(s, k_render, npix, p);
  if (d2h(s, rgba, d_rgba, npix * 4)) return -1;
  if (depth && d2h(s, depth, d_depth, npix * sizeof(float))) return -1;
  return 0;
}

// ------------------------------------------------------------------ fused ScratchItchEnv path
static int scratch_step_enqueue(AgSim* s, const float* action_dev, float* obs, float* reward, float* done, float* info) {
  const int N = s->S.N;
  KP p = kp0(); p.p0 = action_dev; p.p1 = s->SD_dev;
  LAUNCH(s, k_scratch_pre, N, p);
  for (int i = 0; i < s->SD.P.frame_skip * (s->cfg.num_substeps > 0 ? s->cfg.num_substeps : 1); i++) substep(s);
  KP z = kp0();
  LAUNCH(s, k_fk, (size_t)s->S.nb * N, z);
  KP q = kp0(); q.p0 = action_dev; q.p1 = s->SD_dev; q.p2 = obs; q.p3 = reward; q.p4 = done; q.p5 = info;
  LAUNCH(s, k_scratch_post, N, q);
  return 0;
}
int ag_scratch_init(AgSim* s, const AgScratchParams* p, const int32_t* gender_is_male, const int32_t* limb_link, const float* target_local) {
  DevGuard guard__(s->device);
  const int N = s->S.N;
  for (int j = 0; j < 7; j++) if (p->arm_links[j] < 0 || p->arm_links[j] >= s->nl) return fail("ag_scratch_init: bad arm link");
  if (p->ee_link < 0 || p->ee_link >= s->nl || p->tool_tip_link < 0 || p->tool_tip_link >= s->nl || p->tool_link0 < 0 || p->tool_link0 >= s->nl) return fail("ag_scratch_init: bad link");
  for (int e = 0; e < N; e++) if (limb_link[e] < 0 || limb_link[e] >= s->nl) return fail("ag_scratch_init: bad limb link");
  ScratchDev& D = s->SD;
  D.P = *p;
  drop_graph(s->fused[FT_SCRATCH].graph);
  if (!s->fused[FT_SCRATCH].ready) {
    D.male = dalloc<int>(s, N); D.iteration = dalloc<int>(s, N); D.task_success = dalloc<int>(s, N); D.limb_link = dalloc<int>(s, N);
    D.target_local = dalloc<float>(s, (size_t)3 * N); D.prev_contact = dalloc<float>(s, (size_t)3 * N); D.action = dalloc<float>(s, (size_t)7 * N);
    s->SD_dev = dalloc<ScratchDev>(s, 1);
    if (!s->SD_dev) return fail("device allocation failed");
  }
  if (fused_alloc(s, FT_SCRATCH, 30, scratch_step_enqueue)) return -1;
  std::vector<float> tl((size_t)3 * N);
  for (int e = 0; e < N; e++) for (int c = 0; c < 3; c++) tl[(size_t)c * N + e] = target_local[(size_t)e * 3 + c];
  if (h2d(s, D.male, gender_is_male, sizeof(int) * N) || h2d(s, D.limb_link, limb_link, sizeof(int) * N) || h2d(s, D.target_local, tl.data(), sizeof(float) * 3 * N)) return -1;
  if (dev_zero(s, D.iteration, sizeof(int) * N) || dev_zero(s, D.task_success, sizeof(int) * N) || dev_zero(s, D.prev_contact, sizeof(float) * 3 * N)) return -1;   // scratch_itch.py:97
  if (h2d(s, s->SD_dev, &s->SD, sizeof(ScratchDev))) return -1;
  s->fused[FT_SCRATCH].ready = true;
  return 0;
}
int ag_scratch_step_dev(AgSim* s, const float* action_dev, float* obs_dev, float* reward_dev, float* done_dev, float* info_dev) {
  DevGuard guard__(s->device); return fused_step_dev(s, FT_SCRATCH, action_dev, obs_dev, reward_dev, done_dev, info_dev); }
int ag_scratch_step_host(AgSim* s, const float* action, float* obs, float* reward, float* done, float* info) {
  DevGuard guard__(s->device); return fused_step_host(s, FT_SCRATCH, action, obs, reward, done, info); }

// ------------------------------------------------------------------ fused FeedingEnv path
static int feeding_step_enqueue(AgSim* s, const float* action_dev, float* obs, float* reward, float* done, float* info) {
  const int N = s->S.N;
  KP p = kp0(); p.p0 = action_dev; p.p1 = s->F_dev;
  LAUNCH(s, k_feed_pre, N, p);
  for (int i = 0; i < s->F.P.frame_skip * (s->cfg.num_substeps > 0 ? s->cfg.num_substeps : 1); i++) substep(s);
  KP z = kp0();
  LAUNCH(s, k_fk, (size_t)s->S.nb * N, z);
  KP a = kp0(); a.p0 = s->S.movcol; a.i0 = s->S.nmovcol;
  LAUNCH(s, k_aabb, (size_t)s->S.nmovcol * N, a);
  KP l = kp0(); l.p0 = s->S.movlink; l.i0 = s->S.nmovlink;
  LAUNCH(s, k_linkaabb, (size_t)s->S.nmovlink * N, l);
  KP f = kp0(); f.p1 = s->F_dev;
  LAUNCH(s, k_feed_food, (size_t)N * s->F.P.n_foods, f);
  KP q = kp0(); q.p0 = action_dev; q.p1 = s->F_dev; q.p2 = obs; q.p3 = reward; q.p4 = done; q.p5 = info;
  LAUNCH(s, k_feed_post, N, q);
  return 0;
}
int ag_feeding_init(AgSim* s, const AgFeedingParams* p, const int32_t* gender_is_male) {
  DevGuard guard__(s->device);
  const int N = s->S.N;
  FeedDev& F = s->F;
  F.P = *p;
  if (p->n_foods > 16) return fail("too many foods");
  drop_graph(s->fused[FT_FEEDING].graph);          // the captured step refers to the previous FeedDev
  if (!s->fused[FT_FEEDING].ready) {              // buffers are allocated once; a later init (episode reset) only refreshes their contents
    F.male = dalloc<int>(s, N); F.food_state = dalloc<int>(s, N); F.iteration = dalloc<int>(s, N); F.task_success = dalloc<int>(s, N);
    F.food_near = dalloc<int>(s, (size_t)N * 16);
    F.action = dalloc<float>(s, (size_t)N * 7); F.rng = dalloc<unsigned long long>(s, N);
    F.tremor_on = dalloc<int>(s, N); F.tremor_rest = dalloc<float>(s, (size_t)N * 4); F.tremor_amp = dalloc<float>(s, (size_t)N * 4);
    s->F_dev = dalloc<FeedDev>(s, 1);
    if (!s->F_dev) return fail("device allocation failed");
  } else {
    if (dev_zero(s, F.tremor_on, sizeof(int) * N) || dev_zero(s, F.rng, sizeof(unsigned long long) * N)) return -1;
  }
  if (fused_alloc(s, FT_FEEDING, 25, feeding_step_enqueue)) return -1;
  if (h2d(s, F.male, gender_is_male, sizeof(int) * N)) return -1;
  if (!s->F_dev || h2d(s, s->F_dev, &s->F, sizeof(FeedDev))) return fail("FeedDev upload failed");
  s->fused[FT_FEEDING].ready = true;
  return ag_feeding_reset_episode(s, nullptr);
}
int ag_feeding_set_tremor(AgSim* s, const int32_t* on, const float* rest, const float* amplitude) {
  DevGuard guard__(s->device);
  return set_tremor(s, FT_FEEDING, 4, s->F.tremor_on, s->F.tremor_rest, s->F.tremor_amp, on, rest, amplitude);
}

int ag_feeding_reset_episode(AgSim* s, const int32_t* env_mask) {
  DevGuard guard__(s->device);
  if (need_init(s, FT_FEEDING)) return -1;
  const int N = s->S.N;
  std::vector<int> fs(N), it(N), ts(N); std::vector<unsigned long long> rng(N);
  if (d2h(s, fs.data(), s->F.food_state, sizeof(int) * N) || d2h(s, it.data(), s->F.iteration, sizeof(int) * N) ||
      d2h(s, ts.data(), s->F.task_success, sizeof(int) * N) || d2h(s, rng.data(), s->F.rng, sizeof(unsigned long long) * N)) return -1;
  int full = (1 << s->F.P.n_foods) - 1;
  for (int e = 0; e < N; e++) if (!env_mask || env_mask[e]) {
    fs[e] = full | (full << 16); it[e] = 0; ts[e] = 0;
    if (rng[e] == 0) rng[e] = (s->F.P.seed + 0x9E3779B97F4A7C15ull * (unsigned long long)(e + 1)) | 1ull;
  }
  if (h2d(s, s->F.food_state, fs.data(), sizeof(int) * N) || h2d(s, s->F.iteration, it.data(), sizeof(int) * N) ||
      h2d(s, s->F.task_success, ts.data(), sizeof(int) * N) || h2d(s, s->F.rng, rng.data(), sizeof(unsigned long long) * N)) return -1;
  return 0;
}

int ag_feeding_step_dev(AgSim* s, const float* action_dev, float* obs_dev, float* reward_dev, float* done_dev, float* info_dev) {
  DevGuard guard__(s->device); return fused_step_dev(s, FT_FEEDING, action_dev, obs_dev, reward_dev, done_dev, info_dev); }
int ag_feeding_step_host_begin(AgSim* s, const float* action) {
  DevGuard guard__(s->device); return fused_step_host_begin(s, FT_FEEDING, action); }
int ag_feeding_step_host_end(AgSim* s, float* obs, float* reward, float* done, float* info) {
  DevGuard guard__(s->device); return fused_step_host_end(s, FT_FEEDING, obs, reward, done, info); }
int ag_feeding_step_host(AgSim* s, const float* action, float* obs, float* reward, float* done, float* info) {
  DevGuard guard__(s->device); return fused_step_host(s, FT_FEEDING, action, obs, reward, done, info); }

// ------------------------------------------------------------------ fused BedBathingEnv path
static int bathing_step_enqueue(AgSim* s, const float* action_dev, float* obs, float* reward, float* done, float* info) {
  const int N = s->S.N;
  KP p = kp0(); p.p0 = action_dev; p.p1 = s->B_dev;
  LAUNCH(s, k_bath_pre, N, p);
  for (int i = 0; i < s->B.P.frame_skip * (s->cfg.num_substeps > 0 ? s->cfg.num_substeps : 1); i++) substep(s);
  KP z = kp0();
  LAUNCH(s, k_fk, (size_t)s->S.nb * N, z);
  KP a = kp0(); a.p0 = s->S.movcol; a.i0 = s->S.nmovcol;
  LAUNCH(s, k_aabb, (size_t)s->S.nmovcol * N, a);
  KP l = kp0(); l.p0 = s->S.movlink; l.i0 = s->S.nmovlink;
  LAUNCH(s, k_linkaabb, (size_t)s->S.nmovlink * N, l);
  KP d = kp0(); d.p1 = s->B_dev;
  LAUNCH(s, k_bath_dist, (size_t)N * s->B.n_slots, d);
  KP q = kp0(); q.p0 = action_dev; q.p1 = s->B_dev; q.p2 = obs; q.p3 = reward; q.p4 = done; q.p5 = info;
  LAUNCH(s, k_bath_post, N, q);
  return 0;
}
int ag_bathing_init(AgSim* s, const AgBathingParams* p, const int32_t* gender_is_male, const float* targets_world, const int32_t* targets_valid) {
  DevGuard guard__(s->device);
  const int N = s->S.N;
  BathDev& B = s->B;
  B.P = *p;
  drop_graph(s->fused[FT_BATHING].graph);
  const int T = p->n_targets_max;
  if (T <= 0 || T > 4096) return fail("bad target count");
  for (int j = 0; j < 7; j++) if (p->arm_links[j] < 0 || p->arm_links[j] >= s->nl) return fail("bad link");
  if (p->cloth_link < 0 || p->cloth_link >= s->nl || p->ee_link < 0 || p->ee_link >= s->nl) return fail("bad link");
  if (!s->fused[FT_BATHING].ready) {
    B.male = dalloc<int>(s, N); B.iteration = dalloc<int>(s, N); B.task_success = dalloc<int>(s, N); B.total_targets = dalloc<int>(s, N);
    B.action = dalloc<float>(s, (size_t)N * 7);
    B.targets = dalloc<float>(s, (size_t)T * 3 * N); B.alive = dalloc<int>(s, (size_t)T * N);
    B.n_slots = p->human_ncol_m > p->human_ncol_f ? p->human_ncol_m : p->human_ncol_f;
    B.dist_part = dalloc<float>(s, (size_t)(B.n_slots > 0 ? B.n_slots : 1) * N);
    s->B_dev = dalloc<BathDev>(s, 1);
    if (!s->B_dev || !B.dist_part) return fail("device allocation failed");
  } else if (T != s->B.P.n_targets_max) return fail("target count changed");
  if (fused_alloc(s, FT_BATHING, 24, bathing_step_enqueue)) return -1;
  std::vector<float> tw((size_t)T * 3 * N); std::vector<int> al((size_t)T * N), tot(N, 0), zero(N, 0);
  for (int e = 0; e < N; e++)
    for (int t = 0; t < T; t++) {
      int v = targets_valid[(size_t)e * T + t] != 0;
      al[(size_t)t * N + e] = v; tot[e] += v;
      for (int c = 0; c < 3; c++) tw[((size_t)t * 3 + c) * N + e] = targets_world[((size_t)e * T + t) * 3 + c];
    }
  if (h2d(s, B.targets, tw.data(), tw.size() * sizeof(float)) || h2d(s, B.alive, al.data(), al.size() * sizeof(int))) return -1;
  if (h2d(s, B.total_targets, tot.data(), sizeof(int) * N) || h2d(s, B.male, gender_is_male, sizeof(int) * N)) return -1;
  if (h2d(s, B.iteration, zero.data(), sizeof(int) * N) || h2d(s, B.task_success, zero.data(), sizeof(int) * N)) return -1;
  if (h2d(s, s->B_dev, &s->B, sizeof(BathDev))) return fail("BathDev upload failed");
  s->fused[FT_BATHING].ready = true;
  return 0;
}
int ag_bathing_step_dev(AgSim* s, const float* action_dev, float* obs_dev, float* reward_dev, float* done_dev, float* info_dev) {
  DevGuard guard__(s->device); return fused_step_dev(s, FT_BATHING, action_dev, obs_dev, reward_dev, done_dev, info_dev); }
int ag_bathing_step_host(AgSim* s, const float* action, float* obs, float* reward, float* done, float* info) {
  DevGuard guard__(s->device); return fused_step_host(s, FT_BATHING, action, obs, reward, done, info); }

}  // extern "C"

#ifdef AG_CPU_EMU
// harness-only: run the device GJK on two world-space vertex sets (tests/test_kernel_logic_cpu.py)
extern "C" int ag_debug_gjk(const float* A, int nA, const float* B, int nB, float* pa, float* pb, float* nrm, float* dist) {
  std::vector<float> v((size_t)3 * (nA + nB));
  memcpy(v.data(), A, sizeof(float) * 3 * nA); memcpy(v.data() + 3 * nA, B, sizeof(float) * 3 * nB);
  std::vector<float> vqs((size_t)12 * ((nA + 3) / 4 + (nB + 3) / 4) + 4);
  float* vq = (float*)(((uintptr_t)vqs.data() + 15) & ~(uintptr_t)15);
  int gB = (nA + 3) / 4;
  for (int side = 0; side < 2; side++) {
    const float* src = side ? B : A; int nv = side ? nB : nA; float* dstq = vq + (side ? 12 * gB : 0);
    for (int g = 0; g < (nv + 3) / 4; g++) for (int comp = 0; comp < 3; comp++) for (int k = 0; k < 4; k++) { int i = 4 * g + k; dstq[12 * g + 4 * comp + k] = src[3 * (i < nv ? i : 0) + comp]; }
  }
  m3 R; for (int i = 0; i < 9; i++) R.m[i] = (i % 4 == 0) ? 1.f : 0.f;
  f3 a, b, n; float d = 0.f;
  bool ov = gjk_cores(v.data(), vq, 0, 0, nA, nA, gB, nB, R, f3(), a, b, n, d);
  pa[0] = a.x; pa[1] = a.y; pa[2] = a.z; pb[0] = b.x; pb[1] = b.y; pb[2] = b.z; nrm[0] = n.x; nrm[1] = n.y; nrm[2] = n.z; *dist = d;
  return ov ? 1 : 0;
}
#endif
