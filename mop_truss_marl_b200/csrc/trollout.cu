// Host-resident rollout step (include/trollout.h): pieces of the batch flow through three streams so that the
// PCIe upload, the two kernels-with-C-ABI (tactor_act, tfem_step) and the PCIe download overlap.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <new>
#include <chrono>
#include <string>
#include <vector>

#include "../../include/trollout.h"
#include "tfem_kernels.cuh"

namespace {
struct Dev {
  float *x_n = nullptr, *A_s = nullptr, *A_ts = nullptr, *A_cs = nullptr, *raw_n = nullptr, *raw_e = nullptr, *mr = nullptr;
  float *point = nullptr, *a_geo = nullptr, *a_topo = nullptr, *x_p = nullptr, *A_p = nullptr, *A_n = nullptr;
  float *node_y = nullptr, *elem_sec = nullptr;     // compact live columns of the raw tables
  int32_t *status = nullptr, *n_pf = nullptr;
  uint8_t* coin = nullptr;
  uint8_t* family = nullptr;                        // the parent's family ids (an env handle made by tfem_create_mixed)
};
constexpr int PMAX = 50;

// Captured (pinned + mapped) steps move the arrays of a piece across the link with ONE kernel per direction that reads / writes
// the mapped host memory directly, instead of one DMA copy per array: 11 up + 13 down per piece, each with a few microseconds
// of fixed cost on its copy engine -- which is what made more than two pieces a loss.  TROLLOUT_ZEROCOPY=0 goes back to the
// copy engines (2: kernel for the download only, 3: for the upload only); TROLLOUT_ZC_UP / TROLLOUT_ZC_DOWN: CTAs of the two
// kernels (32 each: enough requests in flight for the link, few enough SMs taken from the actor and the env-step).
constexpr int COPY_MAX = 16;
struct CopyList {
  void* dst[COPY_MAX];
  const void* src[COPY_MAX];
  unsigned long long end16[COPY_MAX];       // running total of 16-byte units up to and including array i
  unsigned int bytes[COPY_MAX];             // bytes of array i (the tail below 16 bytes is copied bytewise)
  int n;
};
__global__ void __launch_bounds__(256) copy_arrays_kernel(const __grid_constant__ CopyList L) {
  const unsigned long long total = L.n ? L.end16[L.n - 1] : 0ull;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  // four independent 16-byte loads per thread in flight before the first store (reads of host memory have microseconds of latency)
  for (unsigned long long u0 = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; u0 < total; u0 += 4 * stride) {
    uint4 v[4];
    uint4* out[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const unsigned long long u = u0 + i * stride;
      out[i] = nullptr;
      if (u < total) {
        int a = 0;
        while (u >= L.end16[a]) ++a;
        const unsigned long long k = u - (a ? L.end16[a - 1] : 0ull);
        v[i] = reinterpret_cast<const uint4*>(L.src[a])[k];
        out[i] = reinterpret_cast<uint4*>(L.dst[a]) + k;
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (out[i]) *out[i] = v[i];
  }
  if (blockIdx.x == 0 && threadIdx.x < 16 * COPY_MAX) {                  // byte tails
    const int a = threadIdx.x >> 4, j = threadIdx.x & 15;
    if (a < L.n) {
      const unsigned int full = L.bytes[a] & ~15u;
      if (full + j < L.bytes[a]) reinterpret_cast<unsigned char*>(L.dst[a])[full + j] = reinterpret_cast<const unsigned char*>(L.src[a])[full + j];
    }
  }
}
constexpr size_t MAX_GRAPHS = 4, MAX_SEEN = 8;
}  // namespace

struct trollout_handle_s {
  tfem_handle_t env = nullptr;
  int n_agents = 1;
  tactor_handle_t actors[TROLLOUT_MAX_AGENTS] = {};
  int device = 0, max_batch = 0;
  std::vector<int> piece_len;                      // environments per piece (multiples of 32 but the last), sum >= max_batch
  tfem_dims dims{};
  Dev d;                                           // the parent; the last agent's child is stepped over it in place
  // the child buffers of agent k: kid[n_agents - 1] is `d`; the other children get their own state, move range, point,
  // status, actions and coin, so that no child overwrites what a later act or env-step of the same piece still reads
  Dev kid[TROLLOUT_MAX_AGENTS];
  cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr;
  std::vector<cudaEvent_t> ev_in, ev_run;          // ev_run: one per (piece, agent), index piece * n_agents + agent
  cudaEvent_t ev_join = nullptr;
  std::vector<void*> allocs;
  // CUDA graphs of one whole step (every copy and kernel of every piece), replayed while the caller keeps passing the
  // same pinned buffers (a driver that ping-pongs two state tuples alternates between two graphs); a buffer set is
  // captured the second time it is seen.  The OU-noise seed / call index of every agent travel through h_ctr -> d_ctr.
  struct Graph {
    std::vector<uintptr_t> key;
    cudaGraphExec_t exec = nullptr;
    int64_t env_launches = 0, actor_launches[TROLLOUT_MAX_AGENTS] = {};
    int pieces = 0;
    uint64_t last_use = 0;
  };
  std::vector<Graph> graphs;                       // at most MAX_GRAPHS, least recently used one is replaced
  std::vector<std::vector<uintptr_t>> seen_once;   // at most MAX_SEEN
  uint64_t tick = 0;
  uint64_t* h_ctr = nullptr;      // pinned: [seed, first call index] per agent
  uint64_t* d_ctr = nullptr;
  bool use_graph = true;
  bool timeline = false;                           // TROLLOUT_TIMELINE=1: print per-piece event times (direct path)
  std::vector<cudaEvent_t> tl;
  // TROLLOUT_HOSTTIME=1: host-side time of the graph path, printed by trollout_destroy: [checks + key, graph launch, wait]
  bool zerocopy = true;                            // TROLLOUT_ZEROCOPY=0 turns it off
  bool zc_capture = false;                         // the step being captured: every host buffer is mapped at its own address
  int zc_up = 32, zc_down = 32;                    // CTAs of the copy kernels (TROLLOUT_ZC_UP / TROLLOUT_ZC_DOWN); mode 2: download only, 3: upload only
  int zc_mode = 1;
  bool hosttime = false;
  double host_ns[3] = {0, 0, 0};
  long host_steps = 0;
};

namespace {
thread_local std::string g_roll_err;
int rfail(int code, const std::string& m) { g_roll_err = m; return code; }

template <typename T>
cudaError_t dalloc(trollout_handle_s* h, T** p, size_t count) {
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T) + 256);
  if (e == cudaSuccess) h->allocs.push_back(*p);
  return e;
}
// the child buffers one agent writes (the parent-only inputs x_p, A_p, A_n, n_pf stay null)
cudaError_t alloc_child(trollout_handle_s* h, Dev& c, size_t B) {
  const size_t N = h->dims.N, E = h->dims.E;
  cudaError_t e = dalloc(h, &c.x_n, B * N * 13);
  if (e == cudaSuccess) e = dalloc(h, &c.A_s, B * N * N);
  if (e == cudaSuccess) e = dalloc(h, &c.A_ts, B * N * N);
  if (e == cudaSuccess) e = dalloc(h, &c.A_cs, B * N * N);
  if (e == cudaSuccess) e = dalloc(h, &c.raw_n, B * N * 12);
  if (e == cudaSuccess) e = dalloc(h, &c.raw_e, B * E * 21);
  if (e == cudaSuccess) e = dalloc(h, &c.mr, B * N * 2);
  if (e == cudaSuccess) e = dalloc(h, &c.node_y, B * N);
  if (e == cudaSuccess) e = dalloc(h, &c.elem_sec, B * E);
  if (e == cudaSuccess) e = dalloc(h, &c.point, B * 4);
  if (e == cudaSuccess) e = dalloc(h, &c.a_geo, B * N * 2);
  if (e == cudaSuccess) e = dalloc(h, &c.a_topo, B * N * 3);
  if (e == cudaSuccess) e = dalloc(h, &c.status, B);
  if (e == cudaSuccess) e = dalloc(h, &c.coin, B);
  return e;
}
// an upload-done event per piece, a kernels-done event per piece and agent
cudaError_t piece_events(trollout_handle_s* h, size_t n) {
  cudaError_t e = cudaSuccess;
  auto grow = [&](std::vector<cudaEvent_t>& v, size_t count) {
    while (v.size() < count && e == cudaSuccess) {
      cudaEvent_t a = nullptr;
      e = cudaEventCreateWithFlags(&a, cudaEventDisableTiming);
      if (e == cudaSuccess) v.push_back(a);
    }
  };
  grow(h->ev_in, n);
  grow(h->ev_run, n * (size_t)h->n_agents);
  return e;
}
}  // namespace

extern "C" {

const char* trollout_last_error(void) { return g_roll_err.c_str(); }

int trollout_create(tfem_handle_t env, tactor_handle_t actor, int max_batch, int pieces, trollout_handle_t* out) {
  return trollout_create_agents(env, &actor, 1, max_batch, pieces, out);
}

int trollout_create_agents(tfem_handle_t env, const tactor_handle_t* actors, int n_agents, int max_batch, int pieces,
                           trollout_handle_t* out) {
  if (!env || !actors || !out) return rfail(TFEM_ERR_ARG, "null argument");
  *out = nullptr;
  if (n_agents < 1 || n_agents > TROLLOUT_MAX_AGENTS)
    return rfail(TFEM_ERR_ARG, "n_agents must be in 1.." + std::to_string(TROLLOUT_MAX_AGENTS) + ", got " + std::to_string(n_agents));
  for (int k = 0; k < n_agents; ++k) {
    if (!actors[k]) return rfail(TFEM_ERR_ARG, "null argument");
    // every actor draws its noise from its own call counter: one handle twice would interleave the two agents' calls
    for (int j = 0; j < k; ++j)
      if (actors[j] == actors[k]) return rfail(TFEM_ERR_ARG, "the agents must be distinct actor handles");
  }
  if (max_batch <= 0 || pieces <= 0) return rfail(TFEM_ERR_ARG, "max_batch and pieces must be positive");
  trollout_handle_s* h = new (std::nothrow) trollout_handle_s();
  if (!h) return rfail(TFEM_ERR_ARG, "out of host memory");
  h->env = env; h->max_batch = max_batch; h->n_agents = n_agents;
  for (int k = 0; k < n_agents; ++k) h->actors[k] = actors[k];
  if (tfem_get_dims(env, &h->dims) != TFEM_OK) { delete h; return rfail(TFEM_ERR_ARG, "bad env handle"); }
  int piece = (max_batch + pieces - 1) / pieces;
  piece = (piece + 31) / 32 * 32;                  // piece boundaries on 32 environments: every sub-array stays 16-byte aligned
  for (int lo = 0; lo < max_batch; lo += piece) h->piece_len.push_back(piece);
  h->device = h->dims.device;
  if (h->device < 0) { delete h; return rfail(TFEM_ERR_CUDA, "tables-only env handle: libtfem has no CPU path"); }
  int prev_dev = -1;
  cudaGetDevice(&prev_dev);
  cudaError_t e = cudaSetDevice(h->device);
  const size_t B = (size_t)max_batch, N = h->dims.N;
  if (e == cudaSuccess) e = alloc_child(h, h->d, B);
  if (e == cudaSuccess) e = dalloc(h, &h->d.x_p, B * PMAX * 4);
  if (e == cudaSuccess) e = dalloc(h, &h->d.A_p, B * PMAX * PMAX);
  if (e == cudaSuccess) e = dalloc(h, &h->d.A_n, N * N);
  if (e == cudaSuccess) e = dalloc(h, &h->d.n_pf, B);
  if (e == cudaSuccess && tfem::handle_is_mixed(env)) e = dalloc(h, &h->d.family, B);
  for (int k = 0; k + 1 < n_agents && e == cudaSuccess; ++k) e = alloc_child(h, h->kid[k], B);
  h->kid[n_agents - 1] = h->d;
  if (e == cudaSuccess) {
    std::vector<float> an(N * N);
    if (tfem_get_table(env, TFEM_TAB_A_N, an.data(), an.size() * 4) != TFEM_OK) e = cudaErrorInvalidValue;
    else e = cudaMemcpy(h->d.A_n, an.data(), an.size() * 4, cudaMemcpyHostToDevice);
  }
  if (e == cudaSuccess) e = dalloc(h, &h->d_ctr, 2 * TROLLOUT_MAX_AGENTS);
  if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&h->h_ctr), 16 * TROLLOUT_MAX_AGENTS, cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
  if (const char* v = getenv("TROLLOUT_NO_GRAPH")) h->use_graph = (v[0] == '0');
  if (const char* v = getenv("TROLLOUT_ZEROCOPY")) { h->zc_mode = atoi(v); h->zerocopy = h->zc_mode >= 1; }
  if (const char* v = getenv("TROLLOUT_ZC_UP")) { h->zc_up = atoi(v); if (h->zc_up < 1) h->zc_up = 1; }
  if (const char* v = getenv("TROLLOUT_ZC_DOWN")) { h->zc_down = atoi(v); if (h->zc_down < 1) h->zc_down = 1; }
  if (const char* v = getenv("TROLLOUT_HOSTTIME")) h->hosttime = (v[0] == '1');
  if (const char* v = getenv("TROLLOUT_TIMELINE")) { h->timeline = (v[0] == '1'); if (h->timeline) h->use_graph = false; }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_run, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = piece_events(h, h->piece_len.size());
  if (prev_dev >= 0) cudaSetDevice(prev_dev);
  if (e != cudaSuccess) {
    trollout_destroy(h);
    return rfail(TFEM_ERR_CUDA, std::string("rollout setup: ") + cudaGetErrorString(e));
  }
  *out = h;
  return TFEM_OK;
}

int trollout_destroy(trollout_handle_t h) {
  if (!h) return TFEM_OK;
  if (h->hosttime && h->host_steps)
    fprintf(stderr, "[trollout host time, us per replayed step over %ld steps] checks %.1f | cudaGraphLaunch %.1f | wait %.1f\n",
            h->host_steps, h->host_ns[0] / h->host_steps * 1e-3, h->host_ns[1] / h->host_steps * 1e-3,
            h->host_ns[2] / h->host_steps * 1e-3);
  for (auto& g : h->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->h_ctr) cudaFreeHost(h->h_ctr);
  for (cudaEvent_t ev : h->ev_in) cudaEventDestroy(ev);
  for (cudaEvent_t ev : h->ev_run) cudaEventDestroy(ev);
  if (h->s_in) cudaStreamDestroy(h->s_in);
  if (h->s_run) cudaStreamDestroy(h->s_run);
  if (h->s_out) cudaStreamDestroy(h->s_out);
  for (void* p : h->allocs) cudaFree(p);
  delete h;
  return TFEM_OK;
}

int trollout_bytes_per_env(trollout_handle_t h, int P, int compact_columns, size_t* h2d, size_t* d2h) {
  if (!h) return rfail(TFEM_ERR_ARG, "null argument");
  const size_t N = h->dims.N, E = h->dims.E;
  const size_t graph = 4 * (N * 13 + 3 * N * N + N * 2), tables = 4 * (N * 12 + E * 21), cols = 4 * (N + E);
  const size_t K = (size_t)h->n_agents;             // the parent goes up once with one coin per agent; every child comes down
  const size_t family = tfem::handle_family_count(h->env) > 1 ? 1 : 0;   // the parent's family id
  if (h2d) *h2d = graph + (compact_columns ? cols : tables) + K + family + 4 * ((size_t)P * 4 + (size_t)P * P);
  if (d2h) *d2h = K * (graph + tables + (compact_columns ? cols : 0) + 4 * 4 + 4 + 4 * (N * 2 + N * 3));
  return TFEM_OK;
}

int trollout_set_pieces(trollout_handle_t h, const int32_t* sizes, int n) {
  if (!h || !sizes || n < 1 || n > 64) return rfail(TFEM_ERR_ARG, "1..64 piece sizes are required");
  long long sum = 0;
  for (int i = 0; i < n; ++i) {
    if (sizes[i] <= 0 || (i + 1 < n && sizes[i] % 32 != 0))
      return rfail(TFEM_ERR_ARG, "piece sizes must be positive, and multiples of 32 except the last");
    sum += sizes[i];
  }
  if (sum < h->max_batch) return rfail(TFEM_ERR_ARG, "the piece sizes must add up to max_batch");
  int prev_dev = -1;
  cudaGetDevice(&prev_dev);
  cudaSetDevice(h->device);
  const cudaError_t e = piece_events(h, (size_t)n);
  if (prev_dev >= 0) cudaSetDevice(prev_dev);
  if (e != cudaSuccess) return rfail(TFEM_ERR_CUDA, std::string("rollout pieces: ") + cudaGetErrorString(e));
  h->piece_len.assign(sizes, sizes + n);
  return trollout_forget_buffers(h);               // the cached graphs were captured with the old boundaries
}

int trollout_forget_buffers(trollout_handle_t h) {
  if (!h) return rfail(TFEM_ERR_ARG, "null argument");
  for (auto& g : h->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  h->graphs.clear();
  h->seen_once.clear();
  return TFEM_OK;
}

// Enqueues every copy and kernel of one step on the three streams.  ctr_dev == nullptr: the noise call index is taken
// from the actor handles (tactor_act); otherwise from device memory (tactor_act_dev, graph capture: [seed, first call
// index] of agent k at ctr_dev[2k]).  join: make s_in wait for the last download (needed to close a capture).  Per
// piece: the parent goes up once; then for every agent k in turn act, env-step and the download of child k.
// family != nullptr (host [B]): the ids go up with the parent and the env-steps are tfem_step_mixed.
static int enqueue_step(trollout_handle_s* h, int B, const uint8_t* family, const trollout_agents_io* io, const float* mu,
                        const float* theta, const float* sigma, const uint64_t* seed, const uint64_t* ctr_dev, bool join,
                        int* pieces_out) {
  const trollout_state& si = io->in;
  const int K = h->n_agents;
  const size_t N = h->dims.N, E = h->dims.E, P = (size_t)io->P;
  const Dev& d = h->d;
  const bool compact = si.node_y && si.element_section;
  cudaError_t e = cudaSuccess;
  // a failure in the middle of a step must not return while copies issued for earlier pieces still touch the
  // caller's host buffers
  auto drain = [&]() { cudaStreamSynchronize(h->s_in); cudaStreamSynchronize(h->s_run); cudaStreamSynchronize(h->s_out); };
  // zero-copy path: only for the captured (all-pinned) step
  const bool zc = h->zerocopy && ctr_dev != nullptr && h->zc_capture;
  CopyList ups{}, downs{};
  auto add = [&](CopyList& L, void* dst, const void* src, size_t bytes) {
    if (bytes == 0) return;
    if (L.n >= COPY_MAX || (reinterpret_cast<uintptr_t>(dst) & 15) || (reinterpret_cast<uintptr_t>(src) & 15) || bytes > 0xffffffffull) {
      e = cudaErrorInvalidValue;
      return;
    }
    L.dst[L.n] = dst; L.src[L.n] = src; L.bytes[L.n] = (unsigned int)bytes;
    L.end16[L.n] = (L.n ? L.end16[L.n - 1] : 0ull) + bytes / 16;
    ++L.n;
  };
  const bool zc_u = zc && h->zc_mode != 2, zc_d = zc && h->zc_mode != 3;
  auto flush = [&](CopyList& L, cudaStream_t st) {
    if (e == cudaSuccess && L.n) {
      copy_arrays_kernel<<<(st == h->s_in) ? h->zc_up : h->zc_down, 256, 0, st>>>(L);
      e = cudaGetLastError();
    }
    L.n = 0;
  };
  auto up = [&](void* dst, const void* src, size_t bytes) {
    if (e != cudaSuccess || !src) return;
    if (zc_u) add(ups, dst, src, bytes);
    else e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, h->s_in);
  };
  auto down = [&](void* dst, const void* src, size_t bytes) {
    if (e != cudaSuccess || !dst) return;
    if (zc_d) add(downs, dst, src, bytes);
    else e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, h->s_out);
  };
  if (ctr_dev) {
    up(h->d_ctr, h->h_ctr, 16 * (size_t)K);
    flush(ups, h->s_in);
  }
  if (h->timeline && !ctr_dev) {
    const size_t need = 1 + 4 * h->ev_in.size();
    while (h->tl.size() < need) { cudaEvent_t ev; cudaEventCreate(&ev); h->tl.push_back(ev); }
    cudaEventRecord(h->tl[0], h->s_in);
  }
  // the timeline's run and download events of a piece are re-recorded for every agent: it reports the last child
  int piece_idx = 0;
  for (int lo = 0; lo < B && e == cudaSuccess; lo += h->piece_len[piece_idx], ++piece_idx) {
    const int len = h->piece_len[piece_idx];
    const size_t l = (size_t)lo, nb = (size_t)((lo + len <= B) ? len : (B - lo));
    // ---- upload ----
    up(d.x_n + l * N * 13, si.x_n + l * N * 13, nb * N * 13 * 4);
    up(d.A_s + l * N * N, si.A_s + l * N * N, nb * N * N * 4);
    up(d.A_ts + l * N * N, si.A_n_ts + l * N * N, nb * N * N * 4);
    up(d.A_cs + l * N * N, si.A_n_cs + l * N * N, nb * N * N * 4);
    if (compact) {                                   // only the two columns _set_model reads
      up(d.node_y + l * N, si.node_y + l * N, nb * N * 4);
      up(d.elem_sec + l * E, si.element_section + l * E, nb * E * 4);
    } else {
      up(d.raw_n + l * N * 12, si.nN_x_n + l * N * 12, nb * N * 12 * 4);
      up(d.raw_e + l * E * 21, si.nN_x_e + l * E * 21, nb * E * 21 * 4);
    }
    up(d.mr + l * N * 2, si.move_range + l * N * 2, nb * N * 2 * 4);
    up(d.x_p + l * P * 4, io->x_p + l * P * 4, nb * P * 4 * 4);
    up(d.A_p + l * P * P, io->A_p + l * P * P, nb * P * P * 4);
    for (int k = 0; k < K; ++k)
      if (io->child[k].coin) up(h->kid[k].coin + l, io->child[k].coin + l, nb);
    if (io->n_pf) up(d.n_pf + l, io->n_pf + l, nb * 4);
    if (family) up(d.family + l, family + l, nb);
    flush(ups, h->s_in);
    if (e == cudaSuccess) e = cudaEventRecord(h->ev_in[piece_idx], h->s_in);
    if (h->timeline && !ctr_dev) cudaEventRecord(h->tl[1 + 4 * piece_idx + 0], h->s_in);
    // ---- act + step, then download, agent by agent ----
    if (e == cudaSuccess) e = cudaStreamWaitEvent(h->s_run, h->ev_in[piece_idx], 0);
    if (e != cudaSuccess) break;
    tactor_inputs ai{};
    ai.x_n = d.x_n + l * N * 13; ai.A_n = d.A_n; ai.A_s = d.A_s + l * N * N; ai.A_n_ts = d.A_ts + l * N * N;
    ai.A_n_cs = d.A_cs + l * N * N; ai.x_p = d.x_p + l * P * 4; ai.A_p = d.A_p + l * P * P;
    ai.n_pf = io->n_pf ? d.n_pf + l : nullptr; ai.P = io->P;
    for (int k = 0; k < K && e == cudaSuccess; ++k) {
      const Dev& c = h->kid[k];                       // == d for the last agent: its child is written over the parent
      const trollout_child& ch = io->child[k];
      const trollout_state& so = ch.out;
      int rc = ctr_dev ? tactor_act_dev(h->actors[k], (int)nb, &ai, c.a_geo + l * N * 2, c.a_topo + l * N * 3, mu[k], theta[k],
                                        sigma[k], ctr_dev + 2 * k, (uint32_t)piece_idx, h->s_run)
                       : tactor_act(h->actors[k], (int)nb, &ai, c.a_geo + l * N * 2, c.a_topo + l * N * 3, mu[k], theta[k],
                                    sigma[k], seed[k], h->s_run);
      if (rc != TFEM_OK) { if (!ctr_dev) drain(); return rfail(rc, std::string("rollout: ") + tactor_last_error()); }
      if (c.mr != d.mr)                                // the env-step reads and writes the move range in place
        e = cudaMemcpyAsync(c.mr + l * N * 2, d.mr + l * N * 2, nb * N * 2 * 4, cudaMemcpyDeviceToDevice, h->s_run);
      if (e != cudaSuccess) break;
      tfem_step_in in{};
      if (compact) { in.set_node_y = d.node_y + l * N; in.set_element_section = d.elem_sec + l * E; }
      in.set_node = d.raw_n + l * N * 12; in.set_element = d.raw_e + l * E * 21; in.a_geo = c.a_geo + l * N * 2;
      in.a_topo = c.a_topo + l * N * 3; in.coin = ch.coin ? c.coin + l : nullptr; in.move_range = c.mr + l * N * 2;
      tfem_step_out o{};
      o.x_n = c.x_n + l * N * 13; o.A_s = c.A_s + l * N * N; o.A_n_ts = c.A_ts + l * N * N; o.A_n_cs = c.A_cs + l * N * N;
      o.nN_x_n = c.raw_n + l * N * 12; o.nN_x_e = c.raw_e + l * E * 21; o.point = c.point + l * 4; o.status = c.status + l;
      if (so.node_y) o.node_y = c.node_y + l * N;
      if (so.element_section) o.element_section = c.elem_sec + l * E;
      rc = family ? tfem_step_mixed(h->env, (int)nb, d.family + l, &in, &o, h->s_run)
                  : tfem_step(h->env, (int)nb, &in, &o, h->s_run);
      if (rc != TFEM_OK) { if (!ctr_dev) drain(); return rfail(rc, std::string("rollout: ") + tfem_last_error()); }
      cudaEvent_t done = h->ev_run[(size_t)piece_idx * K + k];
      e = cudaEventRecord(done, h->s_run);
      if (h->timeline && !ctr_dev) cudaEventRecord(h->tl[1 + 4 * piece_idx + 1], h->s_run);
      // ---- download of child k: one list per child (a transfer kernel takes at most COPY_MAX arrays) ----
      if (e == cudaSuccess) e = cudaStreamWaitEvent(h->s_out, done, 0);
      down(so.x_n ? so.x_n + l * N * 13 : nullptr, c.x_n + l * N * 13, nb * N * 13 * 4);
      down(so.A_s ? so.A_s + l * N * N : nullptr, c.A_s + l * N * N, nb * N * N * 4);
      down(so.A_n_ts ? so.A_n_ts + l * N * N : nullptr, c.A_ts + l * N * N, nb * N * N * 4);
      down(so.A_n_cs ? so.A_n_cs + l * N * N : nullptr, c.A_cs + l * N * N, nb * N * N * 4);
      down(so.nN_x_n ? so.nN_x_n + l * N * 12 : nullptr, c.raw_n + l * N * 12, nb * N * 12 * 4);
      down(so.nN_x_e ? so.nN_x_e + l * E * 21 : nullptr, c.raw_e + l * E * 21, nb * E * 21 * 4);
      down(so.move_range ? so.move_range + l * N * 2 : nullptr, c.mr + l * N * 2, nb * N * 2 * 4);
      down(so.node_y ? so.node_y + l * N : nullptr, c.node_y + l * N, nb * N * 4);
      down(so.element_section ? so.element_section + l * E : nullptr, c.elem_sec + l * E, nb * E * 4);
      down(ch.point ? ch.point + l * 4 : nullptr, c.point + l * 4, nb * 4 * 4);
      down(ch.status ? ch.status + l : nullptr, c.status + l, nb * 4);
      down(ch.a_geo ? ch.a_geo + l * N * 2 : nullptr, c.a_geo + l * N * 2, nb * N * 2 * 4);
      down(ch.a_topo ? ch.a_topo + l * N * 3 : nullptr, c.a_topo + l * N * 3, nb * N * 3 * 4);
      flush(downs, h->s_out);
      if (h->timeline && !ctr_dev) cudaEventRecord(h->tl[1 + 4 * piece_idx + 2], h->s_out);
    }
  }
  if (join) {
    if (e == cudaSuccess) e = cudaEventRecord(h->ev_join, h->s_out);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(h->s_in, h->ev_join, 0);
  }
  if (pieces_out) *pieces_out = piece_idx;
  if (e != cudaSuccess) {
    if (!ctr_dev) drain();
    return rfail(TFEM_ERR_CUDA, std::string("rollout step: ") + cudaGetErrorString(e));
  }
  return TFEM_OK;
}

static bool pinned(const void* p, bool* mapped = nullptr) {
  if (!p) return true;
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  if (mapped && a.devicePointer != p) *mapped = false;   // unified addressing: a kernel can use the host address as it is
  return a.type == cudaMemoryTypeHost;
}

static int step_agents(trollout_handle_t h, int B, const uint8_t* family, const trollout_agents_io* io, const float* mu,
                       const float* theta, const float* sigma, const uint64_t* seed) {
  if (B < 0 || B > h->max_batch) return rfail(TFEM_ERR_ARG, "batch exceeds max_batch");
  if (B == 0) return TFEM_OK;
  const int K = h->n_agents;
  const trollout_state& si = io->in;
  const bool compact_in = si.node_y && si.element_section;
  if (!si.x_n || !si.A_s || !si.A_n_ts || !si.A_n_cs || (!compact_in && (!si.nN_x_n || !si.nN_x_e)) || !si.move_range ||
      !io->x_p || !io->A_p)
    return rfail(TFEM_ERR_ARG, "the parent state tuple (tables or their compact columns), x_p and A_p are required");
  if (io->P < 1 || io->P > PMAX) return rfail(TFEM_ERR_ARG, "P must be in 1..50");
  int prev_dev = -1;
  cudaGetDevice(&prev_dev);
  cudaError_t e = (prev_dev == h->device) ? cudaSuccess : cudaSetDevice(h->device);
  struct Restore { int dev; ~Restore() { if (dev >= 0) cudaSetDevice(dev); } } restore{prev_dev == h->device ? -1 : prev_dev};
  if (e != cudaSuccess) return rfail(TFEM_ERR_CUDA, std::string("rollout step: ") + cudaGetErrorString(e));

  // ---- graph path: same pinned buffers as the captured step -> one cudaGraphLaunch instead of ~30 API calls a piece ----
  std::vector<const void*> ptrs = {si.x_n, si.A_s, si.A_n_ts, si.A_n_cs, compact_in ? nullptr : si.nN_x_n,
                                   compact_in ? nullptr : si.nN_x_e, si.move_range, si.node_y, si.element_section,
                                   io->x_p, io->A_p, io->n_pf, family};
  for (int k = 0; k < K; ++k) {
    const trollout_child& c = io->child[k];
    const trollout_state& so = c.out;
    ptrs.insert(ptrs.end(), {c.coin, so.x_n, so.A_s, so.A_n_ts, so.A_n_cs, so.nN_x_n, so.nN_x_e, so.move_range, so.node_y,
                             so.element_section, c.point, c.status, c.a_geo, c.a_topo});
  }
  const auto t_begin = std::chrono::steady_clock::now();
  if (h->use_graph) {
    std::vector<uintptr_t> key;
    for (const void* p : ptrs) key.push_back(reinterpret_cast<uintptr_t>(p));
    key.push_back((uintptr_t)B); key.push_back((uintptr_t)io->P); key.push_back(family != nullptr);
    for (int k = 0; k < K; ++k) {
      uint32_t fb[3];
      memcpy(&fb[0], &mu[k], 4); memcpy(&fb[1], &theta[k], 4); memcpy(&fb[2], &sigma[k], 4);
      key.push_back(fb[0]); key.push_back(fb[1]); key.push_back(fb[2]);
    }
    trollout_handle_s::Graph* hit = nullptr;
    for (auto& g : h->graphs) if (g.key == key) hit = &g;
    if (!hit) {
      bool second = false;
      for (auto& k : h->seen_once) second = second || (k == key);
      if (!second) {
        if (h->seen_once.size() >= MAX_SEEN) h->seen_once.erase(h->seen_once.begin());
        h->seen_once.push_back(key);
      } else {
        bool all_pinned = true, all_mapped = true;
        for (const void* p : ptrs) all_pinned = all_pinned && pinned(p, &all_mapped);
        all_mapped = all_mapped && pinned(h->h_ctr, &all_mapped);
        if (all_pinned) {
          h->zc_capture = all_mapped;
          trollout_handle_s::Graph ng;
          int64_t act0[TROLLOUT_MAX_AGENTS];
          const int64_t env0 = tfem_launch_count(h->env);
          for (int k = 0; k < K; ++k) act0[k] = tactor_launch_count(h->actors[k]);
          e = cudaStreamBeginCapture(h->s_in, cudaStreamCaptureModeRelaxed);
          if (e != cudaSuccess) return rfail(TFEM_ERR_CUDA, std::string("rollout capture: ") + cudaGetErrorString(e));
          const int rc = enqueue_step(h, B, family, io, mu, theta, sigma, seed, h->d_ctr, true, &ng.pieces);
          cudaGraph_t g = nullptr;
          e = cudaStreamEndCapture(h->s_in, &g);
          // the kernels were recorded, not run: take their bookings back (every replay books them)
          ng.env_launches = tfem_launch_count(h->env) - env0;
          tfem_book_launches(h->env, -ng.env_launches);
          for (int k = 0; k < K; ++k) {
            ng.actor_launches[k] = tactor_launch_count(h->actors[k]) - act0[k];
            tactor_reserve_calls(h->actors[k], 0, -ng.actor_launches[k]);
          }
          if (rc != TFEM_OK) { if (g) cudaGraphDestroy(g); cudaGetLastError(); return rc; }
          if (e == cudaSuccess) e = cudaGraphInstantiate(&ng.exec, g, 0);
          if (g) cudaGraphDestroy(g);
          if (e != cudaSuccess) return rfail(TFEM_ERR_CUDA, std::string("rollout capture: ") + cudaGetErrorString(e));
          ng.key = key;
          if (h->graphs.size() >= MAX_GRAPHS) {
            size_t lru = 0;
            for (size_t i = 1; i < h->graphs.size(); ++i) if (h->graphs[i].last_use < h->graphs[lru].last_use) lru = i;
            cudaGraphExecDestroy(h->graphs[lru].exec);
            h->graphs[lru] = ng;
            hit = &h->graphs[lru];
          } else {
            h->graphs.push_back(ng);
            hit = &h->graphs.back();
          }
        }
      }
    }
    if (hit) {
      // the graph's copy nodes were captured for pinned memory: a buffer that was freed and whose address now belongs
      // to a pageable allocation must not be replayed against
      bool still_pinned = true;
      for (const void* p : ptrs) still_pinned = still_pinned && pinned(p);
      if (!still_pinned) {
        trollout_forget_buffers(h);
        hit = nullptr;
      }
    }
    if (hit) {
      hit->last_use = ++h->tick;
      for (int k = 0; k < K; ++k) {                  // the call indices the direct path would have drawn
        const bool noise = !(sigma[k] == 0.f && theta[k] == 0.f);
        h->h_ctr[2 * k] = seed[k];
        h->h_ctr[2 * k + 1] = tactor_reserve_calls(h->actors[k], noise ? (uint32_t)hit->pieces : 0u, hit->actor_launches[k]);
      }
      tfem_book_launches(h->env, hit->env_launches);
      const auto t_launch = std::chrono::steady_clock::now();
      e = cudaGraphLaunch(hit->exec, h->s_in);
      const auto t_wait = std::chrono::steady_clock::now();
      if (e == cudaSuccess) e = cudaStreamSynchronize(h->s_in);
      if (h->hosttime) {
        const auto t_end = std::chrono::steady_clock::now();
        h->host_ns[0] += std::chrono::duration<double, std::nano>(t_launch - t_begin).count();
        h->host_ns[1] += std::chrono::duration<double, std::nano>(t_wait - t_launch).count();
        h->host_ns[2] += std::chrono::duration<double, std::nano>(t_end - t_wait).count();
        ++h->host_steps;
      }
      if (e != cudaSuccess) return rfail(TFEM_ERR_CUDA, std::string("rollout step: ") + cudaGetErrorString(e));
      return TFEM_OK;
    }
  }
  // ---- direct path (pageable buffers, or TROLLOUT_NO_GRAPH=1) ----
  int np_done = 0;
  if (int rc = enqueue_step(h, B, family, io, mu, theta, sigma, seed, nullptr, false, &np_done)) {
    // a piece failed mid-step: copies of earlier pieces may still be reading / writing the caller's host buffers
    cudaStreamSynchronize(h->s_in); cudaStreamSynchronize(h->s_run); cudaStreamSynchronize(h->s_out);
    return rc;
  }
  e = cudaStreamSynchronize(h->s_out);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->s_in);
  if (h->timeline && e == cudaSuccess) {
    fprintf(stderr, "[trollout timeline, ms since first upload]");
    for (int i = 0; i < np_done; ++i) {
      float a = 0, b = 0, c = 0;
      cudaEventElapsedTime(&a, h->tl[0], h->tl[1 + 4 * i + 0]);
      cudaEventElapsedTime(&b, h->tl[0], h->tl[1 + 4 * i + 1]);
      cudaEventElapsedTime(&c, h->tl[0], h->tl[1 + 4 * i + 2]);
      fprintf(stderr, " | piece %d: up %.3f run %.3f down %.3f", i, a, b, c);
    }
    fprintf(stderr, "\n");
  }
  if (e != cudaSuccess) return rfail(TFEM_ERR_CUDA, std::string("rollout step: ") + cudaGetErrorString(e));
  return TFEM_OK;
}

// the plain steps serve an env handle of one family (as tfem_step does)
static int single_family(trollout_handle_t h, const char* call, const char* instead) {
  const int F = tfem::handle_family_count(h->env);
  if (F == 1) return TFEM_OK;
  return rfail(TFEM_ERR_ARG, std::string(call) + ": the env handle holds " + std::to_string(F) + " families; use " + instead);
}

// the _mixed steps need the mixed env-step (tfem_create_mixed) and ids the transfer kernel can read in 16-byte units
static int mixed_family(trollout_handle_t h, const uint8_t* family, const char* call) {
  if (!tfem::handle_is_mixed(h->env))
    return rfail(TFEM_ERR_ARG, std::string(call) + ": the env handle was made by tfem_create; make it with tfem_create_mixed");
  if (!family) return rfail(TFEM_ERR_ARG, std::string(call) + ": the family ids are required");
  if (reinterpret_cast<uintptr_t>(family) & 15)
    return rfail(TFEM_ERR_ALIGN, std::string(call) + ": the family ids must be 16-byte aligned");
  return TFEM_OK;
}

// the one-agent call as a trollout_agents_io of one child
static trollout_agents_io one_child(const trollout_io* io) {
  trollout_agents_io a{};
  a.in = io->in; a.x_p = io->x_p; a.A_p = io->A_p; a.n_pf = io->n_pf; a.P = io->P;
  a.child[0].out = io->out; a.child[0].coin = io->coin; a.child[0].point = io->point; a.child[0].status = io->status;
  a.child[0].a_geo = io->a_geo; a.child[0].a_topo = io->a_topo;
  return a;
}

int trollout_step_host(trollout_handle_t h, int B, const trollout_io* io, float mu, float theta, float sigma,
                       uint64_t seed) {
  if (!h || !io) return rfail(TFEM_ERR_ARG, "null argument");
  if (h->n_agents != 1)
    return rfail(TFEM_ERR_ARG, "the rollout handle runs " + std::to_string(h->n_agents) +
                                   " agents (trollout_create_agents): step it with trollout_step_agents_host");
  if (int rc = single_family(h, "trollout_step_host", "trollout_step_host_mixed")) return rc;
  const trollout_agents_io a = one_child(io);
  return step_agents(h, B, nullptr, &a, &mu, &theta, &sigma, &seed);
}

int trollout_step_agents_host(trollout_handle_t h, int B, const trollout_agents_io* io, const float* mu,
                              const float* theta, const float* sigma, const uint64_t* seed) {
  if (!h || !io || !mu || !theta || !sigma || !seed) return rfail(TFEM_ERR_ARG, "null argument");
  if (int rc = single_family(h, "trollout_step_agents_host", "trollout_step_agents_host_mixed")) return rc;
  return step_agents(h, B, nullptr, io, mu, theta, sigma, seed);
}

int trollout_step_host_mixed(trollout_handle_t h, int B, const uint8_t* family, const trollout_io* io, float mu,
                             float theta, float sigma, uint64_t seed) {
  if (!h || !io) return rfail(TFEM_ERR_ARG, "null argument");
  if (h->n_agents != 1)
    return rfail(TFEM_ERR_ARG, "the rollout handle runs " + std::to_string(h->n_agents) +
                                   " agents (trollout_create_agents): step it with trollout_step_agents_host_mixed");
  if (int rc = mixed_family(h, family, "trollout_step_host_mixed")) return rc;
  const trollout_agents_io a = one_child(io);
  return step_agents(h, B, family, &a, &mu, &theta, &sigma, &seed);
}

int trollout_step_agents_host_mixed(trollout_handle_t h, int B, const uint8_t* family, const trollout_agents_io* io,
                                    const float* mu, const float* theta, const float* sigma, const uint64_t* seed) {
  if (!h || !io || !mu || !theta || !sigma || !seed) return rfail(TFEM_ERR_ARG, "null argument");
  if (int rc = mixed_family(h, family, "trollout_step_agents_host_mixed")) return rc;
  return step_agents(h, B, family, io, mu, theta, sigma, seed);
}

}  // extern "C"
