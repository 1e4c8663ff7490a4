/* trollout.h -- C ABI of the host-resident rollout step (libtfem.so).
 *
 * One call = one pass of the reference driver's inner loop for B environments whose state tuple lives in HOST memory
 * (master_DDPG_truss2D_MO.py:167-260: agents[k].act(state...) then game._game_modify(set_node, set_element, nC_e,
 * actions)): the state tuple goes to the device, the actor acts (tactor_act), the environments step (tfem_step), and
 * the new state tuple, the objective point, the status flags and the clipped actions come back.
 *
 * The environments are independent, so the batch is cut into `pieces` pieces that run through three CUDA streams
 * (upload / act + step / download): piece i+1 uploads while piece i computes and piece i-1 downloads.  Host buffers
 * should be pinned (cudaHostAlloc / torch pin_memory); pageable buffers work but do not overlap.
 *
 * With pinned buffers the whole step (every copy and kernel of every piece) is captured into a CUDA graph the second
 * time a set of buffer addresses is seen and replayed afterwards (four graphs are kept: a driver that ping-pongs two
 * state tuples alternates between two of them); replayed steps give the bits of directly enqueued ones, OU noise
 * included.  TROLLOUT_NO_GRAPH=1 disables the graphs, TROLLOUT_TIMELINE=1 prints a per-piece event timeline to stderr.
 *
 * In a captured step the arrays of a piece cross the link through ONE transfer kernel per direction that reads / writes the
 * pinned host arrays at their mapped addresses (unified addressing, verified per buffer; otherwise, on the uncaptured path
 * and with TROLLOUT_ZEROCOPY=0 every array is a cudaMemcpyAsync on a copy engine).  Same bytes over the link, but none of
 * the per-copy cost of the 11 + 13 arrays of a piece, so the batch can be cut finer (trollout_set_pieces).
 * TROLLOUT_HOSTTIME=1 prints the host-side share of the replayed steps (checks, cudaGraphLaunch, wait) at destroy time.
 *
 * trollout_create_agents / trollout_step_agents_host run the driver's whole inner step -- up to three agents acting on
 * the same parent -- in one call: the parent crosses the link once instead of once per agent, and one graph launch
 * and one pipeline fill serve all agents.
 *
 * trollout_step_host_mixed / trollout_step_agents_host_mixed step a rollout whose env handle was made by
 * tfem_create_mixed: the batch of the training driver, where every episode has its own shape and truss type
 * (train/code/master_DDPG_truss2D_MO.py:787-815).  The parent's family ids go up with the parent, one tfem_step_mixed
 * launch per piece and agent steps environments of every family, and every child keeps its parent's ids.
 */
#ifndef TROLLOUT_H_
#define TROLLOUT_H_

#include <stddef.h>
#include <stdint.h>

#include "tactor.h"
#include "tfem.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct trollout_handle_s* trollout_handle_t;

/* the part of the reference's state tuple that changes from step to step (truss2D_ENV.py:354), host pointers */
typedef struct trollout_state {
  float* x_n;        /* [B,N,13] */
  float* A_s;        /* [B,N,N]  */
  float* A_n_ts;     /* [B,N,N]  */
  float* A_n_cs;     /* [B,N,N]  */
  float* nN_x_n;     /* [B,N,12] */
  float* nN_x_e;     /* [B,E,21] */
  float* move_range; /* [B,N,2]  the model's max_up/max_down left by the previous call (tfem_step_in.move_range) */
  /* optional compact copies of the two table columns _set_model reads (truss2D_ENV.py:365, :369): node_y =
   * nN_x_n[:, :, 1], element_section = nN_x_e[:, :, 0].  `out`: written when non-NULL.  `in`: when BOTH are non-NULL
   * they are uploaded instead of the two full tables (4 (N + E) instead of 4 (12 N + 21 E) bytes per environment), and
   * nN_x_n / nN_x_e of `in` are not read and may be NULL; otherwise the full tables go up as before. */
  float* node_y;          /* [B,N] */
  float* element_section; /* [B,E] */
} trollout_state;

typedef struct trollout_io {
  trollout_state in;       /* parent state (read) */
  const uint8_t* coin;     /* [B] symmetry coin, NULL = all 0 */
  const float* x_p;        /* [B,P,4] Pareto-front graph (truss2D_ENV.py:22-41) */
  const float* A_p;        /* [B,P,P] */
  const int32_t* n_pf;     /* [B] valid Pareto rows, NULL = all P */
  int32_t P;
  trollout_state out;      /* child state (written); may alias `in` */
  float* point;            /* [B,4]  */
  int32_t* status;         /* [B]    */
  float* a_geo;            /* [B,N,2] the actions as _game_modify left them (clipped) */
  float* a_topo;           /* [B,N,3] */
} trollout_io;

/* Several agents on one parent (master_DDPG_truss2D_MO.py:249-260: for k = 0, 1, 2 agents[k].act(state) then
 * _game_modify(...) on that same parent; the training driver's transition holds the parent and the three children,
 * train/code/truss2D_RL.py:439-456).  One child block per agent; each _game_modify draws its own coin
 * (truss2D_ENV.py:460). */
#define TROLLOUT_MAX_AGENTS 3

typedef struct trollout_child {
  trollout_state out;      /* child state (written); must not alias the parent or another child */
  const uint8_t* coin;     /* [B] symmetry coin, NULL = all 0 */
  float* point;            /* [B,4]  */
  int32_t* status;         /* [B]    */
  float* a_geo;            /* [B,N,2] this agent's actions as _game_modify left them (clipped) */
  float* a_topo;           /* [B,N,3] */
} trollout_child;

typedef struct trollout_agents_io {
  trollout_state in;       /* parent state (read), uploaded once for all agents; compact columns as in trollout_io */
  const float* x_p;        /* [B,P,4] Pareto-front graph */
  const float* A_p;        /* [B,P,P] */
  const int32_t* n_pf;     /* [B] valid Pareto rows, NULL = all P */
  int32_t P;
  trollout_child child[TROLLOUT_MAX_AGENTS];   /* entries 0 .. n_agents-1 are used */
} trollout_agents_io;

/* env and actor must live on the same device; max_batch bounds B of later calls (device buffers are allocated once);
 * pieces >= 1 (boundaries are rounded to 32 environments).  env may be a handle of several families (tfem_create_mixed):
 * such a rollout steps with the _mixed calls below. */
const char* trollout_last_error(void);
int trollout_create(tfem_handle_t env, tactor_handle_t actor, int max_batch, int pieces, trollout_handle_t* out);
/* The same for n_agents (1..TROLLOUT_MAX_AGENTS) distinct actor handles, stepped together by trollout_step_agents_host;
 * n_agents = 1 is trollout_create.  Every actor must be of the env's node count and on its device (the actor ABI cannot
 * tell; host_pipeline.HostRollout checks it). */
int trollout_create_agents(tfem_handle_t env, const tactor_handle_t* actors, int n_agents, int max_batch, int pieces,
                           trollout_handle_t* out);
int trollout_destroy(trollout_handle_t h);

/* Replaces the equal pieces of trollout_create by an explicit schedule: n sizes (environments), multiples of 32 except
 * the last, adding up to at least max_batch.  A small first piece starts the downloads early -- the device->host leg is
 * the longest of the three (the child state is twice the parent's live columns) -- while later pieces stay large enough
 * to fill the GPU.  Drops the step graphs cached so far. */
int trollout_set_pieces(trollout_handle_t h, const int32_t* sizes, int n);

/* OU-noise parameters as in tactor_act.  Returns after the last piece has landed in the host buffers.  A handle of
 * several agents returns TFEM_ERR_ARG (use trollout_step_agents_host), and so does an env handle of several families
 * (use trollout_step_host_mixed). */
int trollout_step_host(trollout_handle_t h, int B, const trollout_io* io, float mu, float theta, float sigma,
                       uint64_t seed);

/* Every agent of the handle acts on the same parent and steps its own child: per piece the parent goes up once, then
 * on the compute stream agent k acts on it and its env-step reads it, and child k's download starts as soon as child k
 * is done.  mu, theta, sigma, seed: one entry per agent.  Child k is bit for bit what trollout_step_host on a handle of
 * actor k alone gives on the same parent with coin k and agent k's noise parameters (state tuple, move range, point,
 * status, clipped actions; OU noise included: every actor draws the call indices a single-agent step would). */
int trollout_step_agents_host(trollout_handle_t h, int B, const trollout_agents_io* io, const float* mu,
                              const float* theta, const float* sigma, const uint64_t* seed);

/* The two steps above over a mixed-family batch (tfem_step_mixed): family is a HOST array [B] of uint8 indices into
 * the env handle's families, 16-byte aligned (TFEM_ERR_ALIGN otherwise; pinned for overlap and for the graph).  It goes
 * up with the parent; nothing about it comes down, because every child has its parent's families.  Environment b of
 * every child is bit for bit what the plain call gives on a rollout over a handle of family family[b] alone, with the
 * same pieces.  A captured step reads the ids when it is replayed, so the caller may rewrite them in the same buffer
 * between steps.  An id >= the handle's family count sets TFEM_STATUS_BAD_FAMILY in that environment's status; the
 * child's other host outputs for that environment are then unspecified (they carry whatever the rollout's device
 * buffers held), and every other environment is unaffected.  An env handle made by tfem_create returns TFEM_ERR_ARG.
 * A handle of one family made by tfem_create_mixed may be stepped by both kinds of call. */
int trollout_step_host_mixed(trollout_handle_t h, int B, const uint8_t* family, const trollout_io* io, float mu,
                             float theta, float sigma, uint64_t seed);
int trollout_step_agents_host_mixed(trollout_handle_t h, int B, const uint8_t* family, const trollout_agents_io* io,
                                    const float* mu, const float* theta, const float* sigma, const uint64_t* seed);

/* bytes moved per environment and step: host->device, device->host (for P Pareto rows); compact_columns != 0: the
 * parent tables travel as node_y / element_section and the child state carries them too.  A handle of several agents
 * counts the parent once up and every child down; an env handle of several families adds the parent's family id (1 byte)
 * up. */
int trollout_bytes_per_env(trollout_handle_t h, int P, int compact_columns, size_t* h2d, size_t* d2h);

/* Drops the CUDA graphs cached for the host buffers seen so far.  A cached graph replays copies against the raw host
 * addresses it was captured with: call this before freeing (or un-pinning) buffers that were passed to
 * trollout_step_host, or keep them alive and pinned for the lifetime of the handle. */
int trollout_forget_buffers(trollout_handle_t h);

#ifdef __cplusplus
}
#endif
#endif /* TROLLOUT_H_ */
