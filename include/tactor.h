/* tactor.h -- C ABI of the batched node-agent GCN actor forward pass (libtfem.so).
 *
 * Replaces, for B environments at once, what the reference does one environment at a time:
 *   multimodes_actor.call  (train/code/truss2D_RL.py:75-127)   13 GCNConv layers, hidden 200
 *   multimodals_OneAgent.act (truss2D_RL.py:328-354)            forward + Ornstein-Uhlenbeck noise
 *
 * GCNConv (spektral 1.2.0, use_bias=True, no activation): out = A . (X . W) + b, followed by ReLU /
 * sigmoid in the caller.  All device buffers are caller-owned, contiguous, 16-byte aligned float32.
 * Return value 0 = ok, < 0 = error (tactor_last_error(); same codes as tfem.h).
 */
#ifndef TACTOR_H_
#define TACTOR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TACTOR_HIDDEN 200
#define TACTOR_NLAYERS 13

typedef struct tactor_handle_s* tactor_handle_t;

/* Layer order = the checkpoint's variable names (model/2000pickle_base/AgentK_Actor_pickle.index):
 * gcn_l1_1, l1_2, l1_3 [13,200]; l1_4 [4,200]; l2_1..l2_5, l3_1, l3_2 [200,200]; l4_1 [200,2];
 * l4_2 [200,3].  kernel[i] is row-major [in,out] HOST float32, bias[i] HOST float32 [out]. */
typedef struct tactor_weights {
  const float* kernel[TACTOR_NLAYERS];
  const float* bias[TACTOR_NLAYERS];
} tactor_weights;

/* Inputs of multimodes_actor.call for B environments (device pointers). */
typedef struct tactor_inputs {
  const float* x_n;      /* [B,N,13] */
  const float* A_n;      /* [N,N]    topology constant (TFEM_TAB_A_N), shared by all environments */
  const float* A_s;      /* [B,N,N] */
  const float* A_n_ts;   /* [B,N,N] */
  const float* A_n_cs;   /* [B,N,N] */
  const float* x_p;      /* [B,P,4]  Pareto-front graph features (truss2D_ENV.py:22-41) */
  const float* A_p;      /* [B,P,P] */
  const int32_t* n_pf;   /* [B] valid Pareto rows per environment (<= P); NULL = all P rows */
  int32_t P;             /* padded Pareto-front length (1..50) */
} tactor_inputs;

const char* tactor_last_error(void);

/* nodes = N = 2 num_x: any even count 6..32 (num_x 3..16).  16 and 32 (the test/ families) run natively; a smaller count
 * (12: the 6 x 2 shapes of train/code) keeps its [B,N,...] tensors, which are padded internally to the 16-node build
 * (N <= 16) or the 32-node build (N > 16).  Other counts return TFEM_ERR_UNSUPPORTED before any device call.
 * max_batch = largest B of any later call (workspace is allocated once). */
int tactor_create(const tactor_weights* w, int nodes, int max_batch, int device, tactor_handle_t* out);
int tactor_destroy(tactor_handle_t h);

/* actor_model.set_weights / load_weights on a live handle (truss2D_RL.py:368-379, master...:795): replaces all 13
 * layers (same layout as tactor_create) after the device has finished the forwards already queued. */
int tactor_set_weights(tactor_handle_t h, const tactor_weights* w);

/* The same from DEVICE memory, on `stream` (no host round trip, no device-wide synchronisation): what a learner whose
 * parameters live on the GPU calls after every update (truss2D_RL.py:625 updates actor_model, :340 acts with it).  The
 * operand images of the tensor-core kernel (power-of-two scales, fp16 hi / lo split, core-matrix layout, mma fragment
 * image of the layer-1 kernels) are rebuilt by three small kernels; forwards queued later on the same stream see the new
 * weights, forwards of OTHER streams must be ordered by the caller. */
int tactor_set_weights_device(tactor_handle_t h, const tactor_weights* w_dev, void* stream);

/* geo [B,N,2], topo [B,N,3] = sigmoid outputs of gcn_l4_1 / gcn_l4_2 (no noise). */
int tactor_forward(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo, void* stream);

/* act(): forward + OU noise theta*(mu-x)*1e-4 + sigma*n, n ~ N(0,1) from a counter-based generator
 * keyed by (seed, call counter, element index) -- statistically, not bit-wise, the reference's
 * np.random.randn stream (truss2D_RL.py:41-48).  sigma == 0 and theta == 0 gives tactor_forward. */
int tactor_act(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo,
               float mu, float theta, float sigma, uint64_t seed, void* stream);

/* tactor_act for work that is captured once into a CUDA graph and replayed (trollout_step_host): the noise stream is
 * chosen when the kernels RUN, from device memory: seed = seed_call_dev[0], call index = seed_call_dev[1] + call_offset.
 * Does not advance the handle's call counter; tactor_reserve_calls(h, n, launches) returns the counter, advances it by n
 * calls and books `launches` replayed kernel launches, so that replayed and directly launched steps draw the same
 * noise and tactor_launch_count stays truthful. */
int tactor_act_dev(tactor_handle_t h, int B, const tactor_inputs* in, float* geo, float* topo, float mu, float theta,
                   float sigma, const uint64_t* seed_call_dev, uint32_t call_offset, void* stream);
uint64_t tactor_reserve_calls(tactor_handle_t h, uint32_t n, int64_t replayed_launches);

int64_t tactor_launch_count(tactor_handle_t h);

/* Synchronises the device and returns 0, or TFEM_ERR_CUDA if a kernel of this handle reported a
 * timed-out mbarrier wait (the waits are bounded so that a programming error cannot hang the GPU), or
 * TFEM_ERR_UNSUPPORTED if an activation left the fp16 range of the split tensor-core product (|A.X| > 65504 or a NaN
 * input; the outputs of that forward are not valid).  A reported condition is cleared. */
int tactor_status(tactor_handle_t h);

/* Hardware self-test of the one layout fact the generators of actor_pipe_kernel rely on beyond the PTX fragment tables:
 * tcgen05.st.16x128b.x2 issued at lane offsets 0 and 16 of a warp's 32-lane TMEM window writes the mma accumulator
 * fragment (lane / 4, lane % 4) to (TMEM lane, column) as documented in csrc/tactor_tc.cuh.  0 = holds on this device. */
int tactor_selftest_tmem_layout(int device);

#ifdef __cplusplus
}
#endif
#endif /* TACTOR_H_ */
