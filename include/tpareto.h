/* tpareto.h -- C ABI of the batched Pareto-front bookkeeping (libtfem.so): the step on the far side of the env-step.
 *
 * For B independent environments at once, what the reference driver does per Pareto solution with
 *   utils.simple_cull(points)                        test/00_small_bridge/code/utils.py:11-217
 *   utils.union_rectangles_fastest(front, +1, -1, ref_point)                          :463-530
 * (master_DDPG_truss2D_MO.py:263-368): feasibility cut (con1 > 1 or con2 > 1), strict two-objective dominance, the
 * front sorted by obj1, its spread statistics and its hypervolume against a moving reference point.
 * Each environment holds at most TPARETO_MAX_POINTS points (the reference keeps fronts of <= 50 and culls up to 50 + 150
 * accumulated candidates at the end of a step, master_DDPG_truss2D_MO.py:437).
 */
#ifndef TPARETO_H_
#define TPARETO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TPARETO_MAX_POINTS 256

const char* tpareto_last_error(void);

/* points    [B,P,4] float32 device: obj1, obj2, con1, con2 per point (the `point` tensors of tfem_step)
 * counts    [B] int32 device, valid points per environment, clamped to 0..P (0 or below: no point, as if none were
 *           feasible; NULL = all P)
 * ref_point host double[2] (NULL = {1, 1})
 * front_idx [B,P] int32: indices of the front members in the reference's order (obj1 ascending), -1 padded
 * front_len [B]   int32: 0 when no point is feasible (the reference raises IndexError there)
 * stats     [B,5] double: max_distance, dis_distance, p_norm_inv_cd, sum_distance, std_cd (simple_cull's tuple)
 * hv        [B]   double: union_rectangles_fastest(front, ref_point)
 * Any output may be NULL; the others are written as without it.  Runs on the current device, on `stream`.
 * Non-finite points follow the reference's comparisons: a NaN constraint is feasible (NaN > 1 is false), a NaN objective
 * is never dominated and dominates nothing, NaN tuples are never duplicates.  The list puts a NaN after every number (NumPy's
 * sort convention) in obj1 and, within equal obj1, in the obj2-descending key, then orders by index; the reference's own
 * order there is whatever Python's sort makes of inconsistent comparisons.  Statistics and hypervolume propagate NaN like
 * NumPy (max_distance of a list holding a NaN objective is NaN, not the largest number).
 * Refused (nothing written): P outside 1..TPARETO_MAX_POINTS (TFEM_ERR_ARG), points not 16-byte aligned (TFEM_ERR_ALIGN). */
int tpareto_front_hv(int B, int P, const float* points, const int32_t* counts, const double* ref_point,
                     int32_t* front_idx, int32_t* front_len, double* stats, double* hv, void* stream);

/* The same with the reference's thinning of fronts of more than MAX_FRONT members (utils.py:104-131): the first and the last
 * member (by obj1) stay, max_front - 2 of the others are taken from the list sorted by crowd distance (descending, stable)
 * and keep the order of the draw; statistics and hypervolume are those of the thinned list.  The reference draws with
 * random.sample; here the draw is an input, so the result is deterministic:
 * thin_pick [B, max_front - 2] int32 device = what random.sample(range(F - 2), max_front - 2) returned for that environment
 * (positions in the crowd-sorted list, clamped to 0..F - 3; rows of environments whose front has <= max_front members are
 * not read and may hold anything).  A NaN crowd distance sorts after every number.  The crowd distances round each product
 * as NumPy does, so exact ties (the mirrored gaps of a front symmetric in obj1 <-> obj2) stay ties and the stable order holds.
 * tpareto_front_hv (no draw) leaves larger fronts unthinned.  3 <= max_front <= 64 (the training driver's MAX_FRONT is 20,
 * the test runs' 50); outside it, or with thin_pick NULL, the call returns TFEM_ERR_ARG and writes nothing. */
int tpareto_front_hv_thin(int B, int P, const float* points, const int32_t* counts, const double* ref_point,
                          const int32_t* thin_pick, int max_front, int32_t* front_idx, int32_t* front_len, double* stats,
                          double* hv, void* stream);

/* pareto_state_data (test/00_small_bridge/code/truss2D_ENV.py:22-41) for B fronts at once, padded / cut to P_out rows the
 * way the driver does before it feeds the actor (master_DDPG_truss2D_MO.py:499-517):
 *   x_p[b][i] = (obj1_i, obj2_i, i == index[b], len_b / max_front)   for i < min(len_b, P_out), zero rows behind
 *               (max_front = the ENV module's MAX_FRONT: 50 in test/<run>/code/truss2D_ENV.py:15, 20 in train/code)
 *   A_p[b]    = D^-1/2 (chain + I) D^-1/2 of the len_b-point chain, float32 like np.matmul(D, np.matmul(A, D)), rows / columns
 *               beyond P_out cut, zero rows / columns as padding
 * points    [B,P_in,4] float32 device (obj1, obj2, ...), the `points` of tpareto_front_hv
 * front_idx [B,P_in] int32 device: member i of front b is points[b][front_idx[b][i]] (NULL: identity, points are in order)
 * front_len [B] int32 device (NULL: P_in);  index [B] int32 device: which member the state belongs to (NULL: 0)
 * x_p [B,P_out,4], A_p [B,P_out,P_out] float32 device.  1 <= P_out <= 64, 1 <= P_in <= 256.  Current device, on `stream`. */
int tpareto_state_data(int B, int P_in, int P_out, int max_front, const float* points, const int32_t* front_idx,
                       const int32_t* front_len, const int32_t* index, float* x_p, float* A_p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TPARETO_H_ */
