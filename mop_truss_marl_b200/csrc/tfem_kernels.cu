// Fused env-step kernel for sm_100a: ONE WARP PER ENVIRONMENT, several environments per CTA, every
// intermediate (stiffness band, load vector, value pool) in shared memory, one pass over HBM:
//
//   load  y / section / stale move range / actions          (coalesced, 4.1 KB small / 8.6 KB large)
//   (a5)  action decode, support pinning, round-to-cm       truss2D_ENV.py:379-431   float32 + weak scalars
//   (a6)  three constraint passes per chord column           :434-455
//   (a7)  symmetry copy (warp shuffles) + min(section)       :460-553 / :460-673
//   (a3)  move range of the new geometry                     truss2D_GEN.py:118-133
//   (a8-a12) element stiffness -> banded global K            FEM_2Dtruss.py:99-105, 284-324
//   (a13) K d = P by banded LDL^T (half-bandwidth 7)         :327-337 (reference: LAPACK dgesv)
//   (a14-a17) member forces, stress ratio, energy, reactions :341-431
//   (a19-a21) observation tensors + objective point          truss2D_ENV.py:43-196, 566-587
//   store every output tensor as out[f] = pool[map[f]] with 128-bit coalesced stores
//
// DOF layout inside the kernel: chord column c owns [bottom x, bottom y, top x, top y] = 4c..4c+3, so
// every element couples DOFs at most 7 apart: K is banded (b = 7) instead of the reference numbering's
// 17 / 33.  Restrained DOFs stay in the system as identity rows (d = 0).  The nodal 2x2 diagonal blocks
// are GATHERED in a fixed element order (no atomics): results are bit-reproducible for any batch split.
//
// Numeric contract: the transition and move range reproduce the reference's float32 / python-scalar
// mix bit-exactly (no FMA contraction: explicit __f*_rn / __d*_rn intrinsics); the FEM is float64.
#include "tfem_kernels.cuh"

#include <math_constants.h>

#include <array>
#include <utility>

namespace tfem {

namespace {

#ifndef TFEM_WARPS_PER_CTA
#define TFEM_WARPS_PER_CTA 8
#endif
constexpr int WARPS_PER_CTA = TFEM_WARPS_PER_CTA;
constexpr int BAND = 8;  // stored sub-diagonals + diagonal per column
constexpr int PADC = 8;  // zero columns appended to the band so the elimination needs no bounds checks

// ---- "typed" scalar: value + whether the reference holds it as a python scalar (weak) or np.float32 ----
struct TS {
  double v;
  bool weak;
};
__device__ __forceinline__ TS W(double v) { return TS{v, true}; }
__device__ __forceinline__ TS S(float v) { return TS{(double)v, false}; }
__device__ __forceinline__ float f32(const TS& a) { return __double2float_rn(a.v); }
__device__ __forceinline__ TS ts_add(const TS& a, const TS& b) {
  if (a.weak && b.weak) return TS{__dadd_rn(a.v, b.v), true};
  return TS{(double)__fadd_rn(f32(a), f32(b)), false};
}
__device__ __forceinline__ TS ts_sub(const TS& a, const TS& b) {
  if (a.weak && b.weak) return TS{__dsub_rn(a.v, b.v), true};
  return TS{(double)__fsub_rn(f32(a), f32(b)), false};
}
__device__ __forceinline__ TS ts_abs(const TS& a) { return TS{fabs(a.v), a.weak}; }
__device__ __forceinline__ bool ts_lt(const TS& a, const TS& b) {
  if (a.weak && b.weak) return a.v < b.v;
  return f32(a) < f32(b);
}
__device__ __forceinline__ bool ts_gt(const TS& a, const TS& b) {
  if (a.weak && b.weak) return a.v > b.v;
  return f32(a) > f32(b);
}
__device__ __forceinline__ TS ts_shfl(const TS& a, int src) {
  TS r;
  r.v = __shfl_sync(0xffffffffu, a.v, src);
  r.weak = __shfl_sync(0xffffffffu, (int)a.weak, src) != 0;
  return r;
}

// np.argmax on floats: first maximum; a NaN wins and stops the scan
__device__ __forceinline__ int argmax2(float a, float b) {
  if (a != a) return 0;
  return !(b <= a) ? 1 : 0;
}
__device__ __forceinline__ int argmax3(float a, float b, float c) {
  if (a != a) return 0;
  float mp = a;
  int idx = 0;
  if (!(b <= mp)) { mp = b; idx = 1; if (mp != mp) return idx; }
  if (!(c <= mp)) { idx = 2; }
  return idx;
}
__device__ __forceinline__ float clip01(float v) { return v > 1.f ? 1.f : (v < 0.f ? 0.f : v); }

// np.float32.__round__(2): rint(x*100)/100 in float32
__device__ __forceinline__ float round2(float v) { return __fdiv_rn(rintf(__fmul_rn(v, 100.f)), 100.f); }

// numpy float32 pairwise sum (n <= 128): executed by the whole warp, the array lives in shared memory
__device__ __forceinline__ float pairwise_sum_warp(const float* a, int n, int lane) {
  if (n < 8) {                             // numpy adds fewer than 8 values in order (N = 6 nodes: num_x = 3)
    float res = 0.f;
    for (int i = 0; i < n; ++i) res = __fadd_rn(res, a[i]);
    return res;
  }
  const int k = lane & 7;
  float r = a[k];
  const int nfull = n - (n % 8);
  for (int i = 8; i < nfull; i += 8) r = __fadd_rn(r, a[i + k]);
  float r1 = __fadd_rn(r, __shfl_xor_sync(0xffffffffu, r, 1));     // (r0+r1), (r2+r3), ...
  float r2 = __fadd_rn(r1, __shfl_xor_sync(0xffffffffu, r1, 2));   // ((r0+r1)+(r2+r3)), ...
  float lo = __shfl_sync(0xffffffffu, r2, 0), hi = __shfl_sync(0xffffffffu, r2, 4);
  float res = __fadd_rn(lo, hi);
  for (int i = nfull; i < n; ++i) res = __fadd_rn(res, a[i]);
  return res;
}

// float min/max over the warp with one REDUX each: map the bit pattern to an unsigned key that is
// monotonic over all floats (-0.0 sorts just below +0.0, which is value-equal; +NaN sorts above +inf).
__device__ __forceinline__ unsigned f32_key(float v) {
  const unsigned b = __float_as_uint(v);
  return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float f32_unkey(unsigned k) {
  return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu));
}
__device__ __forceinline__ float warp_max_f32(float v) { return f32_unkey(__reduce_max_sync(0xffffffffu, f32_key(v))); }
__device__ __forceinline__ float warp_min_f32(float v) { return f32_unkey(__reduce_min_sync(0xffffffffu, f32_key(v))); }
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float norm_f32(float v, float mn, float mx) {
  return __fdiv_rn(__fsub_rn(v, mn), __fadd_rn(__fsub_rn(mx, mn), 1e-6f));
}

// 1/a for the 4*NX sequential pivots of the factorisation: MUFU.RCP64H seed (relative error ~2^-20) and two Newton steps
// (-> 2^-80, i.e. full double precision, at worst 1 ulp from the correctly rounded quotient).  The compiler's own IEEE
// division is a 20-instruction sequence with a dependent chain twice as long and a slow-path call; pivots here are normal
// positive numbers, and a zero / negative / non-finite pivot still yields a value the SPD check flags.
__device__ __forceinline__ double pivot_rcp(double a) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(a));
  double e = fma(-a, x, 1.0);
  x = fma(x, e, x);
  e = fma(-a, x, 1.0);
  return fma(x, e, x);
}

// development ablations (profiles/README.md, round 2: what the solve costs inside the step kernel); results are wrong on purpose
#ifdef TFEM_ABLATE_FACTOR
#define ABL_F && j < 1
#else
#define ABL_F
#endif
#ifdef TFEM_ABLATE_BACKSUB
#define ABL_B && j > NI - 2
#else
#define ABL_B
#endif
template <int NX>
struct Dims {
  static constexpr int N = 2 * NX;
  static constexpr int E = 5 * NX - 4;
  static constexpr int NI = 4 * NX;             // internal DOFs (restrained ones kept as identity rows)
  static constexpr int EPL = (E + 31) / 32;     // element passes per lane
  static constexpr int POOL = 2 + 12 * N + 13 * N + 10 * E;
  static constexpr int POOL_PAD = (POOL + 3) & ~3;
  static constexpr int WARP_BYTES = (NI + PADC) * BAND * 8 + (NI + PADC) * 8 + NI * 8 + POOL_PAD * 4;
};

__host__ __device__ constexpr int align16(int v) { return (v + 15) & ~15; }

#ifndef TFEM_MINB_SMALL
#define TFEM_MINB_SMALL 2
#endif
#ifndef TFEM_MINB_LARGE
#define TFEM_MINB_LARGE 2
#endif
// GM = false: env-step / reset / solve-only (args.mode); GM = true: the gene-vector objective (MODE_GENES) -- a separate
// instantiation so that the env-step keeps its register allocation.
// MF = true: mixed-family env-step / reset (tfem_step_mixed, tfem_reset_mixed).  The CTA stages args.n_families tables of
// one topology and ONE copy of the output maps (they depend on N, E and conn only); each environment reads its tables
// through fam = staged + family[b].  Values read before the environment loop are topology and come from table 0.
template <int NX, bool GM, bool MF>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, (NX <= 8) ? TFEM_MINB_SMALL : TFEM_MINB_LARGE)
tfem_step_kernel(const StepArgs args) {
  static_assert(!(GM && MF), "the gene-vector objective has no mixed-family form");
  using D = Dims<NX>;
  constexpr int N = D::N, E = D::E, NI = D::NI, EPL = D::EPL;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  FamilyTables* const fams = reinterpret_cast<FamilyTables*>(smem_raw);
  FamilyTables* fam = fams;
  const int tab_bytes = MF ? args.n_families * (int)sizeof(FamilyTables) : (int)sizeof(FamilyTables);
  uint16_t* maps = reinterpret_cast<uint16_t*>(smem_raw + align16(tab_bytes));

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int mode = GM ? (int)MODE_GENES : args.mode;
  const int warps_total = gridDim.x * WARPS_PER_CTA;
  const int node = lane % N;                 // lanes >= N mirror a node so warp reductions stay exact
  // ---- per-env inputs are fetched one environment ahead (the first batch overlaps the table staging) ----
  float in_y = 0.f, in_at0 = 0.f, in_at1 = 0.f, in_at2 = 0.f, in_sec[EPL];
  float2 in_mr = make_float2(0.f, 0.f), in_ag = make_float2(0.f, 0.f);
  int in_coin = 0, in_fam = 0;
  // the two live columns of the parent tables: compact arrays when the caller has them, else column 1 / column 0
  const float* const col_y = args.in.set_node_y ? args.in.set_node_y : args.in.set_node + 1;
  const float* const col_sec = args.in.set_element_section ? args.in.set_element_section : args.in.set_element;
  const int col_y_stride = args.in.set_node_y ? 1 : 12, col_sec_stride = args.in.set_element_section ? 1 : 21;
  auto fetch_inputs = [&](int b) {
    if constexpr (MF) {
      if (b < args.B) in_fam = args.family[b];
    }
    if (mode != MODE_STEP || b >= args.B) return;
    in_y = col_y[((size_t)b * N + node) * col_y_stride];
    in_mr = reinterpret_cast<const float2*>(args.in.move_range)[(size_t)b * N + node];
    in_ag = reinterpret_cast<const float2*>(args.in.a_geo)[(size_t)b * N + node];
    const float* atp = args.in.a_topo + ((size_t)b * N + node) * 3;
    in_at0 = atp[0]; in_at1 = atp[1]; in_at2 = atp[2];
#pragma unroll
    for (int p = 0; p < EPL; ++p) {
      const int e = lane + 32 * p;
      in_sec[p] = (e < E) ? col_sec[((size_t)b * E + e) * col_sec_stride] : 0.f;
    }
    in_coin = args.in.coin ? (int)args.in.coin[b] : 0;
  };
  {  // stage the family tables and output maps once per CTA (L2-resident, 8..15 KB)
    const uint4* src = reinterpret_cast<const uint4*>(args.fam);
    uint4* dst = reinterpret_cast<uint4*>(fam);
    for (int i = tid; i < tab_bytes / 16; i += blockDim.x) dst[i] = src[i];
    const uint4* msrc = reinterpret_cast<const uint4*>(args.maps);
    uint4* mdst = reinterpret_cast<uint4*>(maps);
    for (int i = tid; i < args.map_entries / 8; i += blockDim.x) mdst[i] = msrc[i];
  }
  // programmatic dependent launch: the kernel may have been started while its predecessor in the stream (the actor, whose
  // actions it reads) is still running; everything above only touches the handle's constant tables
  asm volatile("griddepcontrol.wait;" ::: "memory");
  fetch_inputs(blockIdx.x * WARPS_PER_CTA + warp);
  __syncthreads();
  unsigned char* wbase = smem_raw + align16(tab_bytes) + align16(args.map_entries * 2) + warp * D::WARP_BYTES;
  double* Kb = reinterpret_cast<double*>(wbase);            // [NI][BAND]: Kb[j*8+k] = K[j+k][j]
  double* z = Kb + (NI + PADC) * BAND;                      // [NI + PADC] rhs -> solution
  double* dinv = z + NI + PADC;                             // [NI] 1 / pivot
  float* pool = reinterpret_cast<float*>(dinv + NI);        // value pool
  const PoolLayout pl{N, E};
  float* dyn = pool + pl.dyn_base();
  // scratch that aliases the (not yet written) dynamic pool during transition / assembly
  double* g = reinterpret_cast<double*>(dyn);               // [E][3] element stiffness terms (needs 16B align)
  float* at_s = dyn;                                        // [N][3] clipped a_topo (before g is written)
  int* sec_s = reinterpret_cast<int*>(dyn + 3 * N);         // [E] sections after the action
  if constexpr (!MF)                        // mixed launches copy it per family, in the environment loop
    for (int i = lane; i < pl.dyn_base(); i += 32) pool[i] = fam->pool_const[i];
  __syncwarp();
  int pool_fam = -1;                         // MF: the family whose constant columns the pool holds

  // trailing-update role of this lane: (a, b), 1 <= b <= a <= 7, for lanes 0..27
  int ta = 0, tb = 0;
  {
    int t = 0;
    for (int b = 1; b <= 7; ++b)
      for (int a = b; a <= 7; ++a) { if (t == lane) { ta = a; tb = b; } ++t; }
  }
  const bool node_lane = lane < N;
  const int colc = lane % NX;                // chord column handled in the constraint passes
  const int bi = 4 * (node % NX) + 2 * (node / NX);
  const unsigned res_bits = fam->res[node];
  const bool is_top = fam->top[node] != 0;

  for (int b = blockIdx.x * WARPS_PER_CTA + warp; b < args.B; b += warps_total) {
    if constexpr (MF) {
      const int f = in_fam;
      if (f >= args.n_families) {            // no table is read and nothing but the status is written
        fetch_inputs(b + warps_total);
        if (lane == 0 && args.out.status) args.out.status[b] = TFEM_STATUS_BAD_FAMILY;
        continue;
      }
      fam = fams + f;
      if (f != pool_fam) {                   // normalised x / support / load columns differ between families
        for (int i = lane; i < pl.dyn_base(); i += 32) pool[i] = fam->pool_const[i];
        __syncwarp();
        pool_fam = f;
      }
    }
    int status = 0;
    TS y, yp;                                // this node's height and its vertical pair's
    int sec[EPL];
    // ======================================= geometry =======================================
    if constexpr (GM) {
      // gene-vector decode: read_genes of the MOEA/D benchmark zips (<family>/truss2D_GEN.py:126-195); all float64
      const double* gp = args.genes + (size_t)b * (N + E);
      const double dmin = fam->d_min, ymin = fam->y_min;
      const bool roof = fam->truss_type == TFEM_ROOF;
      const int pr = fam->pair[node];
      double yy = fam->y0[node];
      const double hgt = __dmul_rn(gp[node], args.max_height);
      if (roof ? !(res_bits & 2) : is_top) yy = (dmin > hgt) ? dmin : hgt;        // max([h, d_min])
      if (roof && node == N - 1) yy = 0.0;                                        // the loop's for-else (:141-142)
      const double ytop = __shfl_sync(0xffffffffu, yy, pr);
      if (!is_top && (__dsub_rn(ytop, dmin) < yy)) yy = __dsub_rn(ytop, dmin);    // fix the vertical pair (:155-159)
      const int low = (!is_top && yy < ymin) ? 1 : 0;                             // below y_min (:162-167)
      const int pair_low = __shfl_sync(0xffffffffu, low, pr);
      if (low) yy = ymin;
      if (is_top && pair_low) yy = dmin;
      yy = __shfl_sync(0xffffffffu, yy, fam->sym_src[fam->symmetry == TFEM_SYM_SMALL ? 0 : 1][node]);
      y = W(yy);
      yp = W(__shfl_sync(0xffffffffu, yy, pr));
#pragma unroll
      for (int p = 0; p < EPL; ++p) {
        const int e = lane + 32 * p;
        sec[p] = 0;
        if (e < E) {
          sec[p] = min(max(__double2int_rn(__dmul_rn(gp[N + e], 4.0)), 0), TFEM_NSEC - 1);   // min([4, round(g*4)])
          sec_s[e] = sec[p];
        }
      }
      __syncwarp();
#pragma unroll
      for (int p = 0; p < EPL; ++p) {
        const int e = lane + 32 * p;
        if (e < E) {
          const int partner = fam->sym_elem[e];
          if (partner > e) sec[p] = sec_s[partner];                               // low index <- its mirror
          if (args.sec_out) args.sec_out[(size_t)b * E + e] = sec[p];
        }
      }
      __syncwarp();
    } else if (mode == MODE_STEP) {
      const float y32 = in_y;
      const float2 mr = in_mr;
      float2 ag = in_ag;
      float* atp = args.in.a_topo + ((size_t)b * N + node) * 3;
      float at0 = in_at0, at1 = in_at1, at2 = in_at2;
      const int coin = in_coin != 0;
      ag.x = clip01(ag.x); ag.y = clip01(ag.y);
      at0 = clip01(at0); at1 = clip01(at1); at2 = clip01(at2);
      if (node_lane) {                       // the reference clips the caller's arrays in place
        reinterpret_cast<float2*>(args.in.a_geo)[(size_t)b * N + node] = ag;
        atp[0] = at0; atp[1] = at1; atp[2] = at2;
        at_s[node * 3 + 0] = at0; at_s[node * 3 + 1] = at1; at_s[node * 3 + 2] = at2;
      }
#pragma unroll
      for (int p = 0; p < EPL; ++p) {
        const int e = lane + 32 * p;
        sec[p] = (e < E) ? __float2int_rz(in_sec[p]) : 0;
      }
      fetch_inputs(b + warps_total);          // next environment of this warp (if any)
      // ---- action decode (truss2D_ENV.py:401-416) ----
      y = S(y32);
      {
        const int adj = argmax2(ag.x, ag.y);
        const float a = adj == 0 ? ag.x : ag.y;
        const float range = adj == 0 ? mr.x : mr.y;
        // min([1, a]) * range * 0.25 : float32 products (a python 1 leaves the range unchanged)
        const float step = __fmul_rn((a < 1.f) ? __fmul_rn(a, range) : range, 0.25f);
        y = S(adj == 0 ? __fadd_rn(y32, step) : __fsub_rn(y32, step));
      }
      if (res_bits & 2) y = W(0.0);
      if (!y.weak) y = S(round2((float)y.v));
      __syncwarp();
      // ---- section change from the two end nodes' topology actions (:419-431) ----
#pragma unroll
      for (int p = 0; p < EPL; ++p) {
        const int e = lane + 32 * p;
        if (e < E) {
          const int n0 = fam->conn[e][0], n1 = fam->conn[e][1];
          const float p0 = __fadd_rn(at_s[n0 * 3 + 0], at_s[n1 * 3 + 0]);
          const float p1 = __fadd_rn(at_s[n0 * 3 + 1], at_s[n1 * 3 + 1]);
          const float p2 = __fadd_rn(at_s[n0 * 3 + 2], at_s[n1 * 3 + 2]);
          const int am = argmax3(p0, p1, p2);
          if (am == 0) sec[p] = max(0, sec[p] - 1);
          else if (am == 1) sec[p] = min(TFEM_NSEC - 1, sec[p] + 1);
          sec_s[e] = sec[p];
        }
      }
      // ---- constraint passes, one chord column per lane (:434-455) ----
      TS yb = ts_shfl(y, colc), yt = ts_shfl(y, colc + NX);
      const TS YMIN = W(fam->y_min), YMAX = W(fam->y_max), DMIN = W(fam->d_min);
      if (ts_lt(yb, YMIN)) yb = YMIN;
      if (ts_lt(yt, YMIN)) { yt = DMIN; yb = YMIN; }
      if (ts_gt(yb, YMAX)) { yb = W(fam->ymax_minus_dmin); yt = YMAX; }
      if (ts_gt(yt, YMAX)) yt = YMAX;
      if (ts_lt(ts_abs(ts_sub(yt, yb)), DMIN)) yt = ts_add(yb, DMIN);
      // ---- symmetry copy (:460-502 small / :460-557 large) ----
      const int srcb = fam->sym_src[coin][colc], srct = fam->sym_src[coin][colc + NX] - NX;
      yb = ts_shfl(yb, srcb);
      yt = ts_shfl(yt, srct);
      y = (node < NX) ? yb : yt;
      yp = (node < NX) ? yt : yb;
      __syncwarp();
      // ---- symmetric elements take the smaller section (:505-553 / :560-673) ----
#pragma unroll
      for (int p = 0; p < EPL; ++p) {
        const int e = lane + 32 * p;
        if (e < E) sec[p] = min(sec[p], sec_s[fam->sym_elem[e]]);
      }
      __syncwarp();
    } else if (MF || mode == MODE_RESET) {
      if constexpr (MF) fetch_inputs(b + warps_total);
      y = W(fam->y0[node]);
      yp = W(fam->y0[fam->pair[node]]);
#pragma unroll
      for (int p = 0; p < EPL; ++p) sec[p] = TFEM_NSEC - 1;
    } else {
      y = W(args.so_y[(size_t)b * N + node]);
      yp = W(args.so_y[(size_t)b * N + fam->pair[node]]);
#pragma unroll
      for (int p = 0; p < EPL; ++p) {
        const int e = lane + 32 * p;
        sec[p] = (e < E) ? min(max(args.so_sec[(size_t)b * E + e], 0), TFEM_NSEC - 1) : 0;
      }
    }

    // ======================================= move range (truss2D_GEN.py:118-133) =======================
    TS up = W(0.0), down = W(0.0);
    if (is_top) {
      up = ts_abs(ts_sub(W(fam->y_max), y));
      down = ts_abs(ts_sub(ts_sub(y, yp), W(fam->d_min)));
    } else if (fam->truss_type == TFEM_ROOF) {
      up = ts_abs(ts_sub(ts_sub(yp, y), W(fam->d_min)));
      down = ts_abs(ts_sub(y, W(fam->y_min)));
    }
    const float up32 = f32(up), down32 = f32(down);
    if (node_lane) {
      if (args.out.y) args.out.y[(size_t)b * N + node] = y.v;
      if (args.out.y_weak) args.out.y_weak[(size_t)b * N + node] = y.weak ? 1 : 0;
    }
    if (node_lane) {
      if (mode == MODE_STEP) reinterpret_cast<float2*>(args.in.move_range)[(size_t)b * N + node] = make_float2(up32, down32);
      else if (mode == MODE_RESET && args.reset_move_range)
        reinterpret_cast<float2*>(args.reset_move_range)[(size_t)b * N + node] = make_float2(up32, down32);
    }

    // ======================================= assembly ========================================
    // zero the band, publish float(y) for the element lanes
    for (int i = lane; i < (NI + PADC) * BAND / 2; i += 32) reinterpret_cast<double2*>(Kb)[i] = make_double2(0.0, 0.0);
    if (lane < PADC) z[NI + lane] = 0.0;
    if (node_lane) { z[bi] = y.v; }          // z doubles as y64 storage until the rhs is written
    __syncwarp();
    double eL[EPL], ec[EPL], es[EPL], ek[EPL];
#pragma unroll
    for (int p = 0; p < EPL; ++p) {
      const int e = lane + 32 * p;
      eL[p] = 1.0; ec[p] = 0.0; es[p] = 0.0; ek[p] = 0.0;
      if (e < E) {
        const int n0 = fam->conn[e][0], n1 = fam->conn[e][1];
        const int b0 = 4 * (n0 % NX) + 2 * (n0 / NX), b1 = 4 * (n1 % NX) + 2 * (n1 / NX);
        const double dx = fam->x[n1] - fam->x[n0];
        const double dy = z[b1] - z[b0];
        const double L = sqrt(dx * dx + dy * dy);          // Element.gen_length / gen_global_k
        const double c = dx / L, s = dy / L;
        const double k = fam->young * fam->sec_area[sec[p]] / L;
        eL[p] = L; ec[p] = c; es[p] = s; ek[p] = k;
        const double gxx = k * c * c, gxy = k * c * s, gyy = k * s * s;
        g[e * 3 + 0] = gxx; g[e * 3 + 1] = gxy; g[e * 3 + 2] = gyy;
        // off-diagonal 2x2 block -(g) between the two nodes, stored below the diagonal
        const int lo = min(b0, b1), hi = max(b0, b1);
        const unsigned rlo = fam->res[b0 < b1 ? n0 : n1], rhi = fam->res[b0 < b1 ? n1 : n0];
        const double blk[2][2] = {{gxx, gxy}, {gxy, gyy}};
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            const bool fixed = ((rhi >> a) & 1) || ((rlo >> q) & 1);
            Kb[(lo + q) * BAND + (hi + a - lo - q)] = fixed ? 0.0 : -blk[a][q];
          }
      }
    }
    __syncwarp();
    if (node_lane) {
      double sxx = 0.0, sxy = 0.0, syy = 0.0;
#pragma unroll
      for (int k = 0; k < MAXADJ - 1; ++k) {
        const int e = fam->adj[node][k];
        if (e >= 0) { sxx += g[e * 3 + 0]; sxy += g[e * 3 + 1]; syy += g[e * 3 + 2]; }
      }
      const bool rx = res_bits & 1, ry = res_bits & 2;
      Kb[bi * BAND + 0] = rx ? 1.0 : sxx;
      Kb[bi * BAND + 1] = (rx || ry) ? 0.0 : sxy;
      Kb[(bi + 1) * BAND + 0] = ry ? 1.0 : syy;
      z[bi] = 0.0;
      z[bi + 1] = ry ? 0.0 : fam->fy[node];
    }
    __syncwarp();

    // ======================================= banded LDL^T + forward substitution ==========================
    // Column j: every lane forms 1/pivot; lane (a,b) updates K[j+a][j+b] -= L[j+a][j] * K[j+b][j]; the rhs
    // rows ride along (lanes 28..31 take a = 1..4, lanes 0..2 also take a = 5..7).  The zero padding makes
    // every access in-bounds, and keeping 1/pivot in its own array leaves ONE warp barrier per column.
    {
      const int za = (lane >= 28) ? lane - 27 : (lane < 3 ? lane + 5 : 0);
      const int tgt_off = tb * BAND + (ta - tb);
      double* col = Kb;
#pragma unroll 4
      for (int j = 0; j < NI ABL_F; ++j, col += BAND) {
        const double inv = pivot_rcp(col[0]);
        const double la = col[ta] * inv;                      // L[j+a][j]
        const double upd = fma(-la, col[tb], col[tgt_off]);
        double zl = 0.0;
        if (za) zl = fma(-(col[za] * inv), z[j], z[j + za]);
        if (lane < 28) col[tgt_off] = upd;
        if (za) z[j + za] = zl;
        dinv[j] = inv;
        __syncwarp();
      }
    }
    // SPD check, scale the stored columns to L, apply D^-1
    for (int i = lane; i < NI; i += 32) {
      const double iv = dinv[i];
      if (!(iv > 0.0) || !(iv < CUDART_INF)) status |= TFEM_STATUS_NOT_SPD;
      z[i] *= iv;
    }
    for (int i = lane; i < NI * BAND; i += 32)
      if (i % BAND) Kb[i] *= dinv[i / BAND];
    __syncwarp();
    // back substitution L^T x = w, column oriented
    for (int j = NI - 1; j > 0 ABL_B; --j) {
      const double xj = z[j];
      const int a = lane + 1;
      if (a <= 7 && j - a >= 0) z[j - a] = fma(-Kb[(j - a) * BAND + a], xj, z[j - a]);
      __syncwarp();
    }

    // ======================================= member forces =====================================
    const double ddx = z[bi], ddy = z[bi + 1];               // this node's displacement
    if (!(isfinite(ddx) && isfinite(ddy))) status |= TFEM_STATUS_NONFINITE;
    double q0[EPL], ratio[EPL];
    double u_acc = 0.0, v64 = 0.0, c1 = 0.0;
    float allv[EPL];
#pragma unroll
    for (int p = 0; p < EPL; ++p) {
      const int e = lane + 32 * p;
      q0[p] = 0.0; ratio[p] = 0.0; allv[p] = 0.f;
      if (e < E) {
        const int n0 = fam->conn[e][0], n1 = fam->conn[e][1];
        const int b0 = 4 * (n0 % NX) + 2 * (n0 / NX), b1 = 4 * (n1 % NX) + 2 * (n1 / NX);
        const double u0 = ec[p] * z[b0] + es[p] * z[b0 + 1];   // u = T v          (gen_u)
        const double u2 = ec[p] * z[b1] + es[p] * z[b1 + 1];
        const double q = ek[p] * u0 + (-ek[p]) * u2;           // q = k_local u    (gen_q), + = compression
        const double A = fam->sec_area[sec[p]];
        q0[p] = q;
        ratio[p] = fabs(q / A) / fam->allow;                   // gen_yield
        u_acc += 0.5 * q * (u0 - u2);                          // element strain energy
        v64 += A * eL[p];
        allv[p] = __double2float_rn(A * eL[p]);
        c1 = fmax(c1, ratio[p]);
      }
    }
    status = __reduce_or_sync(0xffffffffu, status);
    const double U = warp_sum(u_acc);
    __syncwarp();                                             // everyone is done reading z and Kb
    if (args.out.reactions) {
      // f = T^T q at both ends (gen_f); restrained DOFs sum them (gen_r)
      double* fxy = Kb;                                       // [E][2], band is dead now
#pragma unroll
      for (int p = 0; p < EPL; ++p) {
        const int e = lane + 32 * p;
        if (e < E) { fxy[2 * e] = ec[p] * q0[p]; fxy[2 * e + 1] = es[p] * q0[p]; }
      }
      __syncwarp();
      if (node_lane && res_bits) {
        double rxs = 0.0, rys = 0.0;
        for (int k = 0; k < MAXADJ - 1; ++k) {
          const int e = fam->adj[node][k];
          if (e >= 0) {
            const double sg = (fam->conn[e][0] == node) ? 1.0 : -1.0;
            rxs += sg * fxy[2 * e]; rys += sg * fxy[2 * e + 1];
          }
        }
        if (res_bits & 1) args.out.reactions[(size_t)b * fam->nres + fam->react_slot[node][0]] = rxs;
        if (res_bits & 2) args.out.reactions[(size_t)b * fam->nres + fam->react_slot[node][1]] = rys;
      }
    }
    // ---- FP64 outputs ----
    if (node_lane && args.out.d) {
      if (!(res_bits & 1)) args.out.d[(size_t)b * fam->ndof + fam->dof[node][0] - 1] = ddx;
      if (!(res_bits & 2)) args.out.d[(size_t)b * fam->ndof + fam->dof[node][1] - 1] = ddy;
    }
#pragma unroll
    for (int p = 0; p < EPL; ++p) {
      const int e = lane + 32 * p;
      if (e < E) {
        if (args.out.axial) args.out.axial[(size_t)b * E + e] = q0[p];
        if (args.out.ratio) args.out.ratio[(size_t)b * E + e] = ratio[p];
      }
    }
    if (lane == 0) {
      if (args.out.U) args.out.U[b] = U;
      if (args.out.status) args.out.status[b] = status;
    }
    if (!GM && mode == MODE_SOLVE_ONLY) { __syncwarp(); continue; }

    // ======================================= observations ======================================
    // node features (state_data / state_data_not_norm, truss2D_ENV.py:65-82, 137-149)
    if constexpr (!GM) {
    const float y32o = f32(y);
    float x9 = 0.f;
    if (is_top) {
      const TS den = ts_add(y, W(1e-6));
      x9 = den.weak ? __double2float_rn(__ddiv_rn(fam->target[node], den.v))
                    : __fdiv_rn(__double2float_rn(fam->target[node]), (float)den.v);
    }
    const float dy32 = __double2float_rn(fabs(ddy));
    const float r = __fdiv_rn(dy32, fam->maxdef32);
    const float x11 = (r > 1.f) ? 1.f : __fmul_rn(r, 0.5f);
    const float x12 = (r > 1.f) ? 1.f : 0.f;
    const float raw11 = (r >= 1.f) ? 1.f : 0.f;
    {
      const float cols[7] = {y32o, up32, down32, x9, dy32, x11, x12};
#pragma unroll
      for (int k = 0; k < 7; ++k) {
        const float mn = warp_min_f32(cols[k]), mx = warp_max_f32(cols[k]);
        if (node_lane) dyn[k * N + node] = norm_f32(cols[k], mn, mx);
      }
      if (node_lane) {
        if (args.out.node_y) args.out.node_y[(size_t)b * N + node] = y32o;
        float* rawd = dyn + 7 * N;
        rawd[0 * N + node] = y32o; rawd[1 * N + node] = up32; rawd[2 * N + node] = down32;
        rawd[3 * N + node] = x9; rawd[4 * N + node] = dy32; rawd[5 * N + node] = raw11;
      }
    }
    }  // !GM
    // objectives (truss2D_ENV.py:566-587)
    float* sum_s = reinterpret_cast<float*>(z);               // z is dead: scratch for the pairwise sums
#pragma unroll
    for (int p = 0; p < EPL; ++p) { const int e = lane + 32 * p; if (e < E) sum_s[e] = allv[p]; }
    __syncwarp();
    const float obj1 = pairwise_sum_warp(sum_s, E, lane);
    __syncwarp();
    float dt32 = 0.f;
    double dt64 = 0.0;
    if (is_top) {
      const TS dt = ts_abs(ts_sub(W(fam->target[node]), y));
      dt32 = f32(dt);
      dt64 = fabs(fam->target[node] - y.v);
    }
    if (node_lane) sum_s[node] = dt32;
    __syncwarp();
    const float obj2 = pairwise_sum_warp(sum_s, N, lane);
    float con1 = 0.f;
#pragma unroll
    for (int p = 0; p < EPL; ++p) con1 = fmaxf(con1, __double2float_rn(ratio[p]));
    con1 = warp_max_f32(con1);
    const float alld = is_top ? 0.f : fabsf(__double2float_rn(__ddiv_rn(ddy, fam->max_def)));
    const float con2 = warp_max_f32(alld);
    if (lane == 0 && args.out.point) {
      reinterpret_cast<float4*>(args.out.point)[b] =
          make_float4(__fdiv_rn(obj1, args.int_obj1 > 0.f ? args.int_obj1 : fam->int_obj1),
                      __fdiv_rn(obj2, args.int_obj2 > 0.f ? args.int_obj2 : fam->int_obj2), con1, con2);
    }
    if (args.out.point64) {
      const double s1 = warp_sum(v64);
      const double s2 = warp_sum(node_lane ? dt64 : 0.0);
      const double m1 = warp_max(c1);
      const double m2 = warp_max((node_lane && !is_top) ? fabs(ddy) / fam->max_def : 0.0);
      if (lane == 0) {
        double* p64 = args.out.point64 + (size_t)b * 4;
        p64[0] = s1; p64[1] = s2; p64[2] = m1; p64[3] = m2;
      }
    }
    if (GM) { __syncwarp(); continue; }
    // element columns of the pool (state_data :84-100, state_data_not_norm :151-172)
    __syncwarp();
#pragma unroll
    for (int p = 0; p < EPL; ++p) {
      const int e = lane + 32 * p;
      if (e < E) {
        float* el = dyn + 13 * N;
        const bool comp = q0[p] > 0.0;
        const double py = ratio[p];
        const float val = __double2float_rn(fmin(py, 1.0) * (py > 1.0 ? 1.0 : 0.5));
        el[EL_SEC * E + e] = (float)sec[p];
        if (args.out.element_section) args.out.element_section[(size_t)b * E + e] = (float)sec[p];
        el[EL_A * E + e] = fam->sec_area32[sec[p]];
        el[EL_L * E + e] = __double2float_rn(eL[p]);
        el[EL_TENS * E + e] = comp ? 0.f : 1.f;
        el[EL_COMP * E + e] = comp ? 1.f : 0.f;
        el[EL_Q * E + e] = __double2float_rn(q0[p]);
        el[EL_VIOL * E + e] = (py > 1.0) ? 1.f : 0.f;
        el[EL_AS * E + e] = fam->sec_as32[sec[p]];
        el[EL_TS * E + e] = comp ? 0.f : val;
        el[EL_CS * E + e] = comp ? val : 0.f;
      }
    }
    __syncwarp();
    // ---- stream the tensors out: out[f] = pool[map[f]], one float4 per lane per iteration ----
    auto emit = [&](float* dst, int map_off, int count) {
      if (!dst) return;
      float4* o = reinterpret_cast<float4*>(dst + (size_t)b * count);
      const uint2* m = reinterpret_cast<const uint2*>(maps + map_off);
      if (count % 4 == 0) {
        for (int q = lane; q < count / 4; q += 32) {
          const uint2 mm = m[q];
          o[q] = make_float4(pool[mm.x & 0xffffu], pool[mm.x >> 16], pool[mm.y & 0xffffu], pool[mm.y >> 16]);
        }
      } else if (count % 2 == 0) {
        // an environment's slice of this tensor is not a multiple of 16 bytes (nN_x_e of the 6 x 2 shapes: 26 x 21 floats,
        // x_n of an odd num_x: 26 num_x floats), so neither are the slice addresses: 64-bit stores
        float2* o2 = reinterpret_cast<float2*>(dst + (size_t)b * count);
        const uint32_t* m1 = reinterpret_cast<const uint32_t*>(maps + map_off);
        for (int q = lane; q < count / 2; q += 32) {
          const uint32_t mm = m1[q];
          o2[q] = make_float2(pool[mm & 0xffffu], pool[mm >> 16]);
        }
      } else {
        // nN_x_e of an odd num_x (21 E floats, E = 5 num_x - 4 odd): 32-bit stores
        float* o1 = dst + (size_t)b * count;
        for (int q = lane; q < count; q += 32) o1[q] = pool[maps[map_off + q]];
      }
    };
    // The path is chosen from the per-environment count, a compile-time constant: 128-bit stores need a count = 0 mod 4,
    // 64-bit stores a count = 0 mod 2, and both need the map section to start on as many entries (build_family starts
    // every section on a multiple of 4).  The adjacency tensors and nN_x_n always take the 128-bit path; x_n (13 N) takes
    // the 64-bit one for odd num_x, nN_x_e (21 E) the 32-bit one.
    static_assert((N * N) % 4 == 0 && (N * 12) % 4 == 0 && (N * 13) % 2 == 0, "vector width of the output streams");
    emit(args.out.x_n, fam->map_xn, N * 13);
    emit(args.out.A_s, fam->map_as, N * N);
    emit(args.out.A_n_ts, fam->map_ts, N * N);
    emit(args.out.A_n_cs, fam->map_cs, N * N);
    emit(args.out.nN_x_n, fam->map_rawn, N * 12);
    emit(args.out.nN_x_e, fam->map_rawe, E * 21);
    __syncwarp();
  }
}

template <int NX>
int smem_bytes_for(int map_entries, int n_tables = 1) {
  return align16(n_tables * (int)sizeof(FamilyTables)) + align16(((map_entries + 7) & ~7) * 2) + WARPS_PER_CTA * Dims<NX>::WARP_BYTES;
}

// The chord lengths the env-step kernel is built for: one lane per node, so N = 2 NX <= 32; NX = 2 leaves no free bottom node
// to carry a bridge's load.  Every NX has the env-step / reset / solve-only, the gene-vector and the mixed-family kernel.
constexpr int NX_MIN = 3, NX_MAX = TFEM_MAX_NX;

using StepKernel = void (*)(const StepArgs);
struct NxKernels {
  StepKernel step, genes, mixed;
  int (*smem)(int map_entries, int n_tables);
};

template <int... I>
constexpr std::array<NxKernels, sizeof...(I)> nx_table(std::integer_sequence<int, I...>) {
  return {{{tfem_step_kernel<NX_MIN + I, false, false>, tfem_step_kernel<NX_MIN + I, true, false>,
            tfem_step_kernel<NX_MIN + I, false, true>, smem_bytes_for<NX_MIN + I>}...}};
}
constexpr auto kNxKernels = nx_table(std::make_integer_sequence<int, NX_MAX - NX_MIN + 1>{});

const NxKernels* kernels_for(int nx) { return (nx >= NX_MIN && nx <= NX_MAX) ? &kNxKernels[nx - NX_MIN] : nullptr; }

cudaError_t configure_one(StepKernel k, int smem, int* ctas) {
  cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (err != cudaSuccess) return err;
  err = cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (err != cudaSuccess) return err;
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas, k, WARPS_PER_CTA * 32, smem);
}

// The opt-in size is an attribute of the function, shared by every live handle of this NX.  It is set to what the
// largest family count needs (capped by the device's per-block limit), never to what one handle needs, so creating a
// handle of few families cannot break a live handle of more.
cudaError_t configure_mixed_nx(const NxKernels& k, int map_entries, int single_ctas, int n_families, int* smem,
                               int* max_families) {
  int dev = 0, optin = 0;
  cudaError_t err = cudaGetDevice(&dev);
  if (err == cudaSuccess) err = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if (err != cudaSuccess) return err;
  int top = TFEM_MAX_FAMILIES;
  while (top > 1 && k.smem(map_entries, top) > optin) --top;
  int ctas = 0;
  err = configure_one(k.mixed, k.smem(map_entries, top), &ctas);
  if (err != cudaSuccess) return err;
  *max_families = 0;
  for (int f = 1; f <= top; ++f) {
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, k.mixed, WARPS_PER_CTA * 32, k.smem(map_entries, f));
    if (err != cudaSuccess) return err;
    if (ctas < single_ctas) break;
    *max_families = f;
  }
  *smem = (n_families <= *max_families) ? k.smem(map_entries, n_families) : 0;
  return cudaSuccess;
}
}  // namespace

int step_kernel_configure(int nx, int device, int map_entries, LaunchInfo* info) {
  const NxKernels* k = kernels_for(nx);
  if (!k) return (int)cudaErrorInvalidValue;
  int ctas = 0, ctas_g = 0, sms = 0;
  const int smem = k->smem(map_entries, 1);
  cudaError_t err = configure_one(k->step, smem, &ctas);
  if (err == cudaSuccess) err = configure_one(k->genes, smem, &ctas_g);
  if (err != cudaSuccess) return (int)err;
  err = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  if (err != cudaSuccess) return (int)err;
  if (ctas < 1) ctas = 1;
  if (ctas_g < 1) ctas_g = 1;
  info->block = WARPS_PER_CTA * 32;
  info->smem_bytes = smem;
  info->ctas_per_sm = ctas;
  info->grid = sms * ctas;          // persistent: a multiple of the SM count, warps stride over envs
  info->grid_genes = sms * ctas_g;
  info->smem_mixed = 0;
  return 0;
}

int step_kernel_configure_mixed(int nx, int map_entries, int n_families, LaunchInfo* info, int* max_families) {
  const NxKernels* k = kernels_for(nx);
  if (!k) return (int)cudaErrorInvalidValue;
  return (int)configure_mixed_nx(*k, map_entries, info->ctas_per_sm, n_families, &info->smem_mixed, max_families);
}

int step_kernel_launch(int nx, const StepArgs& args, const LaunchInfo& info, cudaStream_t stream) {
  if (args.B <= 0) return 0;
  const NxKernels* k = kernels_for(nx);
  if (!k) return (int)cudaErrorInvalidValue;
  const bool gm = args.mode == MODE_GENES, mf = args.family != nullptr;
  if (mf && (gm || info.smem_mixed <= 0)) return (int)cudaErrorInvalidValue;
  const int needed = (args.B + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
  const int full = gm ? info.grid_genes : info.grid;
  const int grid = needed < full ? needed : full;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)info.block);
  cfg.dynamicSmemBytes = (size_t)(mf ? info.smem_mixed : info.smem_bytes); cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // see griddepcontrol.wait in the kernel
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, mf ? k->mixed : gm ? k->genes : k->step, args);
  return (int)(e != cudaSuccess ? e : cudaGetLastError());
}

}  // namespace tfem
