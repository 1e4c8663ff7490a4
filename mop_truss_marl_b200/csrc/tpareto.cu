// Batched Pareto front + spread statistics + hypervolume (include/tpareto.h): one warp per environment, points in
// shared memory, every step O(P^2 / 32) per lane or a warp reduction -- P <= 256 (the driver culls 50 + 150 accumulated
// candidates at the end of a step), fronts beyond MAX_FRONT thinned with the caller's draw.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string>

#include "../../include/tfem.h"
#include "../../include/tpareto.h"

namespace {
thread_local std::string g_pareto_err;
int pfail(int code, const std::string& m) { g_pareto_err = m; return code; }

constexpr int MAXP = TPARETO_MAX_POINTS;          // 256
constexpr int SL = MAXP / 32;                     // point slots per lane
constexpr int WARPS = 4;

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// min / max that propagate NaN like np.minimum / np.maximum / ndarray.max (fmin / fmax drop it); equal to fmin / fmax on
// numbers up to the sign of a zero result, which no output of the kernel depends on
__device__ __forceinline__ double nan_min(double a, double b) { return (a < b || a != a) ? a : b; }
__device__ __forceinline__ double nan_max(double a, double b) { return (a > b || a != a) ? a : b; }
__device__ __forceinline__ double warp_max(double v) {
  for (int o = 16; o; o >>= 1) v = nan_max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ double warp_min(double v) {
  for (int o = 16; o; o >>= 1) v = nan_min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Sort keys with NumPy's NaN convention: a NaN comes after every number, NaNs tie with each other.  Each returns whether
// key a (at index j) goes before key b (at index k), ties by index, so ranks by counting are a permutation for any input;
// a comparison that is not a total order would give two members one rank and leave a slot unwritten.
__device__ __forceinline__ bool key_tie(bool an, bool bn, double a, double b) { return an == bn && (an || a == b); }
__device__ __forceinline__ bool asc_before(double a, int j, double b, int k) {
  const bool an = a != a, bn = b != b;
  return key_tie(an, bn, a, b) ? j < k : (an != bn ? bn : a < b);
}
__device__ __forceinline__ bool desc_before(double a, int j, double b, int k) {
  const bool an = a != a, bn = b != b;
  return key_tie(an, bn, a, b) ? j < k : (an != bn ? bn : a > b);
}
// the front's list order (utils.py:57): obj1 ascending, then obj2 descending, then index
__device__ __forceinline__ bool list_before(float4 q, int j, float4 p, int i) {
  const bool qn = q.x != q.x, pn = p.x != p.x;
  if (!key_tie(qn, pn, q.x, p.x)) return qn != pn ? pn : q.x < p.x;
  return desc_before(q.y, j, p.y, i);
}
__device__ __forceinline__ int warp_isum(int v) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One warp per environment, points in shared memory; every step is O(P^2 / 32) per lane or a warp reduction.
__global__ void __launch_bounds__(WARPS * 32)
pareto_front_hv_kernel(int B, int P, const float* __restrict__ points, const int32_t* __restrict__ counts, double rx,
                       double ry, const int32_t* __restrict__ thin_pick, int max_front, int32_t* __restrict__ front_idx,
                       int32_t* __restrict__ front_len, double* __restrict__ stats, double* __restrict__ hv) {
  // scratch: the environment's points first; once the sorted front exists the same bytes hold the crowd distances and
  // the crowd-sorted interior (thinning), then the x-sorted copy of the thinned front (hypervolume)
  __shared__ __align__(16) unsigned char scratch[WARPS][MAXP * 16];
  __shared__ int order[WARPS][MAXP];       // front members in list order
  __shared__ double fx[WARPS][MAXP], fy[WARPS][MAXP];
  __shared__ unsigned char member[WARPS][MAXP];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float4* pt = reinterpret_cast<float4*>(scratch[warp]);
  for (int b = blockIdx.x * WARPS + warp; b < B; b += gridDim.x * WARPS) {
    const int n = counts ? min(max(counts[b], 0), P) : P;
    for (int i = lane; i < n; i += 32) pt[i] = reinterpret_cast<const float4*>(points)[(size_t)b * P + i];
    __syncwarp();
    // ---- feasibility, duplicates, dominance (utils.py:17-54) ----
    int nf = 0;
    for (int i = lane; i < MAXP; i += 32) {
      bool keep = false;
      if (i < n) {
        const float4 p = pt[i];
        keep = !(p.z > 1.f || p.w > 1.f);
        for (int j = 0; j < n && keep; ++j) {
          const float4 q = pt[j];
          if (q.z > 1.f || q.w > 1.f) continue;
          if (q.x < p.x && q.y < p.y) keep = false;                                      // dominated
          if (j < i && q.x == p.x && q.y == p.y && q.z == p.z && q.w == p.w) keep = false;   // same tuple: kept once
        }
      }
      member[warp][i] = keep ? 1 : 0;
      nf += keep ? 1 : 0;
    }
    int F = warp_isum(nf);
    __syncwarp();
    // ---- rank among the front members by (obj1 ascending, obj2 descending, index) (:57) ----
    for (int i = lane; i < n; i += 32) {
      if (!member[warp][i]) continue;
      const float4 p = pt[i];
      int rank = 0;
      for (int j = 0; j < n; ++j) {
        if (!member[warp][j] || j == i) continue;
        const float4 q = pt[j];
        if (list_before(q, j, p, i)) ++rank;
      }
      order[warp][rank] = i;
      fx[warp][rank] = (double)p.x;
      fy[warp][rank] = (double)p.y;
    }
    __syncwarp();
    // ---- more than MAX_FRONT members (:104-131): first and last stay, MAX_FRONT - 2 of the others are taken from the list
    //      sorted by crowd distance (descending, stable) at the positions the caller drew, in the order of the draw ----
    bool resort = false;
    if (F > max_front && thin_pick && max_front >= 3 && max_front <= 64) {
      double* crowd = reinterpret_cast<double*>(scratch[warp]);              // [MAXP]
      int* sorted = reinterpret_cast<int*>(scratch[warp] + MAXP * 8);        // [MAXP] interior members by crowd distance
      for (int k = lane; k < F; k += 32) {
        auto dist = [&](int a) {
          // each product rounded like NumPy's: a contracted fma(ax, ax, ay * ay) can split a tie the stable sort below
          // must keep, e.g. the mirrored gaps of a front symmetric in obj1 <-> obj2
          const double ax = fx[warp][a] - fx[warp][a + 1], ay = fy[warp][a] - fy[warp][a + 1];
          return sqrt(__dadd_rn(__dmul_rn(ax, ax), __dmul_rn(ay, ay)));
        };
        crowd[k] = (k == 0) ? dist(0) : (k == F - 1) ? dist(F - 2) : dist(k - 1) + dist(k);
      }
      __syncwarp();
      for (int k = 1 + lane; k < F - 1; k += 32) {
        int r = 0;
        const double ck = crowd[k];
        for (int j = 1; j < F - 1; ++j) r += desc_before(crowd[j], j, ck, k) ? 1 : 0;
        sorted[r] = k;
      }
      __syncwarp();
      int src[2];
      double nx[2], ny[2];
      int no[2];
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int t = lane + 32 * s;
        src[s] = -1;
        if (t < max_front) {
          int k = 0;
          if (t == max_front - 1) k = F - 1;
          else if (t > 0) {
            const int pk = thin_pick[(size_t)b * (max_front - 2) + (t - 1)];
            k = sorted[min(max(pk, 0), F - 3)];
          }
          src[s] = k; nx[s] = fx[warp][k]; ny[s] = fy[warp][k]; no[s] = order[warp][k];
        }
      }
      __syncwarp();
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int t = lane + 32 * s;
        if (src[s] >= 0) { fx[warp][t] = nx[s]; fy[warp][t] = ny[s]; order[warp][t] = no[s]; }
      }
      F = max_front;
      resort = true;
      __syncwarp();
    }
    if (front_len && lane == 0) front_len[b] = F;
    if (front_idx)
      for (int i = lane; i < P; i += 32) front_idx[(size_t)b * P + i] = (i < F) ? order[warp][i] : -1;
    // ---- spread statistics (:159-195), over the list in its order ----
    double dsum = 0.0, dmax = 0.0, d[SL];
#pragma unroll
    for (int s = 0; s < SL; ++s) {
      const int k = lane + 32 * s;
      d[s] = 0.0;
      if (k + 1 < F) {
        const double ax = fx[warp][k] - fx[warp][k + 1], ay = fy[warp][k] - fy[warp][k + 1];
        d[s] = sqrt(ax * ax + ay * ay);
        dsum += d[s];
        dmax = nan_max(dmax, d[s]);
      }
    }
    dsum = warp_sum(dsum);
    dmax = warp_max(dmax);
    double max_d = 0.0, dis_d = 1.0, sum_d = 0.0;
    if (F >= 2) {
      const double nd = (double)(F - 1), centre = dmax / nd;
      double acc = 0.0;
#pragma unroll
      for (int s = 0; s < SL; ++s)
        if (lane + 32 * s + 1 < F) acc += (d[s] - centre) * (d[s] - centre);
      acc = warp_sum(acc);
      max_d = dmax; sum_d = dsum; dis_d = sqrt(acc / nd);
    }
    double std_cd = 1.0, p_inv = 0.0;
    if (F > 3) {
      double c[SL], csum = 0.0, cmax = 0.0;
#pragma unroll
      for (int s = 0; s < SL; ++s) {
        const int k = lane + 32 * s;                        // interior point k+1
        c[s] = 0.0;
        if (k + 2 < F) {
          c[s] = fabs(fx[warp][k] - fx[warp][k + 2]) + fabs(fy[warp][k] - fy[warp][k + 2]);
          csum += c[s];
          cmax = nan_max(cmax, c[s]);
        }
      }
      csum = warp_sum(csum);
      cmax = warp_max(cmax);
      if (csum != 0.0) {
        const double nc = (double)(F - 2);
        double mean = 0.0, p10 = 0.0;
#pragma unroll
        for (int s = 0; s < SL; ++s)
          if (lane + 32 * s + 2 < F) { c[s] /= cmax; mean += c[s]; const double c2 = c[s] * c[s], c4 = c2 * c2; p10 += c4 * c4 * c2; }
        mean = warp_sum(mean) / nc;
        p10 = warp_sum(p10);
        double var = 0.0;
#pragma unroll
        for (int s = 0; s < SL; ++s)
          if (lane + 32 * s + 2 < F) var += (c[s] - mean) * (c[s] - mean);
        var = warp_sum(var);
        std_cd = sqrt(var / nc);
        p_inv = pow(p10, 0.1);
      }
    }
    if (stats && lane == 0) {
      double* o = stats + (size_t)b * 5;
      o[0] = max_d; o[1] = dis_d; o[2] = p_inv; o[3] = sum_d; o[4] = std_cd;
    }
    // ---- hypervolume of the list (:463-530): integral of the running maximum height over the x-sorted members ----
    if (hv) {
      const double* sx = fx[warp];
      const double* sy = fy[warp];
      if (resort) {                                          // the thinned list is in draw order: sort a copy by x
        double* tx = reinterpret_cast<double*>(scratch[warp]);
        double* ty = tx + MAXP;
        for (int k = lane; k < F; k += 32) {
          int r = 0;
          const double xk = fx[warp][k];
          for (int j = 0; j < F; ++j) r += asc_before(fx[warp][j], j, xk, k) ? 1 : 0;
          tx[r] = xk; ty[r] = fy[warp][k];
        }
        __syncwarp();
        sx = tx; sy = ty;
      }
      double area = 0.0, minx = INFINITY, miny = INFINITY;
      for (int k = lane; k < F; k += 32) {
        double h = 0.0;
        for (int j = 0; j <= k; ++j) h = nan_max(h, 1.0 - nan_min(sy[j], 1.0));
        const double x0 = nan_min(sx[k], 1.0), x1 = (k + 1 < F) ? nan_min(sx[k + 1], 1.0) : 1.0;
        area += (x1 - x0) * h;
        minx = nan_min(minx, sx[k]);
        miny = nan_min(miny, sy[k]);
      }
      area = warp_sum(area);
      minx = warp_min(minx);
      miny = warp_min(miny);
      double out = 0.0;
      if (F > 0 && !(F == 1 && sx[0] == 1.0 && sy[0] == 1.0))
        out = area - ((1.0 - rx) * (1.0 - minx) + (1.0 - ry) * (1.0 - miny) - (1.0 - rx) * (1.0 - ry));
      if (lane == 0) hv[b] = out;
    }
    __syncwarp();
  }
}

// pareto_state_data + the driver's padding: one CTA per environment; thread t writes row t of x_p, all threads sweep A_p
// (coalesced stores, so a 50 x 50 matrix is 10 KB written once)
__global__ void __launch_bounds__(128)
pareto_state_data_kernel(int B, int P_in, int P_out, double max_front, const float* __restrict__ points, const int32_t* __restrict__ front_idx,
                         const int32_t* __restrict__ front_len, const int32_t* __restrict__ index, float* __restrict__ x_p,
                         float* __restrict__ A_p) {
  const int b = blockIdx.x;
  if (b >= B) return;
  const int len = front_len ? min(max(front_len[b], 0), P_in) : P_in;
  const int sel = index ? index[b] : 0;
  const float frac = (float)((double)len / max_front);       // len(pf) / MAX_FRONT: a Python float stored into a float32 array
  for (int i = threadIdx.x; i < P_out; i += blockDim.x) {
    float4 row = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < len) {
      const int src = front_idx ? front_idx[(size_t)b * P_in + i] : i;
      const float* p = points + ((size_t)b * P_in + (src >= 0 && src < P_in ? src : 0)) * 4;
      row = make_float4(p[0], p[1], i == sel ? 1.f : 0.f, frac);
    }
    reinterpret_cast<float4*>(x_p)[(size_t)b * P_out + i] = row;
  }
  // degree_power(A, -1/2): np.power(float32 degree, -0.5) for degree 1 (a single point), 2 (chain ends), 3 (interior)
  const float d1 = 1.f, d2 = __uint_as_float(0x3f3504f3u), d3 = __uint_as_float(0x3f13cd3au);
  auto dpow = [&](int i) { return len == 1 ? d1 : ((i == 0 || i == len - 1) ? d2 : d3); };
  float* A = A_p + (size_t)b * P_out * P_out;
  for (int idx = threadIdx.x; idx < P_out * P_out; idx += blockDim.x) {
    const int i = idx / P_out, j = idx - i * P_out;
    float v = 0.f;
    if (i < len && j < len && (j - i <= 1) && (i - j <= 1)) v = __fmul_rn(dpow(i), dpow(j));   // D (A D): one product each
    A[idx] = v;
  }
}
}  // namespace

extern "C" {

const char* tpareto_last_error(void) { return g_pareto_err.c_str(); }

static int front_hv_impl(int B, int P, const float* points, const int32_t* counts, const double* ref_point,
                         const int32_t* thin_pick, int max_front, int32_t* front_idx, int32_t* front_len, double* stats,
                         double* hv, void* stream) {
  if (!points) return pfail(TFEM_ERR_ARG, "null argument");
  if (B < 0) return pfail(TFEM_ERR_ARG, "negative batch");
  if (P < 1 || P > TPARETO_MAX_POINTS) return pfail(TFEM_ERR_ARG, "P must be in 1..256");
  if (thin_pick && (max_front < 3 || max_front > 64)) return pfail(TFEM_ERR_ARG, "max_front must be in 3..64");
  if (reinterpret_cast<uintptr_t>(points) & 15u) return pfail(TFEM_ERR_ALIGN, "points must be 16-byte aligned");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return pfail(TFEM_ERR_CUDA, "no CUDA device: no CPU path");
  if (B == 0) return TFEM_OK;
  const double rx = ref_point ? ref_point[0] : 1.0, ry = ref_point ? ref_point[1] : 1.0;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int need = (B + WARPS - 1) / WARPS;
  const int grid = need < sms * 8 ? need : sms * 8;
  pareto_front_hv_kernel<<<grid, WARPS * 32, 0, (cudaStream_t)stream>>>(B, P, points, counts, rx, ry, thin_pick, max_front,
                                                                        front_idx, front_len, stats, hv);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(TFEM_ERR_CUDA, std::string("pareto kernel: ") + cudaGetErrorString(e));
  return TFEM_OK;
}

int tpareto_front_hv(int B, int P, const float* points, const int32_t* counts, const double* ref_point,
                     int32_t* front_idx, int32_t* front_len, double* stats, double* hv, void* stream) {
  return front_hv_impl(B, P, points, counts, ref_point, nullptr, 50, front_idx, front_len, stats, hv, stream);
}

int tpareto_front_hv_thin(int B, int P, const float* points, const int32_t* counts, const double* ref_point,
                          const int32_t* thin_pick, int max_front, int32_t* front_idx, int32_t* front_len, double* stats,
                          double* hv, void* stream) {
  if (!thin_pick) return pfail(TFEM_ERR_ARG, "null thin_pick");
  return front_hv_impl(B, P, points, counts, ref_point, thin_pick, max_front, front_idx, front_len, stats, hv, stream);
}

int tpareto_state_data(int B, int P_in, int P_out, int max_front, const float* points, const int32_t* front_idx,
                       const int32_t* front_len, const int32_t* index, float* x_p, float* A_p, void* stream) {
  if (max_front < 1) return pfail(TFEM_ERR_ARG, "max_front must be positive");
  if (!points || !x_p || !A_p) return pfail(TFEM_ERR_ARG, "null argument");
  if (B < 0) return pfail(TFEM_ERR_ARG, "negative batch");
  if (P_out < 1 || P_out > 64) return pfail(TFEM_ERR_ARG, "P_out must be in 1..64");
  if (P_in < 1 || P_in > 256) return pfail(TFEM_ERR_ARG, "P_in must be in 1..256");
  if (reinterpret_cast<uintptr_t>(x_p) & 15u) return pfail(TFEM_ERR_ALIGN, "x_p must be 16-byte aligned");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return pfail(TFEM_ERR_CUDA, "no CUDA device: no CPU path");
  if (B == 0) return TFEM_OK;
  pareto_state_data_kernel<<<B, 128, 0, (cudaStream_t)stream>>>(B, P_in, P_out, (double)max_front, points, front_idx, front_len, index, x_p, A_p);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(TFEM_ERR_CUDA, std::string("pareto state kernel: ") + cudaGetErrorString(e));
  return TFEM_OK;
}

}  // extern "C"
