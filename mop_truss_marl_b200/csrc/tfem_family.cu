// Host-side builder of the per-family constant tables (no device code in this file).
// Restates truss2D_GEN.gen_model.gennode/generate (truss2D_GEN.py:181-190, 241-434), the DOF numbering
// of FEM_2Dtruss.Model.gen_nsc/gen_tnsc/gen_ndof/gen_jlv (FEM_2Dtruss.py:227-280), the hard-coded
// symmetry lists of truss2D_ENV.py and the topology-constant parts of state_data /
// state_data_not_norm (truss2D_ENV.py:43-196).
#include "tfem_family.h"

#include <math.h>
#include <string.h>
#include <algorithm>

namespace tfem {

float pairwise_sum_f32(const float* a, int n) {
  if (n < 8) {
    float r = 0.f;
    for (int i = 0; i < n; ++i) r = r + a[i];
    return r;
  }
  float r[8];
  for (int k = 0; k < 8; ++k) r[k] = a[k];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int k = 0; k < 8; ++k) r[k] = r[k] + a[i + k];
  float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
  for (; i < n; ++i) res = res + a[i];
  return res;
}

static float norm_col(float v, float mn, float mx) {
  // (x - min) / (max - min + 1e-6) on float32 arrays (truss2D_ENV.py:102)
  volatile float num = v - mn;
  volatile float den = mx - mn;
  den = den + 1e-6f;
  return num / den;
}

bool build_family(const tfem_family_desc& d, Family& f) {
  f.desc = d;
  const int nx = d.num_x;
  if (nx < 3 || nx > TFEM_MAX_NX) {
    f.error = "num_x must be 3.." + std::to_string(TFEM_MAX_NX) + " (one kernel lane per node, at most 32 nodes; num_x = 2 leaves "
              "no free bottom node to carry a load); got " + std::to_string(nx);
    return false;
  }
  if (d.truss_type != TFEM_BRIDGE && d.truss_type != TFEM_ROOF) {
    f.error = "truss_type must be TFEM_BRIDGE or TFEM_ROOF";
    return false;
  }
  if (d.symmetry < TFEM_SYM_NONE || d.symmetry > TFEM_SYM_LARGE) {
    f.error = "bad symmetry convention";
    return false;
  }
  if (d.symmetry != TFEM_SYM_NONE && nx != 6 && nx != 8 && nx != 16) {
    // the reference's symmetry index lists exist only in the 8- and 16-column truss2D_ENV.py files
    f.error = std::string("the ") + (d.symmetry == TFEM_SYM_SMALL ? "small" : "large") +
              " symmetry convention is defined for num_x 6, 8 and 16 only; num_x = " + std::to_string(nx) +
              " takes TFEM_SYM_NONE (train/code's ENV, which has no symmetry step)";
    return false;
  }
  const int N = 2 * nx, E = 5 * nx - 4;
  FamilyTables& t = f.t;
  memset(&t, 0, sizeof(t));
  t.nx = nx; t.N = N; t.E = E; t.truss_type = d.truss_type; t.symmetry = d.symmetry;

  // ---- nodes: row-major, bottom chord first (gennode) ------------------------------------------------
  std::vector<double> xs(nx);
  double acc = 0;
  for (int i = 0; i < nx; ++i) { xs[i] = acc; if (i < nx - 1) acc += d.span_x[i]; }
  const double total_span = acc;
  for (int i = 0; i < N; ++i) {
    t.x[i] = xs[i % nx];
    t.y0[i] = (i < nx) ? 0.0 : d.span_y;
    t.top[i] = (i >= nx);
    t.pair[i] = (uint8_t)((i < nx) ? i + nx : i - nx);
    t.target[i] = (i >= nx) ? d.tar_y[i - nx] : 0.0;
  }
  // ---- elements: chords, verticals, '\' braces, '/' braces (generate) -----------------------------------
  int e = 0;
  for (int row = 0; row < 2; ++row)
    for (int i = 0; i < nx - 1; ++i) { t.conn[e][0] = row * nx + i; t.conn[e][1] = row * nx + i + 1; ++e; }
  for (int i = 0; i < nx; ++i) { t.conn[e][0] = i; t.conn[e][1] = nx + i; ++e; }
  for (int i = 0; i < nx - 1; ++i) { t.conn[e][0] = nx + i; t.conn[e][1] = i + 1; ++e; }
  for (int i = 0; i < nx - 1; ++i) { t.conn[e][0] = i; t.conn[e][1] = nx + i + 1; ++e; }
  // ---- supports ---------------------------------------------------------------------------------------
  double xmin = xs[0], xmax = xs[nx - 1];
  {
    std::vector<double> xc(xs);
    if (d.support_case == 2) xc.pop_back();
    else if (d.support_case == 3) xc.erase(xc.begin());
    else if (d.support_case == 4) { xc.erase(xc.begin()); xc.pop_back(); }
    xmin = *std::min_element(xc.begin(), xc.end());
    xmax = *std::max_element(xc.begin(), xc.end());
  }
  for (int i = 0; i < N; ++i)
    if (t.y0[i] == 0.0 && (t.x[i] == xmax || t.x[i] == xmin)) t.res[i] = 3;
  // ---- loads ------------------------------------------------------------------------------------------
  for (int i = 0; i < N; ++i) {
    bool ld = (d.truss_type == TFEM_BRIDGE) ? (t.y0[i] == 0.0 && !(t.res[i] & 2)) : (t.top[i] == 1);
    t.loaded[i] = ld;
    t.fy[i] = ld ? d.load_y : 0.0;
  }
  // ---- DOF ids: free first, node-major, x then y --------------------------------------------------------
  int c = 1;
  for (int i = 0; i < N; ++i) for (int a = 0; a < 2; ++a) if (!((t.res[i] >> a) & 1)) t.dof[i][a] = c++;
  t.ndof = c - 1;
  for (int i = 0; i < N; ++i) for (int a = 0; a < 2; ++a) if ((t.res[i] >> a) & 1) t.dof[i][a] = c++;
  t.nres = 2 * N - t.ndof;
  for (int i = 0; i < N; ++i) for (int a = 0; a < 2; ++a)
    t.react_slot[i][a] = ((t.res[i] >> a) & 1) ? (int16_t)(t.dof[i][a] - 1 - t.ndof) : (int16_t)-1;
  // ---- adjacency lists (element order = accumulation order of the nodal diagonal block) ----------------
  for (int i = 0; i < N; ++i) for (int k = 0; k < MAXADJ; ++k) t.adj[i][k] = -1;
  for (int el = 0; el < E; ++el)
    for (int s = 0; s < 2; ++s) {
      int nd = t.conn[el][s], k = 0;
      while (t.adj[nd][k] >= 0) ++k;
      if (k >= MAXADJ - 1) { f.error = "node degree too large"; return false; }
      t.adj[nd][k] = (int8_t)el;
    }
  // ---- symmetry ---------------------------------------------------------------------------------------
  for (int i = 0; i < N; ++i) t.sym_src[0][i] = t.sym_src[1][i] = (int8_t)i;
  for (int el = 0; el < E; ++el) t.sym_elem[el] = (int8_t)el;
  if (d.symmetry != TFEM_SYM_NONE) {
    std::vector<int8_t> left_from_right(N), right_from_left(N);
    for (int i = 0; i < N; ++i) left_from_right[i] = right_from_left[i] = (int8_t)i;
    for (int row = 0; row < 2; ++row)
      for (int ci = 0; ci < nx / 2; ++ci) {
        int a = row * nx + ci, b = row * nx + (nx - 1 - ci);
        if (d.symmetry == TFEM_SYM_SMALL && row == 0 && ci == 0) continue;  // support pair not listed
        left_from_right[a] = (int8_t)b;
        right_from_left[b] = (int8_t)a;
      }
    for (int i = 0; i < N; ++i) {
      // small: coin true copies right -> left ; large: coin true copies left -> right
      t.sym_src[1][i] = (d.symmetry == TFEM_SYM_SMALL) ? left_from_right[i] : right_from_left[i];
      t.sym_src[0][i] = (d.symmetry == TFEM_SYM_SMALL) ? right_from_left[i] : left_from_right[i];
    }
    const int nb = nx - 1;
    auto link = [&](int a, int b) { t.sym_elem[a] = (int8_t)b; t.sym_elem[b] = (int8_t)a; };
    for (int row = 0; row < 2; ++row) for (int k = 0; k < nb / 2; ++k) link(row * nb + k, row * nb + nb - 1 - k);
    const int base = 2 * nb;
    for (int k = 0; k < nx / 2; ++k) link(base + k, base + nx - 1 - k);
    const int b3 = base + nx, b4 = base + nx + nb;
    for (int k = 0; k < nb; ++k) link(b3 + k, b4 + nb - 1 - k);
  }
  // ---- scalars ----------------------------------------------------------------------------------------
  t.y_max = d.span_y; t.y_min = 0.0; t.d_min = d.d_min;
  t.ymax_minus_dmin = d.span_y - d.d_min;
  t.max_def = 0.001 * total_span;           // truss2D_GEN.py:78
  t.maxdef32 = (float)t.max_def;
  t.young = d.young; t.allow = d.allow_stress; t.load_y = d.load_y;
  const double amax = d.section_area_cm2[TFEM_NSEC - 1] * 1e-4;
  for (int s = 0; s < TFEM_NSEC; ++s) {
    t.sec_area[s] = d.section_area_cm2[s] * 1e-4;
    t.sec_area32[s] = (float)t.sec_area[s];
    t.sec_as32[s] = (float)(t.sec_area[s] / amax);
  }
  // ---- initial objectives (Game_research04.__init__, truss2D_ENV.py:267-277) ---------------------------
  {
    std::vector<float> all_v(E), all_dt(N, 0.f);
    for (int el = 0; el < E; ++el) {
      double dx = t.x[t.conn[el][1]] - t.x[t.conn[el][0]];
      double dy = t.y0[t.conn[el][1]] - t.y0[t.conn[el][0]];
      double L = pow(pow(dx, 2.0) + pow(dy, 2.0), 0.5);      // Element.gen_length, python float **
      all_v[el] = (float)(amax * L);
    }
    for (int i = 0; i < N; ++i) if (t.top[i]) all_dt[i] = (float)fabs(t.target[i] - t.y0[i]);
    t.int_obj1 = pairwise_sum_f32(all_v.data(), E);
    t.int_obj2 = pairwise_sum_f32(all_dt.data(), N);
  }
  // ---- host-visible tables -----------------------------------------------------------------------------
  f.conn.resize(2 * E); f.tnsc.resize(2 * N); f.res.resize(2 * N); f.top.resize(N); f.pair.resize(N);
  f.loaded.resize(N); f.sym_src.resize(2 * N); f.sym_elem.resize(E);
  f.x.assign(t.x, t.x + N); f.y0.assign(t.y0, t.y0 + N); f.target.assign(t.target, t.target + N);
  for (int el = 0; el < E; ++el) { f.conn[2 * el] = t.conn[el][0]; f.conn[2 * el + 1] = t.conn[el][1]; f.sym_elem[el] = t.sym_elem[el]; }
  f.loadvec.assign(t.ndof, 0.0);
  for (int i = 0; i < N; ++i) {
    for (int a = 0; a < 2; ++a) {
      f.tnsc[2 * i + a] = t.dof[i][a];
      f.res[2 * i + a] = (t.res[i] >> a) & 1;
      if (t.dof[i][a] <= t.ndof) f.loadvec[t.dof[i][a] - 1] = (a == 1) ? t.fy[i] : 0.0;
    }
    f.top[i] = t.top[i]; f.pair[i] = t.pair[i]; f.loaded[i] = t.loaded[i];
    f.sym_src[i] = t.sym_src[0][i]; f.sym_src[N + i] = t.sym_src[1][i];
  }
  // A_n = D^-1/2 (A + I) D^-1/2 in float32; mask; c_e
  f.A_n.assign(N * N, 0.f); f.mask.assign(N * N, 0.f); f.nC_e.assign(E * N, 0.f);
  std::vector<float> adjm(N * N, 0.f);
  for (int el = 0; el < E; ++el) {
    int a = t.conn[el][0], b = t.conn[el][1];
    adjm[a * N + b] = adjm[b * N + a] = 1.f;
    f.mask[a * N + b] = f.mask[b * N + a] = 1.f;
    f.nC_e[el * N + a] = 1.f; f.nC_e[el * N + b] = 1.f;
  }
  std::vector<float> dm(N);
  for (int i = 0; i < N; ++i) {
    adjm[i * N + i] += 1.f;
    float deg = 0.f;
    for (int j = 0; j < N; ++j) deg += adjm[i * N + j];
    // np.power(float32 deg, -1/2).  NumPy's AVX-512 float32 `power` loop (SVML) is what the reference
    // executes on this image's hosts; it is 1 ulp away from the correctly rounded value for deg = 6, 7.
    // The table below holds its results (bit patterns) for every degree a 2-chord truss can have.
    static const uint32_t kDegPowBits[9] = {0u, 1065353216u, 1060439283u, 1058262330u, 1056964608u,
                                            1055193390u, 1053885931u, 1052869776u, 1052050675u};
    const int ideg = (int)deg;
    if (ideg >= 1 && ideg <= 8) memcpy(&dm[i], &kDegPowBits[ideg], 4);
    else dm[i] = powf(deg, -0.5f);
  }
  for (int i = 0; i < N; ++i)
    for (int j = 0; j < N; ++j) {
      volatile float inner = adjm[i * N + j] * dm[j];
      f.A_n[i * N + j] = dm[i] * inner;
    }
  // ---- value pool constants and output maps -------------------------------------------------------------
  PoolLayout pl{N, E};
  t.pool_const[0] = 0.f; t.pool_const[1] = 1.f;
  {
    float raw[6][MAXN];
    for (int i = 0; i < N; ++i) {
      raw[0][i] = (float)t.x[i];
      raw[1][i] = (float)(t.res[i] & 1);
      raw[2][i] = (float)((t.res[i] >> 1) & 1);
      raw[3][i] = t.loaded[i] ? 1.f : 0.f;       // abs(has_loady), has_loady forced to 1 (:425,:430)
      raw[4][i] = (float)t.top[i];
      raw[5][i] = (float)(t.top[i] ? 0 : 1);
    }
    for (int k = 0; k < 6; ++k) {
      float mn = raw[k][0], mx = raw[k][0];
      for (int i = 1; i < N; ++i) { mn = std::min(mn, raw[k][i]); mx = std::max(mx, raw[k][i]); }
      for (int i = 0; i < N; ++i) {
        t.pool_const[pl.xn_const(k) + i] = norm_col(raw[k][i], mn, mx);
        t.pool_const[pl.raw_const(k) + i] = raw[k][i];
      }
    }
  }
  auto& mp = f.maps;
  mp.clear();
  // every section starts on a multiple of 4 entries: the kernel reads a section's map with 64- or 128-bit loads (only an
  // odd num_x, whose x_n map has 26 num_x entries, needs the padding)
  auto section = [&mp](int32_t* off) { while (mp.size() % 4) mp.push_back(0); *off = (int)mp.size(); };
  static const int xn_const_col[13] = {0, -1, 1, 2, 3, 4, 5, -1, -1, -1, -1, -1, -1};
  static const int xn_dyn_col[13] = {-1, 0, -1, -1, -1, -1, -1, 1, 2, 3, 4, 5, 6};
  static const int raw_const_col[12] = {0, -1, 1, 2, 3, 4, 5, -1, -1, -1, -1, -1};
  static const int raw_dyn_col[12] = {-1, 0, -1, -1, -1, -1, -1, 1, 2, 3, 4, 5};
  section(&t.map_xn);
  for (int i = 0; i < N; ++i)
    for (int k = 0; k < 13; ++k)
      mp.push_back((uint16_t)(xn_const_col[k] >= 0 ? pl.xn_const(xn_const_col[k]) + i : pl.xn_dyn(xn_dyn_col[k]) + i));
  std::vector<int> pair_el(N * N, -1);
  for (int el = 0; el < E; ++el) {
    int a = t.conn[el][0], b = t.conn[el][1];
    pair_el[a * N + b] = pair_el[b * N + a] = el;
  }
  const int adj_cols[3] = {EL_AS, EL_TS, EL_CS};
  int32_t* adj_off[3] = {&t.map_as, &t.map_ts, &t.map_cs};
  for (int m = 0; m < 3; ++m) {
    section(adj_off[m]);
    for (int i = 0; i < N * N; ++i) mp.push_back((uint16_t)(pair_el[i] >= 0 ? pl.el(adj_cols[m]) + pair_el[i] : 0));
  }
  section(&t.map_rawn);
  for (int i = 0; i < N; ++i)
    for (int k = 0; k < 12; ++k)
      mp.push_back((uint16_t)(raw_const_col[k] >= 0 ? pl.raw_const(raw_const_col[k]) + i : pl.raw_dyn(raw_dyn_col[k]) + i));
  section(&t.map_rawe);
  for (int el = 0; el < E; ++el) {
    for (int k = 0; k < 7; ++k) mp.push_back((uint16_t)(pl.el(k) + el));
    for (int s = 0; s < 2; ++s) {
      int nd = t.conn[el][s];
      mp.push_back((uint16_t)(pl.raw_const(0) + nd));   // x
      mp.push_back((uint16_t)(pl.raw_dyn(0) + nd));     // y
      mp.push_back((uint16_t)(pl.raw_const(1) + nd));   // res x
      mp.push_back((uint16_t)(pl.raw_const(2) + nd));   // res y
      mp.push_back((uint16_t)(pl.raw_const(3) + nd));   // |load|
      mp.push_back((uint16_t)(pl.raw_dyn(4) + nd));     // |dy|
      mp.push_back((uint16_t)(pl.raw_dyn(5) + nd));     // deflection flag (>= 1)
    }
  }
  t.map_total = (int)mp.size();
  while (mp.size() % 8) mp.push_back(0);
  return true;
}

}  // namespace tfem
