// C ABI of libtfem (see include/tfem.h for the contract and the reference interfaces it replaces).
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <atomic>
#include <new>
#include <string>

#include "tfem_kernels.cuh"

namespace {
thread_local std::string g_err;
int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return TFEM_ERR_CUDA;
}
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
}  // namespace

struct tfem_handle_s {
  tfem::Family fam;                  // the only family, or the first of a mixed handle
  int n_families = 1;                // tfem_create_mixed: tables of all families follow each other in d_tables
  int device = 0;
  tfem::FamilyTables* d_tables = nullptr;
  uint16_t* d_maps = nullptr;
  tfem::LaunchInfo launch{};
  std::atomic<int64_t> launches{0};
  // scratch for tfem_step_host
  unsigned char* d_scratch = nullptr;
  size_t scratch_bytes = 0;
};

namespace {

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { ok = false; return; }
    if (prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// entry points that serve one family refuse a handle of several
int single_family(tfem_handle_t h, const char* call, const char* instead) {
  if (h->n_families == 1) return 0;
  return fail(TFEM_ERR_ARG, std::string(call) + ": the handle holds " + std::to_string(h->n_families) +
                                " families; use " + instead + " (or a handle of one family)");
}

// the mixed entry points need the mixed kernel configured (tfem_create_mixed); a tables-only handle fails at launch
int mixed_family(tfem_handle_t h, const char* call) {
  if (h->device < 0 || tfem::handle_is_mixed(h)) return 0;
  return fail(TFEM_ERR_ARG, std::string(call) + ": the handle was made by tfem_create; use tfem_create_mixed");
}

// first topology table in which family b differs from family a, or nullptr.  These are what the kernel reads once per
// launch (or once before its environment loop) and what the output maps are built from.
const char* topology_mismatch(const tfem::Family& a, const tfem::Family& b) {
  const tfem::FamilyTables &s = a.t, &t = b.t;
  if (s.nx != t.nx) return "num_x";
  if (memcmp(s.conn, t.conn, sizeof(s.conn))) return "CONN";
  if (memcmp(s.top, t.top, sizeof(s.top))) return "TOP";
  if (memcmp(s.pair, t.pair, sizeof(s.pair))) return "PAIR";
  if (memcmp(s.adj, t.adj, sizeof(s.adj))) return "adjacency";
  if (a.maps != b.maps || s.map_xn != t.map_xn || s.map_as != t.map_as || s.map_ts != t.map_ts || s.map_cs != t.map_cs ||
      s.map_rawn != t.map_rawn || s.map_rawe != t.map_rawe || s.map_total != t.map_total)
    return "output maps";
  if (memcmp(s.res, t.res, sizeof(s.res))) return "RES";
  if (memcmp(s.dof, t.dof, sizeof(s.dof)) || s.ndof != t.ndof || s.nres != t.nres) return "TNSC";
  if (memcmp(s.react_slot, t.react_slot, sizeof(s.react_slot))) return "reaction slots";
  return nullptr;
}

int check_out_alignment(const tfem_step_out* o) {
  const void* ps[] = {o->x_n, o->A_s, o->A_n_ts, o->A_n_cs, o->nN_x_n, o->nN_x_e, o->point, o->point64,
                      o->d, o->axial, o->ratio, o->U, o->reactions};
  for (const void* p : ps)
    if (p && !aligned16(p)) return fail(TFEM_ERR_ALIGN, "output buffers must be 16-byte aligned");
  return 0;
}

}  // namespace

extern "C" {

const char* tfem_version(void) { return "tfem 0.1.0 (sm_100a)"; }
const char* tfem_last_error(void) { return g_err.c_str(); }

int tfem_create(const tfem_family_desc* desc, int device, tfem_handle_t* out) {
  if (!desc || !out) return fail(TFEM_ERR_ARG, "null argument");
  *out = nullptr;
  tfem_handle_s* h = new (std::nothrow) tfem_handle_s();
  if (!h) return fail(TFEM_ERR_ARG, "out of host memory");
  if (!tfem::build_family(*desc, h->fam)) {
    std::string msg = h->fam.error;
    delete h;
    return fail(TFEM_ERR_UNSUPPORTED, msg);
  }
  if (device < 0) {          // tables-only handle (host logic / tests): every compute entry point fails
    h->device = -1;
    *out = h;
    return TFEM_OK;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    delete h;
    return fail(TFEM_ERR_CUDA, "no CUDA device: libtfem has no CPU path");
  }
  if (device < 0 || device >= ndev) { delete h; return fail(TFEM_ERR_ARG, "bad device index"); }
  h->device = device;
  DeviceGuard guard(device);
  if (!guard.ok) { delete h; return fail(TFEM_ERR_CUDA, "cudaSetDevice failed"); }
  e = cudaMalloc(&h->d_tables, sizeof(tfem::FamilyTables));
  if (e == cudaSuccess) e = cudaMalloc(&h->d_maps, h->fam.maps.size() * sizeof(uint16_t));
  if (e == cudaSuccess) e = cudaMemcpy(h->d_tables, &h->fam.t, sizeof(tfem::FamilyTables), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_maps, h->fam.maps.data(), h->fam.maps.size() * sizeof(uint16_t), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { tfem_destroy(h); return cuda_fail(e, "table upload"); }
  int rc = tfem::step_kernel_configure(h->fam.t.nx, device, h->fam.t.map_total, &h->launch);
  if (rc != 0) { tfem_destroy(h); return cuda_fail((cudaError_t)rc, "kernel configure"); }
  *out = h;
  return TFEM_OK;
}

int tfem_create_mixed(const tfem_family_desc* descs, int n_families, int device, tfem_handle_t* out) {
  if (!descs || !out) return fail(TFEM_ERR_ARG, "null argument");
  *out = nullptr;
  if (n_families < 1 || n_families > TFEM_MAX_FAMILIES)
    return fail(TFEM_ERR_ARG, "n_families must be 1.." + std::to_string(TFEM_MAX_FAMILIES) + ", got " + std::to_string(n_families));
  std::vector<tfem::Family> fams(n_families);
  for (int i = 0; i < n_families; ++i) {
    if (!tfem::build_family(descs[i], fams[i])) return fail(TFEM_ERR_UNSUPPORTED, "family " + std::to_string(i) + ": " + fams[i].error);
    if (i == 0) continue;
    if (const char* tab = topology_mismatch(fams[0], fams[i]))
      return fail(TFEM_ERR_UNSUPPORTED, "family " + std::to_string(i) + " differs from family 0 in the " + tab +
                                            " table: the families of one handle must share num_x and support_case");
  }
  tfem_handle_s* h = new (std::nothrow) tfem_handle_s();
  if (!h) return fail(TFEM_ERR_ARG, "out of host memory");
  h->fam = fams[0];
  h->n_families = n_families;
  if (device < 0) {
    h->device = -1;
    *out = h;
    return TFEM_OK;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) { delete h; return fail(TFEM_ERR_CUDA, "no CUDA device: libtfem has no CPU path"); }
  if (device >= ndev) { delete h; return fail(TFEM_ERR_ARG, "bad device index"); }
  h->device = device;
  DeviceGuard guard(device);
  if (!guard.ok) { delete h; return fail(TFEM_ERR_CUDA, "cudaSetDevice failed"); }
  const size_t tab_bytes = sizeof(tfem::FamilyTables);
  e = cudaMalloc(&h->d_tables, n_families * tab_bytes);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_maps, h->fam.maps.size() * sizeof(uint16_t));
  for (int i = 0; i < n_families && e == cudaSuccess; ++i)
    e = cudaMemcpy(h->d_tables + i, &fams[i].t, tab_bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->d_maps, h->fam.maps.data(), h->fam.maps.size() * sizeof(uint16_t), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { tfem_destroy(h); return cuda_fail(e, "table upload"); }
  int rc = tfem::step_kernel_configure(h->fam.t.nx, device, h->fam.t.map_total, &h->launch);
  int max_families = 0;
  if (rc == 0) rc = tfem::step_kernel_configure_mixed(h->fam.t.nx, (int)h->fam.maps.size(), n_families, &h->launch, &max_families);
  if (rc != 0) { tfem_destroy(h); return cuda_fail((cudaError_t)rc, "kernel configure"); }
  if (n_families > max_families) {
    const int nx = h->fam.t.nx, ctas = h->launch.ctas_per_sm;
    tfem_destroy(h);
    return fail(TFEM_ERR_UNSUPPORTED, "num_x = " + std::to_string(nx) + ": at most " + std::to_string(max_families) +
                                          " families fit the shared memory of one CTA at the env-step kernel's " +
                                          std::to_string(ctas) + " CTAs per SM; got " + std::to_string(n_families));
  }
  *out = h;
  return TFEM_OK;
}

int tfem_destroy(tfem_handle_t h) {
  if (!h) return TFEM_OK;
  if (h->device < 0) { delete h; return TFEM_OK; }
  DeviceGuard guard(h->device);
  if (h->d_tables) cudaFree(h->d_tables);
  if (h->d_maps) cudaFree(h->d_maps);
  if (h->d_scratch) cudaFree(h->d_scratch);
  delete h;
  return TFEM_OK;
}

int tfem_get_dims(tfem_handle_t h, tfem_dims* out) {
  if (!h || !out) return fail(TFEM_ERR_ARG, "null argument");
  const tfem::FamilyTables& t = h->fam.t;
  out->N = t.N; out->E = t.E; out->ndof = t.ndof; out->nres = t.nres;
  out->num_x = t.nx; out->n_internal = 4 * t.nx; out->band = 7; out->device = h->device;
  return TFEM_OK;
}

int tfem_get_table(tfem_handle_t h, int which, void* dst, size_t bytes) {
  if (!h || !dst) return fail(TFEM_ERR_ARG, "null argument");
  const tfem::Family& f = h->fam;
  const void* src = nullptr;
  size_t n = 0;
  if (h->n_families > 1) {
    switch (which) {
      case TFEM_TAB_CONN: case TFEM_TAB_TNSC: case TFEM_TAB_RES: case TFEM_TAB_TOP: case TFEM_TAB_PAIR:
      case TFEM_TAB_A_N: case TFEM_TAB_MASK: case TFEM_TAB_NC_E: break;
      default:
        if (which < TFEM_TAB_CONN || which > TFEM_TAB_SCALARS) return fail(TFEM_ERR_ARG, "unknown table id");
        return fail(TFEM_ERR_ARG, "table " + std::to_string(which) + " differs between the " + std::to_string(h->n_families) +
                                      " families of this handle: read it from a tables-only handle of one family");
    }
  }
  float int_obj[2] = {f.t.int_obj1, f.t.int_obj2};
  double scal[8] = {f.t.y_max, f.t.y_min, f.t.d_min, f.t.max_def, f.t.young, f.t.allow, f.t.load_y, 0.0};
  switch (which) {
    case TFEM_TAB_CONN: src = f.conn.data(); n = f.conn.size() * 4; break;
    case TFEM_TAB_TNSC: src = f.tnsc.data(); n = f.tnsc.size() * 4; break;
    case TFEM_TAB_RES: src = f.res.data(); n = f.res.size() * 4; break;
    case TFEM_TAB_TOP: src = f.top.data(); n = f.top.size() * 4; break;
    case TFEM_TAB_PAIR: src = f.pair.data(); n = f.pair.size() * 4; break;
    case TFEM_TAB_LOADED: src = f.loaded.data(); n = f.loaded.size() * 4; break;
    case TFEM_TAB_LOADVEC: src = f.loadvec.data(); n = f.loadvec.size() * 8; break;
    case TFEM_TAB_X: src = f.x.data(); n = f.x.size() * 8; break;
    case TFEM_TAB_Y0: src = f.y0.data(); n = f.y0.size() * 8; break;
    case TFEM_TAB_TARGET: src = f.target.data(); n = f.target.size() * 8; break;
    case TFEM_TAB_A_N: src = f.A_n.data(); n = f.A_n.size() * 4; break;
    case TFEM_TAB_MASK: src = f.mask.data(); n = f.mask.size() * 4; break;
    case TFEM_TAB_NC_E: src = f.nC_e.data(); n = f.nC_e.size() * 4; break;
    case TFEM_TAB_SYM_SRC: src = f.sym_src.data(); n = f.sym_src.size() * 4; break;
    case TFEM_TAB_SYM_ELEM: src = f.sym_elem.data(); n = f.sym_elem.size() * 4; break;
    case TFEM_TAB_INT_OBJ: src = int_obj; n = sizeof(int_obj); break;
    case TFEM_TAB_SCALARS: src = scal; n = sizeof(scal); break;
    default: return fail(TFEM_ERR_ARG, "unknown table id");
  }
  if (bytes != n) return fail(TFEM_ERR_ARG, "table size mismatch: expected " + std::to_string(n) + " bytes");
  memcpy(dst, src, n);
  return TFEM_OK;
}

static int launch(tfem_handle_t h, tfem::StepArgs& a, void* stream) {
  if (h->device < 0) return fail(TFEM_ERR_CUDA, "tables-only handle (device < 0): libtfem has no CPU path");
  a.fam = h->d_tables;
  a.maps = h->d_maps;
  a.map_entries = (int)h->fam.maps.size();
  DeviceGuard guard(h->device);
  if (!guard.ok) return fail(TFEM_ERR_CUDA, "cudaSetDevice failed");
  int rc = tfem::step_kernel_launch(h->fam.t.nx, a, h->launch, (cudaStream_t)stream);
  if (rc != 0) return cuda_fail((cudaError_t)rc, "kernel launch");
  h->launches.fetch_add(1);
  return TFEM_OK;
}

int tfem_reset(tfem_handle_t h, int B, float* move_range_out, const tfem_step_out* out, void* stream) {
  if (!h || !out) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = single_family(h, "tfem_reset", "tfem_reset_mixed")) return rc;
  if (B < 0) return fail(TFEM_ERR_ARG, "negative batch");
  if (int rc = check_out_alignment(out)) return rc;
  if (move_range_out && !aligned16(move_range_out)) return fail(TFEM_ERR_ALIGN, "move_range must be 16-byte aligned");
  tfem::StepArgs a{};
  a.B = B; a.mode = tfem::MODE_RESET; a.out = *out; a.reset_move_range = move_range_out;
  return launch(h, a, stream);
}

static int check_step_in(const tfem_step_in* in) {
  if ((!in->set_node && !in->set_node_y) || (!in->set_element && !in->set_element_section) || !in->a_geo || !in->a_topo ||
      !in->move_range)
    return fail(TFEM_ERR_ARG, "set_node (or set_node_y), set_element (or set_element_section), a_geo, a_topo and move_range are required");
  if ((in->set_node && !aligned16(in->set_node)) || (in->set_element && !aligned16(in->set_element)) || !aligned16(in->a_geo) ||
      !aligned16(in->a_topo) || !aligned16(in->move_range))
    return fail(TFEM_ERR_ALIGN, "input buffers must be 16-byte aligned");
  return 0;
}

int tfem_step(tfem_handle_t h, int B, const tfem_step_in* in, const tfem_step_out* out, void* stream) {
  if (!h || !in || !out) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = single_family(h, "tfem_step", "tfem_step_mixed")) return rc;
  if (B < 0) return fail(TFEM_ERR_ARG, "negative batch");
  if (B == 0) return TFEM_OK;
  if (int rc = check_step_in(in)) return rc;
  if (int rc = check_out_alignment(out)) return rc;
  tfem::StepArgs a{};
  a.B = B; a.mode = tfem::MODE_STEP; a.in = *in; a.out = *out;
  return launch(h, a, stream);
}

int tfem_reset_mixed(tfem_handle_t h, int B, const uint8_t* family, float* move_range_out, const tfem_step_out* out,
                     void* stream) {
  if (!h || !family || !out) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = mixed_family(h, "tfem_reset_mixed")) return rc;
  if (B < 0) return fail(TFEM_ERR_ARG, "negative batch");
  if (int rc = check_out_alignment(out)) return rc;
  if (move_range_out && !aligned16(move_range_out)) return fail(TFEM_ERR_ALIGN, "move_range must be 16-byte aligned");
  tfem::StepArgs a{};
  a.B = B; a.mode = tfem::MODE_RESET; a.out = *out; a.reset_move_range = move_range_out;
  a.family = family; a.n_families = h->n_families;
  return launch(h, a, stream);
}

int tfem_step_mixed(tfem_handle_t h, int B, const uint8_t* family, const tfem_step_in* in, const tfem_step_out* out,
                    void* stream) {
  if (!h || !family || !in || !out) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = mixed_family(h, "tfem_step_mixed")) return rc;
  if (B < 0) return fail(TFEM_ERR_ARG, "negative batch");
  if (B == 0) return TFEM_OK;
  if (int rc = check_step_in(in)) return rc;
  if (int rc = check_out_alignment(out)) return rc;
  tfem::StepArgs a{};
  a.B = B; a.mode = tfem::MODE_STEP; a.in = *in; a.out = *out;
  a.family = family; a.n_families = h->n_families;
  return launch(h, a, stream);
}

int tfem_solve_only(tfem_handle_t h, int B, const double* y, const int32_t* section, double* d, double* axial,
                    double* ratio, double* U, double* reactions, int32_t* status, void* stream) {
  if (!h || !y || !section) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = single_family(h, "tfem_solve_only", "a handle of one family")) return rc;
  if (B < 0) return fail(TFEM_ERR_ARG, "negative batch");
  tfem::StepArgs a{};
  a.B = B; a.mode = tfem::MODE_SOLVE_ONLY; a.so_y = y; a.so_sec = section;
  a.out.d = d; a.out.axial = axial; a.out.ratio = ratio; a.out.U = U; a.out.reactions = reactions; a.out.status = status;
  return launch(h, a, stream);
}

int tfem_read_genes(tfem_handle_t h, int B, const double* genes, double max_height, float int_obj1, float int_obj2,
                    const tfem_genes_out* out, void* stream) {
  if (!h || !genes || !out) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = single_family(h, "tfem_read_genes", "a handle of one family")) return rc;
  if (B < 0) return fail(TFEM_ERR_ARG, "negative batch");
  if (!(max_height > 0.0)) return fail(TFEM_ERR_ARG, "max_height must be positive");
  if (out->point && !aligned16(out->point)) return fail(TFEM_ERR_ALIGN, "point must be 16-byte aligned");
  if (B == 0) return TFEM_OK;
  tfem::StepArgs a{};
  a.B = B; a.mode = tfem::MODE_GENES; a.genes = genes; a.max_height = max_height; a.sec_out = out->section;
  a.int_obj1 = int_obj1; a.int_obj2 = int_obj2;
  a.out.point = out->point; a.out.point64 = out->point64; a.out.y = out->y; a.out.d = out->d; a.out.axial = out->axial;
  a.out.ratio = out->ratio; a.out.U = out->U; a.out.reactions = out->reactions; a.out.status = out->status;
  return launch(h, a, stream);
}

int tfem_solve_dense_dmma(tfem_handle_t h, int B, const double* y, const int32_t* section, double* d,
                          int32_t* status, void* stream) {
  if (!h || !y || !section || !d) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = single_family(h, "tfem_solve_dense_dmma", "a handle of one family")) return rc;
  if (B < 0) return fail(TFEM_ERR_ARG, "negative batch");
  if (h->device < 0) return fail(TFEM_ERR_CUDA, "tables-only handle (device < 0): libtfem has no CPU path");
  if (B == 0) return TFEM_OK;
  DeviceGuard guard(h->device);
  if (!guard.ok) return fail(TFEM_ERR_CUDA, "cudaSetDevice failed");
  const int rc = tfem::dense_solve_launch(h->d_tables, B, y, section, d, status, (cudaStream_t)stream);
  if (rc != 0) return cuda_fail((cudaError_t)rc, "dense DMMA solve");
  h->launches.fetch_add(1);
  return TFEM_OK;
}

int tfem_step_host(tfem_handle_t h, int B, const tfem_step_in* in, const tfem_step_out* out, void* stream_) {
  if (!h || !in || !out) return fail(TFEM_ERR_ARG, "null argument");
  if (int rc = single_family(h, "tfem_step_host", "tfem_step_mixed on device buffers")) return rc;
  if (B <= 0) return B == 0 ? TFEM_OK : fail(TFEM_ERR_ARG, "negative batch");
  if (!in->set_node || !in->set_element || !in->a_geo || !in->a_topo || !in->move_range)
    return fail(TFEM_ERR_ARG, "set_node, set_element, a_geo, a_topo and move_range are required");
  const tfem::FamilyTables& t = h->fam.t;
  const size_t N = t.N, E = t.E, nb = (size_t)B;
  cudaStream_t stream = (cudaStream_t)stream_;
  if (h->device < 0) return fail(TFEM_ERR_CUDA, "tables-only handle (device < 0): libtfem has no CPU path");
  DeviceGuard guard(h->device);
  if (!guard.ok) return fail(TFEM_ERR_CUDA, "cudaSetDevice failed");
  // carve the scratch arena (256-byte aligned slices)
  struct Slice { size_t off, bytes; };
  size_t total = 0;
  auto take = [&](size_t bytes) { Slice s{total, bytes}; total += (bytes + 255) & ~size_t(255); return s; };
  Slice s_node = take(nb * N * 12 * 4), s_elem = take(nb * E * 21 * 4), s_geo = take(nb * N * 2 * 4),
        s_topo = take(nb * N * 3 * 4), s_coin = take(nb), s_mr = take(nb * N * 2 * 4);
  Slice o_xn = take(nb * N * 13 * 4), o_as = take(nb * N * N * 4), o_ts = take(nb * N * N * 4),
        o_cs = take(nb * N * N * 4), o_pt = take(nb * 16), o_p64 = take(nb * 32), o_d = take(nb * t.ndof * 8),
        o_ax = take(nb * E * 8), o_ra = take(nb * E * 8), o_u = take(nb * 8), o_re = take(nb * t.nres * 8),
        o_st = take(nb * 4), o_y = take(nb * N * 8), o_yw = take(nb * N);
  if (total > h->scratch_bytes) {
    if (h->d_scratch) cudaFree(h->d_scratch);
    h->d_scratch = nullptr; h->scratch_bytes = 0;
    cudaError_t e = cudaMalloc(&h->d_scratch, total);
    if (e != cudaSuccess) return cuda_fail(e, "scratch allocation");
    h->scratch_bytes = total;
  }
  unsigned char* base = h->d_scratch;
  cudaError_t e = cudaSuccess;
  auto h2d = [&](const Slice& s, const void* src) {
    if (e == cudaSuccess) e = cudaMemcpyAsync(base + s.off, src, s.bytes, cudaMemcpyHostToDevice, stream);
  };
  h2d(s_node, in->set_node); h2d(s_elem, in->set_element); h2d(s_geo, in->a_geo); h2d(s_topo, in->a_topo);
  h2d(s_mr, in->move_range);
  if (in->coin) h2d(s_coin, in->coin);
  if (e != cudaSuccess) return cuda_fail(e, "host->device copy");
  tfem_step_in din{};
  din.set_node = (const float*)(base + s_node.off); din.set_element = (const float*)(base + s_elem.off);
  din.a_geo = (float*)(base + s_geo.off); din.a_topo = (float*)(base + s_topo.off);
  din.coin = in->coin ? (const uint8_t*)(base + s_coin.off) : nullptr;
  din.move_range = (float*)(base + s_mr.off);
  tfem_step_out dout{};
  // the raw tables are updated in place on the device (read-before-write per environment)
  dout.x_n = out->x_n ? (float*)(base + o_xn.off) : nullptr;
  dout.A_s = out->A_s ? (float*)(base + o_as.off) : nullptr;
  dout.A_n_ts = out->A_n_ts ? (float*)(base + o_ts.off) : nullptr;
  dout.A_n_cs = out->A_n_cs ? (float*)(base + o_cs.off) : nullptr;
  dout.nN_x_n = out->nN_x_n ? (float*)(base + s_node.off) : nullptr;
  dout.nN_x_e = out->nN_x_e ? (float*)(base + s_elem.off) : nullptr;
  dout.point = out->point ? (float*)(base + o_pt.off) : nullptr;
  dout.point64 = out->point64 ? (double*)(base + o_p64.off) : nullptr;
  dout.d = out->d ? (double*)(base + o_d.off) : nullptr;
  dout.axial = out->axial ? (double*)(base + o_ax.off) : nullptr;
  dout.ratio = out->ratio ? (double*)(base + o_ra.off) : nullptr;
  dout.U = out->U ? (double*)(base + o_u.off) : nullptr;
  dout.reactions = out->reactions ? (double*)(base + o_re.off) : nullptr;
  dout.status = out->status ? (int32_t*)(base + o_st.off) : nullptr;
  dout.y = out->y ? (double*)(base + o_y.off) : nullptr;
  dout.y_weak = out->y_weak ? (uint8_t*)(base + o_yw.off) : nullptr;
  tfem::StepArgs a{};
  a.B = B; a.mode = tfem::MODE_STEP; a.in = din; a.out = dout;
  if (int rc = launch(h, a, stream)) return rc;
  auto d2h = [&](void* dst, const void* src, size_t bytes) {
    if (dst && e == cudaSuccess) e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream);
  };
  d2h(in->a_geo, din.a_geo, s_geo.bytes);            // clipped in place, like the reference
  d2h(in->a_topo, din.a_topo, s_topo.bytes);
  d2h(in->move_range, din.move_range, s_mr.bytes);
  d2h(out->x_n, dout.x_n, o_xn.bytes); d2h(out->A_s, dout.A_s, o_as.bytes);
  d2h(out->A_n_ts, dout.A_n_ts, o_ts.bytes); d2h(out->A_n_cs, dout.A_n_cs, o_cs.bytes);
  d2h(out->nN_x_n, dout.nN_x_n, s_node.bytes); d2h(out->nN_x_e, dout.nN_x_e, s_elem.bytes);
  d2h(out->point, dout.point, o_pt.bytes); d2h(out->point64, dout.point64, o_p64.bytes);
  d2h(out->d, dout.d, o_d.bytes); d2h(out->axial, dout.axial, o_ax.bytes); d2h(out->ratio, dout.ratio, o_ra.bytes);
  d2h(out->U, dout.U, o_u.bytes); d2h(out->reactions, dout.reactions, o_re.bytes);
  d2h(out->status, dout.status, o_st.bytes);
  d2h(out->y, dout.y, o_y.bytes); d2h(out->y_weak, dout.y_weak, o_yw.bytes);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  if (e != cudaSuccess) return cuda_fail(e, "device->host copy");
  return TFEM_OK;
}

int64_t tfem_launch_count(tfem_handle_t h) { return h ? h->launches.load() : 0; }
void tfem_book_launches(tfem_handle_t h, int64_t n) { if (h) h->launches.fetch_add(n); }

}  // extern "C"

int tfem::handle_family_count(tfem_handle_t h) { return h ? h->n_families : 0; }
bool tfem::handle_is_mixed(tfem_handle_t h) { return h && h->launch.smem_mixed > 0; }
