/* tfem.h -- C ABI of the B200-native batched 2D-truss FEM environment step.
 *
 * The reference (kupc25648/MOP-truss-MARL) has no FFI: its de-facto operator boundary is the Python
 * module surface the drivers star-import (SURVEY.md section 8b).  Every entry point below names the
 * reference interface it stands in for; INTEGRATION.md shows the ctypes stub a maintainer would add.
 *
 * Conventions
 *   - plain C, no exceptions, no torch / Python types; return value 0 = ok, < 0 = argument or CUDA
 *     error (text via tfem_last_error()); per-environment numerical trouble is reported in status[].
 *   - all buffers are caller-owned, contiguous, 16-byte aligned; "device" pointers are CUDA device
 *     pointers valid on the handle's device, "host" pointers are (preferably pinned) host memory.
 *   - one handle per (GPU, geometry family), or per (GPU, set of families of one topology) for the mixed
 *     entry points; re-entrant per handle; the only hidden state is the families' constant tables.
 *     stream is a cudaStream_t passed as void*.
 *   - B = number of independent environments in the call.  N = 2*num_x nodes, E = 5*num_x-4 elements,
 *     ndof = free DOFs in the reference numbering (FEM_2Dtruss.py:227-261).
 */
#ifndef TFEM_H_
#define TFEM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TFEM_MAX_NX 16
#define TFEM_NSEC 5
#define TFEM_MAX_FAMILIES 16

enum { TFEM_BRIDGE = 0, TFEM_ROOF = 1 };
/* symmetry convention of truss2D_ENV.py: none = train/code, small = test/00,01 (:460-553),
 * large = test/02,03 (:460-673; opposite coin direction, also copies the support column) */
enum { TFEM_SYM_NONE = 0, TFEM_SYM_SMALL = 1, TFEM_SYM_LARGE = 2 };

/* status[] bits */
enum { TFEM_STATUS_OK = 0, TFEM_STATUS_NOT_SPD = 1, TFEM_STATUS_NONFINITE = 2, TFEM_STATUS_BAD_FAMILY = 4 };

/* error codes */
enum {
  TFEM_OK = 0, TFEM_ERR_ARG = -1, TFEM_ERR_CUDA = -2, TFEM_ERR_UNSUPPORTED = -3, TFEM_ERR_ALIGN = -4
};

typedef struct tfem_handle_s* tfem_handle_t;

/* Arguments of truss2D_GEN.gen_model(num_x, num_y, span_x, span_y, tar_y, dmin, loadx, loady,
 * truss_type, support_case, topo_code) (truss2D_GEN.py:42-50) plus the section catalogue it reads
 * from section_data/01_brace_rod2.csv (:60-61).  num_y is always 2, loadx is never applied
 * (Load.set_size(0, loady), :374), topo_code is unused. */
typedef struct tfem_family_desc {
  int32_t num_x;
  int32_t truss_type;                 /* TFEM_BRIDGE | TFEM_ROOF */
  int32_t support_case;               /* 1..4, anything else behaves like 1 (:404-418) */
  int32_t symmetry;                   /* TFEM_SYM_* : which truss2D_ENV.py is being replaced */
  double span_x[TFEM_MAX_NX - 1];
  double span_y;                      /* span_y[0] == y_max */
  double tar_y[TFEM_MAX_NX];
  double d_min;
  double load_y;
  double section_area_cm2[TFEM_NSEC];
  double section_inertia_cm4[TFEM_NSEC];
  double young;                       /* 2e11  (truss2D_GEN.py:59) */
  double allow_stress;                /* 235e6/1.5 (FEM_2Dtruss.py:93-94) */
} tfem_family_desc;

typedef struct tfem_dims {
  int32_t N, E, ndof, nres;           /* nres = 2N - ndof restrained DOFs */
  int32_t num_x, n_internal, band;    /* internal banded system: n_internal = 4*num_x, half-bandwidth */
  int32_t device;                     /* CUDA device of the handle, -1 for a tables-only handle */
} tfem_dims;

/* constant tables (tfem_get_table): what the reference recomputes on every call although it never
 * changes for a topology */
enum {
  TFEM_TAB_CONN = 0,        /* int32 [E,2]   element end nodes, 0-based   (truss2D_GEN.py:280-353) */
  TFEM_TAB_TNSC = 1,        /* int32 [N,2]   1-based DOF ids, free first  (FEM_2Dtruss.py:227-251) */
  TFEM_TAB_RES = 2,         /* int32 [N,2]   restraint flags              (truss2D_GEN.py:400-418) */
  TFEM_TAB_TOP = 3,         /* int32 [N]     top_node                      (:307-310) */
  TFEM_TAB_PAIR = 4,        /* int32 [N]     vertical_pair index           (:312-313) */
  TFEM_TAB_LOADED = 5,      /* int32 [N]     node carries the load         (:421-430) */
  TFEM_TAB_LOADVEC = 6,     /* double [ndof] P in free-DOF order           (FEM_2Dtruss.py:264-280) */
  TFEM_TAB_X = 7,           /* double [N]    node x */
  TFEM_TAB_Y0 = 8,          /* double [N]    generated node y */
  TFEM_TAB_TARGET = 9,      /* double [N]    tar_y on top nodes, 0 elsewhere */
  TFEM_TAB_A_N = 10,        /* float [N,N]   D^-1/2 (A+I) D^-1/2           (truss2D_ENV.py:104-110) */
  TFEM_TAB_MASK = 11,       /* float [N,N]   adjacency                     (:92-93) */
  TFEM_TAB_NC_E = 12,       /* float [E,N]   incidence c_e                 (:181-182) */
  TFEM_TAB_SYM_SRC = 13,    /* int32 [2,N]   y[i] <- y[src]; row 0: coin false, row 1: coin true */
  TFEM_TAB_SYM_ELEM = 14,   /* int32 [E]     symmetric partner element (self if none) */
  TFEM_TAB_INT_OBJ = 15,    /* float [2]     int_obj1, int_obj2             (truss2D_ENV.py:267-277) */
  TFEM_TAB_SCALARS = 16     /* double [8]    y_max, y_min, d_min, max_deformation, young, allow, load_y, 0 */
};

/* Inputs of Game_research04._game_modify(set_node, set_element, nC_e, actions)
 * (truss2D_ENV.py:373).  nC_e is a family constant and is not passed. */
typedef struct tfem_step_in {
  const float* set_node;      /* [B,N,12]  nN_x_n of the parent state; only column 1 (y) is read (:365)  */
  const float* set_element;   /* [B,E,21]  nN_x_e of the parent state; only column 0 (section) (:369)  */
  float* a_geo;               /* [B,N,2]   actions[0], clipped to [0,1] IN PLACE (:379-384) */
  float* a_topo;              /* [B,N,3]   actions[1], clipped to [0,1] IN PLACE (:386-391) */
  const uint8_t* coin;        /* [B]       1 when random.random() >= 0.5 (:460); NULL = all 0 */
  float* move_range;          /* [B,N,2]   in : max_up/max_down left on the model by the previous
                                           call (the reference's hidden state, :405,:410);
                                           out: the range set_moveRange() leaves behind (:557) */
  /* The two table columns _set_model actually reads (:365, :369), as compact arrays.  When non-NULL they are read
   * INSTEAD of set_node / set_element (which may then be NULL): a caller that keeps the state on the host uploads
   * 4 (N + E) bytes per environment instead of the 4 (12 N + 21 E) of the full tables (trollout_step_host). */
  const float* set_node_y;          /* [B,N]  = set_node[:, :, 1] */
  const float* set_element_section; /* [B,E]  = set_element[:, :, 0] */
} tfem_step_in;

/* Everything _game_modify returns (point, St_S) plus the FP64 fields of the solved model.
 * Any pointer may be NULL (that output is skipped).  set_node/set_element may alias the outputs
 * nN_x_n/nN_x_e (in-place state update). */
typedef struct tfem_step_out {
  float* x_n;        /* [B,N,13]  normalised node features      (state_data, truss2D_ENV.py:43-112) */
  float* A_s;        /* [B,N,N]   section-size adjacency */
  float* A_n_ts;     /* [B,N,N]   tension stress-ratio adjacency */
  float* A_n_cs;     /* [B,N,N]   compression stress-ratio adjacency */
  float* nN_x_n;     /* [B,N,12]  raw node table                (state_data_not_norm, :115-196) */
  float* nN_x_e;     /* [B,E,21]  raw element table */
  float* point;      /* [B,4]     obj1/int_obj1, obj2/int_obj2, con1, con2 (float32, :566-587) */
  double* point64;   /* [B,4]     obj1, obj2, con1, con2 without any float32 rounding (not normalised) */
  double* d;         /* [B,ndof]  Model.d in the reference DOF order (FEM_2Dtruss.py:337) */
  double* axial;     /* [B,E]     Element.e_q[0][0], + = compression (:383-386) */
  double* ratio;     /* [B,E]     Element.prop_yeield (:414-431) */
  double* U;         /* [B]       Model.U_full (:374-379) */
  double* reactions; /* [B,nres]  Model.r at the restrained DOFs (:393-411) */
  int32_t* status;   /* [B]       TFEM_STATUS_* bits */
  double* y;         /* [B,N]     node.coord[1] after the transition, as float(...) of what the reference holds */
  uint8_t* y_weak;   /* [B,N]     1 where the reference holds a python int/float (assigned by a constraint
                                  pass or a support), 0 where it holds an np.float32 */
  float* node_y;          /* [B,N]  = nN_x_n[:, :, 1] of the child state (the next call's set_node_y) */
  float* element_section; /* [B,E]  = nN_x_e[:, :, 0] of the child state (the next call's set_element_section) */
} tfem_step_out;

const char* tfem_version(void);
const char* tfem_last_error(void);

/* gen_model(...) + Game_research04(...): builds the mesh, supports, loads, DOF map, symmetry tables
 * and the initial objectives for one family on CUDA device `device`.  device < 0 gives a tables-only
 * handle (tfem_get_dims / tfem_get_table work, every compute entry point returns TFEM_ERR_CUDA).
 * Families: 3 <= num_x <= TFEM_MAX_NX (one kernel lane per node; num_x = 2 leaves no free bottom node to carry
 * a load) with TFEM_SYM_NONE, the ENV of train/code; the small and large symmetry conventions only for
 * num_x 6, 8 and 16, the chord lengths whose truss2D_ENV.py carries their index lists.  Anything else
 * returns TFEM_ERR_UNSUPPORTED, and tfem_last_error names the limit. */
int tfem_create(const tfem_family_desc* desc, int device, tfem_handle_t* out);
int tfem_destroy(tfem_handle_t h);
int tfem_get_dims(tfem_handle_t h, tfem_dims* out);
int tfem_get_table(tfem_handle_t h, int which, void* host_dst, size_t bytes);

/* Game_research04._game_get_1_state() on the freshly generated geometry (truss2D_ENV.py:339-354),
 * replicated for B environments.  move_range_out [B,N,2] receives set_moveRange()'s result. */
int tfem_reset(tfem_handle_t h, int B, float* move_range_out, const tfem_step_out* out, void* stream);

/* Game_research04._game_modify (truss2D_ENV.py:373-589) for B independent environments. */
int tfem_step(tfem_handle_t h, int B, const tfem_step_in* in, const tfem_step_out* out, void* stream);

/* Model.restore(); Model.gen_all() only (FEM_2Dtruss.py:434-459) on explicit FP64 geometry:
 * y [B,N] double, section [B,E] int32 -> d, axial, ratio, U, reactions, status (any may be NULL). */
int tfem_solve_only(tfem_handle_t h, int B, const double* y, const int32_t* section,
                    double* d, double* axial, double* ratio, double* U, double* reactions,
                    int32_t* status, void* stream);

/* The solve of tfem_solve_only in the formulation BASELINE.json's north_star names for the large meshes: K assembled
 * dense in the reference's own free-DOF order (FEM_2Dtruss.py:227-261, 310-324) and factored by a blocked (8-wide)
 * right-looking Cholesky whose trailing updates run on the FP64 tensor cores (mma.sync.m8n8k4.f64 = DMMA), one CTA
 * per environment.  Kept as a measured alternative to the banded production solve (DESIGN.md section 3.1); d [B,ndof]
 * in reference DOF order, status bit 0 = non-positive pivot.  Assembly uses shared-memory atomics, so the last bits
 * of d depend on the order of the element contributions. */
int tfem_solve_dense_dmma(tfem_handle_t h, int B, const double* y, const int32_t* section, double* d,
                          int32_t* status, void* stream);

/* Gene-vector objective of the MOEA/D benchmark: gen_model.read_genes(genes, int_obj1, int_obj2)
 * (test/benchmarks/MOEAD/<family>.zip:<family>/truss2D_GEN.py:117-228, one call per individual from
 * MOEAD_master.py:103-121) for B individuals in ONE launch of the env-step kernel (gene decode, forced symmetry,
 * FEM, objectives).  genes [B,N+E] float64 in [0,1]: the first N scale to node heights (x max_height: 8 in the small
 * zips, 6 in the large ones, truss2D_GEN.py:127), the last E to section numbers min(4, round(4 g)).  Everything is
 * float64 like the reference (python floats); point [B,4] float32 is what read_genes returns.  int_obj1/int_obj2 <= 0
 * select the family's own initial objectives (what MOEAD_master.py:53-64 computes).  The reference keeps one
 * persistent model, but every node read_genes does not assign ends each call at its generated height, so the call
 * is pure.  Genes outside [0,1] clamp the section to 0..4 (the reference would index the catalogue from the end).
 * Any output may be NULL. */
typedef struct tfem_genes_out {
  float* point;      /* [B,4]   obj1/int_obj1, obj2/int_obj2, con1, con2 */
  double* point64;   /* [B,4]   the same four without float32 rounding, not normalised */
  double* y;         /* [B,N]   decoded node heights */
  int32_t* section;  /* [B,E]   decoded section numbers */
  double* d;         /* [B,ndof] */
  double* axial;     /* [B,E] */
  double* ratio;     /* [B,E] */
  double* U;         /* [B] */
  double* reactions; /* [B,nres] */
  int32_t* status;   /* [B] */
} tfem_genes_out;
int tfem_read_genes(tfem_handle_t h, int B, const double* genes, double max_height, float int_obj1, float int_obj2,
                    const tfem_genes_out* out, void* stream);

/* Same call as tfem_step with HOST buffers (the reference's calling convention: numpy arrays in,
 * numpy arrays out).  Copies inputs host->device, runs the step, copies every non-NULL output back
 * and synchronises the stream before returning.  Scratch device memory is owned by the handle. */
int tfem_step_host(tfem_handle_t h, int B, const tfem_step_in* in_host, const tfem_step_out* out_host,
                   void* stream);

/* Mixed-family batches: the reference's training driver draws one of the five 6 x 2 shapes and a truss type for
 * every episode (train/code/master_DDPG_truss2D_MO.py:787-815), so B episodes run in parallel form a batch of mixed
 * families.  tfem_create_mixed builds one handle from n_families (1..TFEM_MAX_FAMILIES) descriptions that share the
 * topology: num_x (mesh, element order, output maps) and the DOF map that support_case fixes (TNSC, RES tables).  A
 * mismatch returns TFEM_ERR_UNSUPPORTED with the name of the differing table.  Everything else (spans, span_y, tar_y,
 * d_min, load_y, truss type, symmetry convention, sections, young, allow_stress) may differ.  The large meshes fit
 * fewer families per launch than the small ones: a count that would lower the kernel's CTAs per SM is refused with
 * TFEM_ERR_UNSUPPORTED and the limit in the error text.  device < 0 gives a tables-only handle, as for tfem_create.
 *
 * family [B] (device, uint8) holds one index into descs per environment; it is an input of every call and is not
 * kept by the handle.  Environment b is tfem_reset / tfem_step of family family[b]: the same outputs, the same
 * point normalisation by that family's int_obj, the same status bits.  An index >= n_families sets
 * status[b] = TFEM_STATUS_BAD_FAMILY and writes nothing else for that environment.
 *
 * With n_families == 1 the handle also serves every single-family entry point, exactly like tfem_create.  With more
 * families those (tfem_reset, tfem_step, tfem_solve_only, tfem_read_genes, tfem_step_host, tfem_solve_dense_dmma)
 * return TFEM_ERR_ARG, and tfem_get_table serves only the topology tables (CONN, TNSC, RES, TOP, PAIR, A_N, MASK,
 * NC_E); a tables-only handle of one family serves the others. */
int tfem_create_mixed(const tfem_family_desc* descs, int n_families, int device, tfem_handle_t* out);
int tfem_reset_mixed(tfem_handle_t h, int B, const uint8_t* family, float* move_range_out, const tfem_step_out* out,
                     void* stream);
int tfem_step_mixed(tfem_handle_t h, int B, const uint8_t* family, const tfem_step_in* in, const tfem_step_out* out,
                    void* stream);

/* number of kernels this library launched on behalf of the handle since creation; tfem_book_launches adds kernel
 * launches that were replayed from a CUDA graph captured around tfem_step (trollout_step_host) */
int64_t tfem_launch_count(tfem_handle_t h);
void tfem_book_launches(tfem_handle_t h, int64_t n);

#ifdef __cplusplus
}
#endif
#endif /* TFEM_H_ */
