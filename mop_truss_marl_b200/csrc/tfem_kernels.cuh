// Launch interface between the C ABI (tfem_capi.cu) and the device code (tfem_kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include "tfem_family.h"

namespace tfem {

enum StepMode { MODE_STEP = 0, MODE_RESET = 1, MODE_SOLVE_ONLY = 2, MODE_GENES = 3 };

struct StepArgs {
  const FamilyTables* fam;     // device copy; n_families consecutive tables for the mixed launches
  const uint16_t* maps;        // device copy of Family::maps
  int map_entries;             // padded to a multiple of 8
  int B;
  int mode;
  tfem_step_in in;             // device pointers (MODE_STEP)
  tfem_step_out out;           // device pointers
  const double* so_y;          // MODE_SOLVE_ONLY: [B,N]
  const int32_t* so_sec;       // MODE_SOLVE_ONLY: [B,E]
  float* reset_move_range;     // MODE_RESET: [B,N,2]
  const double* genes;         // MODE_GENES: [B,N+E]
  double max_height;           // MODE_GENES
  int32_t* sec_out;            // MODE_GENES: decoded sections [B,E] (optional)
  float int_obj1, int_obj2;    // > 0: normalisers of point[0], point[1] instead of the family's
  const uint8_t* family;       // mixed launches (MODE_STEP / MODE_RESET): [B] index into fam[]
  int n_families;              // mixed launches: entries of fam[]
};

struct LaunchInfo {
  int grid, block, smem_bytes, ctas_per_sm, grid_genes;
  int smem_mixed;              // dynamic shared memory of the mixed-family launch (0: not configured)
};

// one-time per-handle setup (opt-in shared memory, occupancy query); returns cudaError_t as int
int step_kernel_configure(int nx, int device, int map_entries, LaunchInfo* info);
// additionally configures the mixed-family kernel for n_families tables.  *max_families receives the most families that
// keep the single-family kernel's CTAs per SM; the caller refuses n_families above it (info->smem_mixed is then 0).
int step_kernel_configure_mixed(int nx, int map_entries, int n_families, LaunchInfo* info, int* max_families);
// args.family != nullptr selects the mixed-family kernel
int step_kernel_launch(int nx, const StepArgs& args, const LaunchInfo& info, cudaStream_t stream);

// families staged by a handle (tfem_create_mixed); internal to the library, not part of the C ABI
__attribute__((visibility("hidden"))) int handle_family_count(tfem_handle_t h);
// the handle has the mixed-family kernel configured (made by tfem_create_mixed on a device): tfem_step_mixed serves it
__attribute__((visibility("hidden"))) bool handle_is_mixed(tfem_handle_t h);

// dense blocked Cholesky with DMMA trailing updates (tfem_dense.cu); returns cudaError_t as int
int dense_solve_launch(const FamilyTables* d_tables, int B, const double* y, const int32_t* section, double* d,
                       int32_t* status, cudaStream_t stream);

}  // namespace tfem
