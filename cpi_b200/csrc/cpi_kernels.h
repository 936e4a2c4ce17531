// Kernel parameter blocks and host-side launchers shared by capi.cu and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cpi {

struct PreintParams {
    int64_t n_windows;
    const int64_t* offsets;   // device, may be null (uniform windows)
    int64_t ns_uniform;
    const void* samples;      // device, double (dtype 64) or float (dtype 32)
    const void* lin;          // device
    void* out;                // device
    const void* init;         // device, may be null: records holding the state to CONTINUE from (may alias `out`); tri-lane kernels only
    double q_w, q_wb, q_a, q_ab;   // sigma^2  (CpiBase.h:54-57)
    int wpb;                  // windows per block; 0 on entry = let preint_launch choose (one wave if possible)
};

struct FactorParams {
    int64_t n;
    const double* states;
    const int64_t* idx_i;
    const int64_t* idx_j;
    const double* records;
    const double* lin;
    double* e;
    double* H1;
    double* H2;
};

int preint_pick_wpb(int model, int dtype, int64_t n_windows, int num_sms);
int preint_ws_cap(int dtype);
int preint_cap(int model, int dtype, int flags, int num_sms);
// tri-lane kernels (preintegrate_tri.cu)
bool preint_tri_supported(int model, int flags);
int preint_tri_cap(int model, int dtype);
cudaError_t preint_launch_tri(int model, int dtype, const PreintParams& p, int num_sms, cudaStream_t st);
cudaError_t preint_launch(int model, int dtype, int flags, const PreintParams& p0, int num_sms, int max_smem_bytes, cudaStream_t st, int* launches);
cudaError_t factor_launch(int model, const FactorParams& p, cudaStream_t st);
cudaError_t predict_launch(int model, int64_t n, const double* states, const double* records, const double* lin, double* out, cudaStream_t st);
cudaError_t hessian_launch(int rd, int64_t n, const double* records, const double* e, const double* H1, const double* H2,
                           double* G11, double* G12, double* G22, double* g1, double* g2, double* f, cudaStream_t st);
cudaError_t whiten_launch(int rd, int64_t n, const double* records, const double* e, const double* H1, const double* H2, double* A1, double* A2, double* b, cudaStream_t st);
cudaError_t chain_assemble_launch(int64_t nf, const double* G11, const double* G12, const double* G22, const double* g1, const double* g2, double lambda,
                                  int diagonal_damping, const double* prior_info, const double* prior_rhs, double* D, double* E, double* rhs, cudaStream_t st);
int64_t chain_solve_workspace_bytes(int64_t n_states);
cudaError_t chain_solve_launch(int64_t n_states, const double* D, const double* E, const double* b, double* x, double* ws, cudaStream_t st, int* launches);
cudaError_t chain_marginals_launch(int64_t n_states, const double* D, const double* E, double* S_diag, double* S_off, double* ws, cudaStream_t st,
                                   int* launches);
cudaError_t retract_launch(int64_t n, const double* states, const double* xi, double* out, cudaStream_t st);

}  // namespace cpi
