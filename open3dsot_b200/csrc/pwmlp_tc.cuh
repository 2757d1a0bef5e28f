// Tensor-core GEMM entry points (pwmlp_tc.cu) that only the stack sequencer (stack.cu) calls; arguments as in the
// o3d_pw_*_tc entry points of include/o3d_b200.h.
//
// rev != 0: the forward kernel walks the position tiles from the last to the first.  The stack alternates the direction
// from layer to layer, so that a layer starts on the rows the previous kernel touched last, which are still in L2.  The
// public o3d_pw_fwd_tc always walks forward, and so does every dgrad.
#pragma once
#include <stdint.h>
#include "../../include/o3d_b200.h"

int pw_fwd_tc(const float* x, int ldx, const float* in_scale, const float* in_shift, int in_relu, const void* wtiles,
              const float* bias, int P, int K, int N, float* y, int ldy, double* sum, double* sumsq, int S, float* ymax,
              float* ymin, int32_t* arg, int ldp, int rev, void* stream);

// The GEMMs of the layer AFTER a lifted first layer (o3d_lift_t): they read Y0 through gidx, so Y0 is never stored.
// pw_wgrad_tc_lift runs the split-K kernel of o3d_pw_wgrad_tc2; `part` (part_floats = o3d_pw_wgrad_tc2_workspace_floats()
// floats) is required.
int pw_fwd_tc_lift(const o3d_lift_t* lf, const int32_t* gidx, const float* in_scale, const float* in_shift, int in_relu,
                   const void* wtiles, const float* bias, int P, int K, int N, float* y, int ldy, double* sum, double* sumsq,
                   int S, float* ymax, float* ymin, int32_t* arg, int ldp, int rev, void* stream);
int pw_dgrad_tc_lift(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                     const float* dpool, const int32_t* sel, int S, int ldp, const void* wtiles_t, int P, int Cout, int Cin,
                     float* out, int ldo, const o3d_lift_t* lf, const int32_t* gidx, const float* pscale, const float* pshift,
                     int prelu, double* s1, double* s2y, void* stream);
int pw_wgrad_tc_lift(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                     const float* dpool, const int32_t* sel, int S, int ldp, const o3d_lift_t* lf, const int32_t* gidx,
                     const float* in_scale, const float* in_shift, int in_relu, int P, int Cout, int Cin, float* dw, int lddw,
                     float* part, long long part_floats, void* stream);
