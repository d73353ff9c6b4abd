// invmgmt_jit.cuh -- run-time specialisation of the serial multi-echelon env's fused rollout (see invmgmt_jit.cu)
#pragma once
#include <string>
#include <vector>

#include "common.cuh"
#include "invmgmt_jit_args.cuh"

struct InvJitSpec {  // host-side copy of everything the generator bakes into the kernel
    int n, T, backlog;
    int L[ORGYM_INV_MAX_STAGES];
    long long c[ORGYM_INV_MAX_STAGES], I0[ORGYM_INV_MAX_STAGES];
    double up[ORGYM_INV_MAX_STAGES + 1], uc[ORGYM_INV_MAX_STAGES + 1], kc[ORGYM_INV_MAX_STAGES + 1],
        hc[ORGYM_INV_MAX_STAGES + 1];
    std::vector<double> disc;  // alpha**t
    int log2k, base;           // alias table geometry of the demand distribution
    long long xbound;          // bound on |on-hand|, |backlog|, |sales| of any stage in any period (0 = unknown)
    // per-term bounds behind the exactness proof (0 <= j <= n): |units sold by stage j| (retail sales, fulfilled order
    // of stage j-1), on-hand inventory above zero, unfulfilled quantity.  profit_mag() = sum_j coefficient x bound.
    double sale_bound[ORGYM_INV_MAX_STAGES + 1], inv_bound[ORGYM_INV_MAX_STAGES + 1], unf_bound[ORGYM_INV_MAX_STAGES + 1];
    // sign facts from the same proof: stage i's on-hand inventory after any period is >= 0 (its clamp at 0 is dropped)
    bool inv_nonneg[ORGYM_INV_MAX_STAGES];
    // policy baked into the kernel: 0 = base-stock with the integer levels `target`, 1 = uniform random orders
    int policy;
    long long target[ORGYM_INV_MAX_STAGES];
};
// bound on the sum of |terms| of one period's profit (so also on every partial sum in any evaluation order)
double inv_jit_profit_mag(const InvJitSpec& S);
// log2 of the finest quantum Q all price / cost coefficients are integer multiples of; false if a coefficient is not a
// finite non-negative float32 value
bool inv_jit_quantum(const InvJitSpec& S, int* qexp);
// true when every float64 operation of a period's profit is exact (see invmgmt_jit.cu); `periods` > 1 asks the same
// for the running sum of that many undiscounted period profits
bool inv_jit_profit_is_exact(const InvJitSpec& S, int periods = 1);
#define INV_JIT_THREADS 128
// configurations the generator covers (everything else runs the ahead-of-time kernel)
bool inv_jit_eligible(const InvJitSpec& S);
// complete translation unit with ONE kernel, `inv_jit_rollout_bs` (S.policy == 0: base-stock, the levels are literals)
// or `inv_jit_rollout_rnd` (S.policy == 1)
std::string inv_jit_source(const InvJitSpec& S);
const char* inv_jit_kernel_name(int policy);
