// mlp.cuh -- the MLP actor (orgym_mlp_t) shared by the fused rollout kernels of the serial env (inv_mlp_rollout_kernel)
// and the newsvendor (nv_mlp_rollout_kernel).
//
// A CTA of MLP_THREADS threads stages the weights in shared memory once and evaluates the network on a sub-tile of E
// envs per period.  Activations are feature-major [feature][env] float32 tiles; a hidden layer is a register-tiled SGEMM
// in which each thread computes blocks of MLP_TE envs x MLP_TN neurons, so one 16-byte load of activations and one of
// weights feed 16 FMAs.  Every output accumulates in ascending k from its bias with __fmaf_rn (the numerics contract
// of orgym_mlp_t in the header), so the result does not depend on E or on the tiling.
//
// The host half validates an orgym_mlp_t against the env's (obs_dim, act_dim) and lays out the weights; each env family
// adds its own observation tile, activation buffers and state to the shared-memory plan.
#pragma once
#include <algorithm>

#include "common.cuh"

#define MLP_THREADS 256
#define MLP_TE 4
#define MLP_TN 4
#define MLP_SMEM_BUDGET (227 * 1024 - 1024)  // sm_100 opt-in limit per block, less the static partial-sum rows

// The network and the layout of its weights in the float area of shared memory (offsets in floats, 16-byte aligned):
// hidden layer l as Wt[k][Np[l]] (transposed, output columns zero-padded to MLP_TN) with a zero-padded bias, the last
// layer as given ([K[L]][K[L-1]] row-major).
struct MlpNet {
    int L, act;
    int K[ORGYM_MLP_MAX_LAYERS + 1];  // widths
    int Np[ORGYM_MLP_MAX_LAYERS];     // output widths of the hidden layers padded to MLP_TN (zero weights and biases)
    const float* W[ORGYM_MLP_MAX_LAYERS];
    const float* b[ORGYM_MLP_MAX_LAYERS];
    int w_off[ORGYM_MLP_MAX_LAYERS], b_off[ORGYM_MLP_MAX_LAYERS];
    int wfloats, hmax;  // floats of all weights and biases; widest padded hidden layer (0 without one)
};

__device__ __forceinline__ float mlp_act(float x, int act) {
    // accurate tanhf (tanh.approx.f32 has ~2^-11 relative error: far more truncated actions would flip); ReLU keeps NaN
    return act == ORGYM_MLP_TANH ? tanhf(x) : (x < 0.f ? 0.f : x);
}

// out[n][e] = act(b[n] + sum_k Wt[k][n] in[k][e]) for the E envs of the tile; each output accumulates in k order
__device__ __forceinline__ void mlp_hidden_layer(const float* __restrict__ in, float* __restrict__ out,
                                                 const float* __restrict__ Wt, const float* __restrict__ bias, int K,
                                                 int Np, int E, int log2E, int act) {
    const int egs = E / MLP_TE, log2egs = log2E - 2;
    const int ntile = egs * (Np / MLP_TN);
    for (int tile = threadIdx.x; tile < ntile; tile += MLP_THREADS) {
        const int eg = tile & (egs - 1), ng = tile >> log2egs;
        const float* xp = in + eg * MLP_TE;
        const float* wp = Wt + ng * MLP_TN;
        const float4 bv = *reinterpret_cast<const float4*>(bias + ng * MLP_TN);
        float acc[MLP_TE][MLP_TN];
#pragma unroll
        for (int i = 0; i < MLP_TE; i++) {
            acc[i][0] = bv.x;
            acc[i][1] = bv.y;
            acc[i][2] = bv.z;
            acc[i][3] = bv.w;
        }
#pragma unroll 4
        for (int k = 0; k < K; k++) {
            const float4 x4 = *reinterpret_cast<const float4*>(xp + k * E);
            const float4 w4 = *reinterpret_cast<const float4*>(wp + k * Np);
            const float x[4] = {x4.x, x4.y, x4.z, x4.w}, w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
            for (int i = 0; i < MLP_TE; i++)
#pragma unroll
                for (int j = 0; j < MLP_TN; j++) acc[i][j] = __fmaf_rn(w[j], x[i], acc[i][j]);
        }
#pragma unroll
        for (int j = 0; j < MLP_TN; j++)
            *reinterpret_cast<float4*>(out + (ng * MLP_TN + j) * E + eg * MLP_TE) =
                make_float4(mlp_act(acc[0][j], act), mlp_act(acc[1][j], act), mlp_act(acc[2][j], act),
                            mlp_act(acc[3][j], act));
    }
}

// Copies the weights and biases from global memory into the float area fs of shared memory, laid out as MlpNet says.
// M is an MlpNet or a plan with the same fields (L, K, Np, W, b, w_off, b_off).
template <class Plan>
__device__ __forceinline__ void mlp_stage_weights(const Plan& M, float* fs) {
    const int tid = threadIdx.x;
    for (int l = 0; l < M.L; l++) {
        const int Kl = M.K[l], Nl = M.K[l + 1];
        const float* Wg = M.W[l];
        const float* bg = M.b[l];
        float* Ws = fs + M.w_off[l];
        float* bs = fs + M.b_off[l];
        if (l < M.L - 1) {
            const int Np = M.Np[l];
            for (int idx = tid; idx < Kl * Np; idx += MLP_THREADS) {
                const int k = idx / Np, j = idx - k * Np;
                Ws[idx] = j < Nl ? Wg[(size_t)j * Kl + k] : 0.f;
            }
            for (int j = tid; j < Np; j += MLP_THREADS) bs[j] = (j < Nl && bg) ? bg[j] : 0.f;
        } else {
            for (int idx = tid; idx < Kl * Nl; idx += MLP_THREADS) Ws[idx] = Wg[idx];
            for (int j = tid; j < Nl; j += MLP_THREADS) bs[j] = bg ? bg[j] : 0.f;
        }
    }
}

// Checks a non-null orgym_mlp_t against the env's observation and action widths (ORGYM_E_INVALID with the reason) and
// lays out its weights.  act_what names the action width in the error message.
static int mlp_net_plan(const orgym_mlp_t* mlp, int obs_dim, int act_dim, const char* act_what, MlpNet* M) {
    const int L = mlp->num_layers;
    ORGYM_REQUIRE(L >= 1 && L <= ORGYM_MLP_MAX_LAYERS, "mlp: num_layers = %d, must be 1..%d", L, ORGYM_MLP_MAX_LAYERS);
    ORGYM_REQUIRE(L == 1 || mlp->activation == ORGYM_MLP_TANH || mlp->activation == ORGYM_MLP_RELU,
                  "mlp: activation %d is neither ORGYM_MLP_TANH nor ORGYM_MLP_RELU", mlp->activation);
    for (int l = 0; l <= L; l++)
        ORGYM_REQUIRE(mlp->width[l] >= 1 && mlp->width[l] <= ORGYM_MLP_MAX_WIDTH, "mlp: width[%d] = %d outside 1..%d", l,
                      mlp->width[l], ORGYM_MLP_MAX_WIDTH);
    ORGYM_REQUIRE(mlp->width[0] == obs_dim, "mlp: width[0] = %d differs from obs_dim = %d", mlp->width[0], obs_dim);
    ORGYM_REQUIRE(mlp->width[L] == act_dim, "mlp: width[%d] = %d differs from %s = %d", L, mlp->width[L], act_what,
                  act_dim);
    for (int l = 0; l < L; l++) ORGYM_REQUIRE(mlp->weight_dev[l], "mlp: weight_dev[%d] is NULL", l);
    memset(M, 0, sizeof(*M));
    M->L = L;
    M->act = L > 1 ? mlp->activation : ORGYM_MLP_TANH;
    for (int l = 0; l <= L; l++) M->K[l] = mlp->width[l];
    for (int l = 0; l < L; l++) {
        M->W[l] = mlp->weight_dev[l];
        M->b[l] = mlp->bias_dev[l];
        if (l < L - 1) {
            M->Np[l] = (int)round_up(M->K[l + 1], MLP_TN);
            M->hmax = std::max(M->hmax, M->Np[l]);
        }
    }
    int f = 0;
    for (int l = 0; l < L; l++) {
        M->w_off[l] = f;
        f += (int)round_up(M->K[l] * (l < L - 1 ? M->Np[l] : M->K[l + 1]), 4);  // float offsets stay 16-byte aligned
        M->b_off[l] = f;
        f += (int)round_up(l < L - 1 ? M->Np[l] : M->K[l + 1], 4);
    }
    M->wfloats = f;
    return ORGYM_OK;
}
