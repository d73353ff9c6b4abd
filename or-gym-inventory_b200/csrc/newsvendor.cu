// newsvendor.cu -- multi-period newsvendor with lead time (reference: newsvendor.py).
//
//   nv_reset_kernel    reset (newsvendor.py:100-123): five-uniform parameter recipe from the env's Philox stream
//   nv_step_kernel     one period (:125-204) + observation (:206-208)
//   nv_rollout_kernel  fused reset + step_limit periods with on-device drivers (order-up-to, classic newsvendor,
//                      (s,S)) and per-env Poisson demand (PTRS / inversion)
//   nv_mlp_rollout_kernel  the same fused rollout with an MLP actor evaluated on the device every period
//
// The reward is a chain of mixed float32 / float64 / Python-float operations whose precision depends on which
// branch produced each operand (NumPy >= 2 promotion rules); `Sc` carries the operand kind so the chain is
// reproduced bit for bit.  Pipeline state is float32 like the reference's `state` vector.
#include "common.cuh"
#include "launch_util.cuh"
#include "mlp.cuh"
#include "poisson_mu.cuh"

#define NV_MAXL ORGYM_NV_MAX_LEAD
#define NV_STEP_MINB 8
#define NV_ROLL_MINB 5

struct NvDev {
    const double* rcp;  // reciprocal table (orgym_rcp_table)
    PoisTabDev pt;      // alias tables of the demand sampler (orgym_poisson_tables)
    int L, T, obs_dim;
    double max_inv, max_q, p_max, h_max, k_max, mu_max;
};

struct NvHandle {
    HandleBase base;
    NvDev dev;
    int64_t npad;
    std::vector<void*> allocs;
    double* partials;
};

// state layout (field[slot][env], stride npad): [key u64][params f64 x5][pipe f32 x L][step i32][episode u32]
// Bit 31 of the episode word marks an env whose parameters were pinned by reset(options={'fixed_params': ...}): its
// automatic resets keep them (benchmark_newsvendor_sb3_rllib.py:276-291 re-applies fixed_params on every reset)
// instead of drawing new ones.  The Philox counters use the low 31 bits only.
#define NV_EP_FIXED 0x80000000u
struct NvState {
    uint64_t* key;
    double* par;
    float* pipe;
    int32_t* step;
    uint32_t* episode;
    int64_t npad;
    __host__ __device__ NvState(void* base, int64_t npad_, int L) : npad(npad_) {
        char* p = (char*)base;
        key = (uint64_t*)p;
        p += 8 * npad;
        par = (double*)p;
        p += 8 * 5 * npad;
        pipe = (float*)p;
        p += 4 * (size_t)L * npad;
        step = (int32_t*)p;
        p += 4 * npad;
        episode = (uint32_t*)p;
    }
};
static int64_t nv_state_bytes(int64_t npad, int L) { return npad * (8 + 40 + 4 * (int64_t)L + 8); }

// ---- numpy scalar kinds (NEP 50): PY = Python int/float (weak), F32 = np.float32, F64 = np.float64 -----------------
enum { K_PY = 0, K_F32 = 1, K_F64 = 2 };
struct Sc {
    double v;
    int k;
};
__device__ __forceinline__ Sc mk(double v, int k) {
    Sc s;
    s.v = v;
    s.k = k;
    return s;
}
// Result kind = max(kind a, kind b) (PY < F32 < F64): float64 wins, two Python scalars stay Python (float64 arithmetic),
// anything else is float32.  Branch-free: both precisions are computed and one is selected -- the kinds differ from
// lane to lane (they depend on which operand a min/max picked), so branches would diverge anyway.
__device__ __forceinline__ Sc sc_mul(Sc a, Sc b) {
    const double r64 = a.v * b.v;
    const double r32 = (double)((float)a.v * (float)b.v);
    const int k = a.k > b.k ? a.k : b.k;
    return mk(k == K_F32 ? r32 : r64, k);
}
__device__ __forceinline__ Sc sc_sub(Sc a, Sc b) {
    const double r64 = a.v - b.v;
    const double r32 = (double)((float)a.v - (float)b.v);
    const int k = a.k > b.k ? a.k : b.k;
    return mk(k == K_F32 ? r32 : r64, k);
}

struct NvParams {
    double price, cost, h, k, mu;
};

// newsvendor.py:105-111 from five uniforms
__device__ __forceinline__ NvParams nv_draw_params(const NvDev& P, uint64_t key, uint32_t episode) {
    uint4 b0 = philox_block(key, 0u, episode, STREAM_PARAMS, 0u);
    uint4 b1 = philox_block(key, 1u, episode, STREAM_PARAMS, 0u);
    uint4 b2 = philox_block(key, 2u, episode, STREAM_PARAMS, 0u);
    double u0 = u53(b0.x, b0.y), u1 = u53(b0.z, b0.w), u2 = u53(b1.x, b1.y), u3 = u53(b1.z, b1.w), u4 = u53(b2.x, b2.y);
    NvParams q;
    double x = u0 * P.p_max;
    q.price = x > 1.0 ? x : 1.0;  // max(1, .)
    x = u1 * q.price;
    q.cost = x > 1.0 ? x : 1.0;
    q.h = u2 * (P.h_max < q.cost ? P.h_max : q.cost);  // min(cost, h_max)
    q.k = u3 * P.k_max;
    q.mu = u4 * P.mu_max;
    return q;
}

// fp32 np.sum over the logical pipeline (oldest first); get(j) returns element j
template <typename F>
__device__ __forceinline__ float nv_pipe_sum(int L, F get) {
    if (L < 8) {
        float r = 0.0f;
        for (int j = 0; j < L; j++) r = r + get(j);
        return r;
    }
    float r[8];
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = get(j);
    int full = L - (L % 8), i = 8;
    for (; i < full; i += 8) {
#pragma unroll
        for (int j = 0; j < 8; j++) r[j] = r[j] + get(i + j);
    }
    float res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < L; i++) res = res + get(i);
    return res;
}

// one period (newsvendor.py:125-204).  pipe0 = state[5] (arriving now), psum = fp32 sum of the pipeline.
// returns the reward; *oq_out = order actually placed (float32 value stored in the pipeline); parts optional.
__device__ __forceinline__ double nv_period(const NvDev& P, const NvParams& q, float action, long long demand, float pipe0,
                                            float psum, float* oq_out, double* parts, double* su_out, double* ex_out,
                                            double* sh_out) {
    double a = (double)action;                        // .item() -> Python float (:131)
    a = a < 0.0 ? 0.0 : (a > P.max_q ? P.max_q : a);  // np.clip -> np.float64 (:132)
    Sc order = mk(a, K_F64);
    Sc inv = P.L > 0 ? mk((double)pipe0, K_F32) : order;     // :136-139
    Sc cap = mk((double)((float)P.max_inv - psum), K_F32);   // int - np.float32 -> float32 (:143)
    Sc mn = cap.v < order.v ? cap : order;                   // min(order_qty, cap)
    Sc oq = mn.v > 0.0 ? mn : mk(0.0, K_PY);                 // max(0, .)
    Sc dem = mk((double)demand, K_PY);
    Sc su = dem.v < inv.v ? dem : inv;                       // min(inv_on_hand, demand) (:149)
    Sc rev = sc_mul(su, mk(q.price, K_PY));                  // :150
    Sc ex = sc_sub(inv, dem);
    Sc exs = ex.v > 0.0 ? ex : mk(0.0, K_PY);                // :152
    Sc sh = sc_sub(dem, inv);
    Sc shs = sh.v > 0.0 ? sh : mk(0.0, K_PY);                // :153
    Sc pc = sc_mul(oq, mk(q.cost, K_PY));                    // :162
    Sc hc = sc_mul(exs, mk(q.h, K_PY));                      // :166
    Sc lp = sc_mul(shs, mk(q.k, K_PY));                      // :167
    Sc rew = sc_sub(sc_sub(sc_sub(rev, pc), hc), lp);        // :170
    *oq_out = (float)oq.v;                                   // new_pipeline[-1] = order_qty (:179)
    if (parts) {
        parts[0] = rev.v;
        parts[1] = pc.v;
        parts[2] = hc.v;
        parts[3] = lp.v;
    }
    if (su_out) {
        *su_out = su.v;
        *ex_out = exs.v;
        *sh_out = shs.v;
    }
    return rew.v;
}

// The same period for lead_time > 0 with the kind logic resolved by hand instead of carried through every operation.
// With L > 0 the operand kinds are fixed up to four predicates (Sc notation of nv_period above):
//   inv = F32 (state[5]);  order = F64;  cap = F32;  dem = PY
//   capped = cap < order            -> order_qty is cap (F32) instead of order (F64);   pos = min(.) > 0 else PY 0
//   B      = dem < inv              -> sales is dem (PY: revenue = dem * price in float64) else inv (F32: float32 product)
//   excess = inv - dem, short = dem - inv are float32 differences; the positive one stays F32, the other becomes PY 0
// so purchase cost is a float64 product (not capped), a float32 product (capped) or 0.0; holding cost / penalty are
// float32 products or 0.0.  reward = ((rev - pc) - hc) - lp then evaluates
//   * entirely in float64 when pc is F64 (float64 wins every promotion),
//   * otherwise in float32 from the first F32 operand on -- subtracting a PY 0 never changes a value, so that is the
//     float32 chain started from float32(rev) -- and stays the float64 rev when every operand is PY.
// qf holds float32(price, cost, h, k), which is what NumPy uses when a Python float meets a float32 scalar (NEP 50).
struct NvPar32 {
    float price, cost, h, k;
};
__device__ __forceinline__ double nv_period_lt(const NvDev& P, const NvParams& q, const NvPar32& qf, float action,
                                               long long demand, float pipe0, float psum, float* oq_out, double* parts,
                                               double* su_out, double* ex_out, double* sh_out) {
    double a64 = (double)action;                                  // .item() -> Python float (:131)
    a64 = a64 < 0.0 ? 0.0 : (a64 > P.max_q ? P.max_q : a64);      // np.clip -> np.float64 (:132)
    const float capf = (float)P.max_inv - psum;                   // int - np.float32 -> float32 (:143)
    const double capd = (double)capf;
    const bool capped = capd < a64;                               // min(order_qty, cap)
    const double mnv = capped ? capd : a64;
    const bool pos = mnv > 0.0;                                   // max(0, .)
    const bool pcF32 = pos && capped, pcF64 = pos && !capped;
    *oq_out = pos ? (capped ? capf : (float)a64) : 0.0f;          // new_pipeline[-1] = order_qty (:179)
    const double dd = (double)demand;
    const float df = (float)dd, invf = pipe0;
    const double invd = (double)invf;
    const bool B = dd < invd;                                     // min(inv_on_hand, demand) (:149)
    const double revd = dd * q.price;                             // PY * PY
    const float revf = invf * qf.price;                           // F32 * PY
    const float exf = invf - df, shf = df - invf;                 // :152-153
    const bool exP = exf > 0.0f, shP = shf > 0.0f;
    const double pcd = a64 * q.cost;                              // F64 * PY (:162)
    const float pcf = pcF32 ? capf * qf.cost : 0.0f;              // F32 * PY, or PY 0 * PY = 0.0
    const float hcf = exP ? exf * qf.h : 0.0f;                    // :166
    const float lpf = shP ? shf * qf.k : 0.0f;                    // :167
    const double rev_v = B ? revd : (double)revf, hc_v = (double)hcf, lp_v = (double)lpf;
    const double r64 = ((rev_v - pcd) - hc_v) - lp_v;             // pc is F64: float64 throughout (:170)
    const float s32 = B ? (float)revd : revf;
    const float r32 = ((s32 - pcf) - hcf) - lpf;                  // float32 from the first F32 operand on
    const bool any32 = !B || pcF32 || exP || shP;
    const double rew = pcF64 ? r64 : (any32 ? (double)r32 : revd);
    if (parts) {
        parts[0] = rev_v;
        parts[1] = pcF64 ? pcd : (double)pcf;
        parts[2] = hc_v;
        parts[3] = lp_v;
    }
    if (su_out) {
        *su_out = B ? dd : invd;
        *ex_out = exP ? (double)exf : 0.0;
        *sh_out = shP ? (double)shf : 0.0;
    }
    return rew;
}

// ---- reset ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) nv_reset_kernel(const __grid_constant__ NvDev P, int64_t N, int64_t npad,
                                                       void* state, int reseed, uint64_t seed, int64_t env_offset,
                                                       const uint8_t* __restrict__ mask, const double* __restrict__ fixed,
                                                       float* __restrict__ obs) {
    __shared__ float par32[256][5];
    const int64_t e0 = (int64_t)blockIdx.x * 256, e = e0 + threadIdx.x;
    if (e < N && (!mask || mask[e])) {
        NvState st(state, npad, P.L);
        uint64_t key;
        uint32_t ep;
        if (reseed) {
            key = seed + (uint64_t)(env_offset + e);
            ep = 0;
            st.key[e] = key;
        } else {
            key = st.key[e];
            ep = ((st.episode[e] & ~NV_EP_FIXED) + 1) & ~NV_EP_FIXED;
        }
        st.episode[e] = ep | (fixed ? NV_EP_FIXED : 0u);
        NvParams q;
        if (fixed) {
            q.price = fixed[e * 5 + 0]; q.cost = fixed[e * 5 + 1]; q.h = fixed[e * 5 + 2]; q.k = fixed[e * 5 + 3];
            q.mu = fixed[e * 5 + 4];
        } else
            q = nv_draw_params(P, key, ep);
        for (int z = 0; z < 5; z++) {
            st.par[(size_t)z * npad + e] = (&q.price)[z];
            par32[threadIdx.x][z] = (float)(&q.price)[z];  // :115
        }
        for (int j = 0; j < P.L; j++) st.pipe[(size_t)j * npad + e] = 0.0f;
        st.step[e] = 0;
    }
    __syncthreads();
    // first observation [price, cost, h, k, mu, 0 ...] written cooperatively (coalesced)
    const int W = P.obs_dim;
    const int nrows = (int)((N - e0) < 256 ? (N - e0) : 256);
    int r = 0, c = threadIdx.x;
    while (c >= W) { c -= W; r++; }
    for (int i = threadIdx.x; i < nrows * W; i += 256) {
        if (!mask || mask[e0 + r]) obs[e0 * W + i] = c < 5 ? par32[r][c] : 0.0f;
        c += 256;
        while (c >= W) { c -= W; r++; }
    }
}

// ---- step ------------------------------------------------------------------------------------------------------
struct NvStepArgs {
    int64_t N, npad;
    void* state;
    const float* actions;
    const int64_t* demand;
    int autoreset;
    float* obs;
    double* reward;
    uint8_t* terminated;
    uint8_t* truncated;
    int64_t* info_demand;
    double* info_parts;
    int64_t info_ld;  // 0: parts row-major [N][4]; > 0: column-major [4][info_ld]
    float* final_obs;
    uint32_t* err;
    int use_bulk;
};

__global__ void __launch_bounds__(ORGYM_TILE, NV_STEP_MINB) nv_step_kernel(const __grid_constant__ NvDev P, const NvStepArgs A) {
    extern __shared__ __align__(128) unsigned char smem[];
    float* tile = (float*)smem;
    const int tid = threadIdx.x, W = P.obs_dim;
    const int64_t e0 = (int64_t)blockIdx.x * ORGYM_TILE, e = e0 + tid;
    const int nvalid = (int)((A.N - e0) < ORGYM_TILE ? (A.N - e0) : ORGYM_TILE);
    const bool valid = tid < nvalid;
    const bool dense = (W % 4) != 0;  // <= 2-way bank conflicts on the dense tile
    const int stride = dense ? W : W + 1;
    const bool bulk = A.use_bulk && dense && nvalid == ORGYM_TILE;
    NvState st(A.state, A.npad, P.L);
    if (valid) {
        float* row = tile + tid * stride;
        // the pipeline goes straight into this env's row of the observation tile with asynchronous copies issued
        // before anything else: they overlap the scalar loads, the demand draw and its table gather
        {
            const float* pp = st.pipe + e;
            for (int j = 0; j < P.L; j++) cp_async4(row + 5 + j, pp + (size_t)j * A.npad);
        }
        int sc = st.step[e];
        const uint32_t epw = st.episode[e];
        const uint32_t pinned = epw & NV_EP_FIXED;
        uint32_t ep = epw & ~NV_EP_FIXED;
        uint64_t key = st.key[e];
        NvParams q;
        q.price = st.par[0 * A.npad + e]; q.cost = st.par[1 * A.npad + e]; q.h = st.par[2 * A.npad + e];
        q.k = st.par[3 * A.npad + e]; q.mu = st.par[4 * A.npad + e];
        bool do_step = true;
        if (sc >= P.T) {
            do_step = false;
            cp_async_wait_all();
            if (A.autoreset == ORGYM_AUTORESET_NEXT_STEP) {
                ep = (ep + 1) & ~NV_EP_FIXED;
                if (!pinned) {
                    q = nv_draw_params(P, key, ep);
                    for (int z = 0; z < 5; z++) st.par[(size_t)z * A.npad + e] = (&q.price)[z];
                }
                st.episode[e] = ep | pinned;
                for (int j = 0; j < P.L; j++) st.pipe[(size_t)j * A.npad + e] = 0.0f;
                st.step[e] = 0;
                for (int z = 0; z < 5; z++) row[z] = (float)(&q.price)[z];
                for (int j = 0; j < P.L; j++) row[5 + j] = 0.0f;
                A.reward[e] = 0.0; A.terminated[e] = 0; A.truncated[e] = 0;
            } else {
                atomicOr(A.err, ORGYM_ERR_STEP_PAST_END);
                const float* old = A.obs + e * W;
                for (int z = 0; z < W; z++) row[z] = old[z];
                A.reward[e] = 0.0; A.terminated[e] = 0; A.truncated[e] = 1;
            }
        }
        if (do_step) {
            const int64_t np_ = A.npad;
            long long d = A.demand ? A.demand[e] : poisson_mu(P.pt, P.rcp, q.mu, key, ep, sc);
            cp_async_wait_all();
            float psum = nv_pipe_sum(P.L, [&](int j) { return row[5 + j]; });
            float pipe0 = P.L > 0 ? row[5] : 0.0f;
            float oq;
            double parts[4];
            double r;
            if (P.L > 0) {
                const NvPar32 qf = {(float)q.price, (float)q.cost, (float)q.h, (float)q.k};
                r = nv_period_lt(P, q, qf, A.actions[e], d, pipe0, psum, &oq, parts, nullptr, nullptr, nullptr);
            } else
                r = nv_period(P, q, A.actions[e], d, pipe0, psum, &oq, parts, nullptr, nullptr, nullptr);
            int sc1 = sc + 1;
            bool trunc = sc1 >= P.T;  // :190
            bool reset_now = trunc && A.autoreset == ORGYM_AUTORESET_SAME_STEP;
            for (int z = 0; z < 5; z++) row[z] = (float)(&q.price)[z];
            {
                float* pw = st.pipe + e;
                for (int j = 0; j < P.L; j++) {  // shift left, append the new order (:177); one pass for tile and state
                    const float x = j + 1 < P.L ? row[5 + j + 1] : oq;
                    row[5 + j] = x;
                    if (!reset_now) pw[(size_t)j * np_] = x;
                }
            }
            if (!reset_now) {
                st.step[e] = sc1;
            } else {
                if (A.final_obs)
                    for (int z = 0; z < W; z++) A.final_obs[e * W + z] = row[z];
                ep = (ep + 1) & ~NV_EP_FIXED;
                if (!pinned) {
                    q = nv_draw_params(P, key, ep);
                    for (int z = 0; z < 5; z++) st.par[(size_t)z * A.npad + e] = (&q.price)[z];
                }
                st.episode[e] = ep | pinned;
                for (int j = 0; j < P.L; j++) st.pipe[(size_t)j * A.npad + e] = 0.0f;
                st.step[e] = 0;
                for (int z = 0; z < 5; z++) row[z] = (float)(&q.price)[z];
                for (int j = 0; j < P.L; j++) row[5 + j] = 0.0f;
            }
            A.reward[e] = r;
            A.terminated[e] = 0;
            A.truncated[e] = trunc ? 1 : 0;
            if (A.info_demand) A.info_demand[e] = d;
            if (A.info_parts)
                for (int z = 0; z < 4; z++) A.info_parts[A.info_ld ? z * A.info_ld + e : e * 4 + z] = parts[z];
        }
    }
    float* g = A.obs + (size_t)e0 * W;
    if (bulk) {
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            bulk_s2g(g, tile, (uint32_t)(ORGYM_TILE * W * 4));
            bulk_commit();
            bulk_wait_read0();
        }
    } else {
        __syncthreads();
        int total = nvalid * W;
        for (int i = tid; i < total; i += ORGYM_TILE) {
            int r = i / W, c = i - r * W;
            g[i] = tile[r * stride + c];
        }
    }
}

__global__ void nv_export_params_kernel(int64_t N, int64_t npad, int L, const void* state, double* __restrict__ out) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    NvState st((void*)state, npad, L);
    for (int z = 0; z < 5; z++) out[e * 5 + z] = st.par[(size_t)z * npad + e];
}

// ---- Poisson quantile: smallest k with cdf(k) >= q (scipy.stats.poisson.ppf) ---------------------------------------
// pmf recurrence summed in ascending order from 9 sigma below the mean (the mass below is < 3e-18); the per-term
// division is a reciprocal-multiply (1 ulp), which can only matter when q sits within ~1e-13 of a CDF step.
// The search advances four terms per trip: the partial sums are formed in the same order as a term-by-term loop
// (identical floating-point values), but only the last one is compared with q -- the CDF is non-decreasing, so the
// quantile lies in the block iff its last partial sum reaches q.
// four consecutive table entries from a 32-byte aligned address as ONE 256-bit load (sm_100: LDG.E.256): a lane's block
// of reciprocals is exactly one L1 sector, fetched with one request instead of two
struct D4 { double x, y, z, w; };
__device__ __forceinline__ D4 ld_rcp4(const double* p) {
    D4 v;
    asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(v.x), "=d"(v.y), "=d"(v.z), "=d"(v.w) : "l"(p));
    return v;
}
// The search is written as three pieces over one state (a kernel can then interleave the searches of several episodes
// with exactly the arithmetic of the plain loop: see nv_level_kernel).
struct PpfState {
    double q, mu, cdf, term, res;  // term = pmf(k), cdf = P(X < k)
    int k, kmu;                    // for integer k: k > mu <=> k > floor(mu) = kmu
    bool done;
};
// Every lane walks the reciprocal table at its own k, so a warp load is a gather: with four 8-byte loads per block at
// an arbitrary offset it touched ~20 sectors per load and the L1 data stage bounded the search (ncu, round 2).
// Up to three single steps first bring k + 1 to a multiple of 4; the block's four reciprocals are then one aligned
// 32-byte piece -- one 256-bit load, one sector per lane.  Term-by-term the arithmetic is unchanged.
// Single exit: the result is carried in (res, done) instead of returning from inside the loops.  With early returns
// the lanes of a warp left the alignment steps on different paths and were not reconverged before the block loop,
// which then ran once per alignment class (ncu: twice the trips of the warp's slowest lane).
__device__ __forceinline__ void ppf_init(PpfState& S, double q, double mu, const double* __restrict__ rcp) {
    S.q = q; S.mu = mu; S.cdf = 0.0; S.term = 0.0; S.res = 0.0; S.k = 0; S.kmu = 0; S.done = false;
    if (!(q > 0.0)) { S.res = -1.0; S.done = true; return; }
    if (q >= 1.0) { S.res = INFINITY; S.done = true; return; }
    double lo = floor(mu - 9.0 * sqrt(mu) - 9.0);
    if (lo < 0.0) lo = 0.0;
    S.term = exp(-mu + lo * log(mu) - lgamma(lo + 1.0));
    S.k = (int)lo;
    S.kmu = mu < 1e9 ? (int)mu : 1000000000;
#pragma unroll
    for (int s = 0; s < 3; s++) {
        if (!S.done && ((S.k + 1) & 3) != 0 && S.k + 1 <= ORGYM_RCP_N) {
            const double c = S.cdf + S.term;
            if (c >= q) {
                S.res = (double)S.k;
                S.done = true;
            } else {
                S.term *= mu * rcp[S.k + 1];
                ++S.k;
                if (S.term == 0.0 && S.k > S.kmu) {
                    S.res = (double)S.k;
                    S.done = true;
                }
                S.cdf = c;
            }
        }
    }
}
// Eight terms (two aligned 32-byte pieces of the reciprocal table) with the partial sums formed in term order; requires
// !S.done and S.k + 8 <= ORGYM_RCP_N.  (cdf, term, k) advance unconditionally -- they are dead once done is set, so no
// copies of the old values stay alive across a block.
__device__ __forceinline__ void ppf_step8(PpfState& S, const double* __restrict__ rcp) {
    const double q = S.q, mu = S.mu;
    const int k = S.k, kmu = S.kmu;
    const D4 ra = ld_rcp4(rcp + k + 1), rb = ld_rcp4(rcp + k + 5);
    const double t0 = S.term, t1 = t0 * (mu * ra.x), t2 = t1 * (mu * ra.y), t3 = t2 * (mu * ra.z), t4 = t3 * (mu * ra.w),
                 t5 = t4 * (mu * rb.x), t6 = t5 * (mu * rb.y), t7 = t6 * (mu * rb.z), t8 = t7 * (mu * rb.w);
    const double c0 = S.cdf + t0, c1 = c0 + t1, c2 = c1 + t2, c3 = c2 + t3, c4 = c3 + t4, c5 = c4 + t5, c6 = c5 + t6,
                 c7 = c6 + t7;
    if (c7 >= q) {
        const int j = c3 >= q ? (c0 >= q ? 0 : (c1 >= q ? 1 : (c2 >= q ? 2 : 3)))
                              : (c4 >= q ? 4 : (c5 >= q ? 5 : (c6 >= q ? 6 : 7)));
        S.res = (double)(k + j);
        S.done = true;
    } else if (t8 == 0.0 && k + 8 > kmu) {  // underflow beyond the mean: q is within rounding of 1
        const double tt[8] = {t1, t2, t3, t4, t5, t6, t7, t8};
        int j = 8;
#pragma unroll
        for (int i = 7; i >= 1; i--)
            if (tt[i - 1] == 0.0 && k + i > kmu) j = i;
        S.res = (double)(k + j);
        S.done = true;
    }
    S.cdf = c7;
    S.term = t8;
    S.k = k + 8;
}
// the last block of four inside the table, then term by term beyond it (means in the thousands); requires !S.done
__device__ __forceinline__ void ppf_tail(PpfState& S, const double* __restrict__ rcp) {
    const double q = S.q, mu = S.mu;
    const int kmu = S.kmu;
    if (S.k + 4 <= ORGYM_RCP_N) {
        const int k = S.k;
        const D4 ra = ld_rcp4(rcp + k + 1);
        const double t0 = S.term, t1 = t0 * (mu * ra.x), t2 = t1 * (mu * ra.y), t3 = t2 * (mu * ra.z),
                     t4 = t3 * (mu * ra.w);
        const double c0 = S.cdf + t0, c1 = c0 + t1, c2 = c1 + t2, c3 = c2 + t3;
        if (c3 >= q) {
            S.res = (double)(k + (c0 >= q ? 0 : (c1 >= q ? 1 : (c2 >= q ? 2 : 3))));
            S.done = true;
        } else if (t4 == 0.0 && k + 4 > kmu) {
            S.res = (double)(k + ((t1 == 0.0 && k + 1 > kmu) ? 1 : ((t2 == 0.0 && k + 2 > kmu) ? 2 : ((t3 == 0.0 && k + 3 > kmu) ? 3 : 4))));
            S.done = true;
        }
        S.cdf = c3;
        S.term = t4;
        S.k = k + 4;
    }
    if (!S.done) {
        int k = S.k;
        double cdf = S.cdf, term = S.term;
        for (;;) {
            cdf += term;
            if (cdf >= q) break;
            ++k;
            term *= mu * (k <= ORGYM_RCP_N ? rcp[k] : __drcp_rn((double)k));
            if (term == 0.0 && (double)k > mu) break;
        }
        S.res = (double)k;
        S.done = true;
    }
}
__device__ __forceinline__ double poisson_ppf_dev(double q, double mu, const double* __restrict__ rcp) {
    PpfState S;
    ppf_init(S, q, mu, rcp);
    while (!S.done && S.k + 8 <= ORGYM_RCP_N) ppf_step8(S, rcp);
    if (!S.done) ppf_tail(S, rcp);
    return S.res;
}

// ---- fused rollout ----------------------------------------------------------------------------------------------
struct NvRolloutArgs {
    int64_t N, env_offset;
    uint64_t seed;
    uint32_t episode;
    int policy;
    double param0;
    const float* actions;
    int64_t a_se, a_st;
    const int64_t* demand;
    int64_t d_se, d_st;
    const double* fixed;
    const double* level_in;  // classic / (s,S): the episode's order-up-to level, computed by nv_level_kernel (else null)
    double* ep_return;
    double* stats;
    double* reward_traj;
    float* action_traj;
    float* final_obs;
    double* partials;
};

#define NV_ROLL_THREADS 128

// per-episode order-up-to level of the classic-newsvendor and (s,S) drivers: they only read the float32 observation
// entries h, k, mu (benchmark_newsvendor.py:113-161, benchmark_newsvendor_sb3_rllib.py:363-371)
__device__ __forceinline__ bool nv_classic_fallback(float fh, float fk) {
    const float hk = fh + fk;
    return hk <= 1e-6f || fk < 0.0f || fh < 0.0f;
}
// the level is poisson_ppf(*q, *mu) passed through nv_level_finish when this returns true, 0 otherwise
__device__ __forceinline__ bool nv_level_query(int policy, double param0, int L, float fh, float fk, float fmu, double* q,
                                               double* mu) {
    if (policy == ORGYM_NV_POLICY_CLASSIC) {
        if (nv_classic_fallback(fh, fk)) return false;
        const float cr = fk / (fh + fk);
        const float eff = (fmu * (float)(L + 1)) * (float)param0;
        *q = (double)cr;
        *mu = eff > 1e-6f ? (double)eff : 1e-6;
        return true;
    }
    if (!(fh + fk > 1e-6f)) return false;
    float cr = fk / (fh + fk);
    cr = cr < 0.001f ? 0.001f : (cr > 0.999f ? 0.999f : cr);
    const float eff = fmu * (float)(L + 1);
    *q = (double)cr;
    *mu = eff > 1e-6f ? (double)eff : 1e-6;
    return true;
}
__device__ __forceinline__ double nv_level_finish(int policy, double ppf) {
    return policy == ORGYM_NV_POLICY_CLASSIC ? ppf : (ppf > 0.0 ? ppf : 0.0);
}
__device__ __forceinline__ double nv_policy_level(const NvDev& P, int policy, double param0, int L, float fh, float fk, float fmu) {
    double q, mu;
    if (!nv_level_query(policy, param0, L, fh, fk, fmu, &q, &mu)) return 0.0;
    return nv_level_finish(policy, poisson_ppf_dev(q, mu, P.rcp));
}

// demand of period t of one env in a fused rollout: replayed, PTRS (large means), or the alias table plus the small-table
// inversion of the Poisson remainder with one Philox block per two periods (the same words as poisson_mu).  pcdf is the
// env's column of the remainder's CDF tile ([k][env], stride pstride); dw carries the block from even to odd periods.
__device__ __forceinline__ long long nv_roll_demand(const NvDev& P, const NvRolloutArgs& A, const NvParams& q,
                                                    const PoisSplit& ps, uint64_t key, int64_t e, bool valid, int t,
                                                    uint4& dw, const double* pcdf, int pstride) {
    if (A.demand) return valid ? A.demand[e * A.d_se + (int64_t)t * A.d_st] : 0;
    if (ps.i0 < 0) return poisson_ptrs(q.mu, key, A.episode, t);
    if ((t & 1) == 0) dw = philox_block(key, (uint32_t)t >> 1, A.episode, STREAM_POISSON_TAB, 0);
    const uint32_t wa = (t & 1) ? dw.z : dw.x, wi = (t & 1) ? dw.w : dw.y;
    return poisson_tab_alias(P.pt, ps, wa) +
           poisson_small_lookup(((double)wi + 0.5) * (1.0 / 4294967296.0), pcdf, pstride, ps.r, ps.p0, P.rcp);
}

__device__ __forceinline__ float clipf(float q, float hi) { return q < 0.0f ? 0.0f : (q > hi ? hi : q); }

// LT > 0: the lead time is the compile-time constant LT (1..7): the pipeline lives in LT registers, summed and shifted
// with static indices (LT adds, LT - 1 moves per period) instead of a shared-memory ring with modular indexing.
// (Unrolling the period loop by LT to avoid even the moves was measured slower: 5x the code, instruction-fetch stalls.)
// LT == 0: any lead time, ring in shared memory.
template <int LT>
__global__ void __launch_bounds__(NV_ROLL_THREADS, NV_ROLL_MINB) nv_rollout_kernel(const __grid_constant__ NvDev P,
                                                                     const __grid_constant__ NvRolloutArgs A) {
    extern __shared__ __align__(128) unsigned char smem[];
    float* ring = (float*)smem;  // [L][threads], logical index j lives at slot (head + j) % L
    const int tid = threadIdx.x, L = LT > 0 ? LT : P.L;
    const int64_t e = (int64_t)blockIdx.x * NV_ROLL_THREADS + tid;
    const bool valid = e < A.N;
    if (LT == 0)
        for (int j = 0; j < L; j++) ring[j * NV_ROLL_THREADS + tid] = 0.0f;
    const uint64_t key = A.seed + (uint64_t)(A.env_offset + e);
    NvParams q;
    if (A.fixed && valid) {
        q.price = A.fixed[e * 5 + 0]; q.cost = A.fixed[e * 5 + 1]; q.h = A.fixed[e * 5 + 2]; q.k = A.fixed[e * 5 + 3];
        q.mu = A.fixed[e * 5 + 4];
    } else
        q = nv_draw_params(P, key, A.episode);
    const float fh = (float)q.h, fk = (float)q.k, fmu = (float)q.mu, hi = (float)P.max_q;
    const NvPar32 qf = {(float)q.price, (float)q.cost, fh, fk};
    // per-episode constants of the drivers (they only read the float32 observation entries h, k, mu)
    double level = 0.0;
    bool fallback = false;
    if (A.policy == ORGYM_NV_POLICY_CLASSIC) {  // benchmark_newsvendor.py:113-161 (k_vs_h)
        fallback = nv_classic_fallback(fh, fk);
        level = A.level_in ? (valid ? A.level_in[e] : 0.0) : nv_policy_level(P, A.policy, A.param0, L, fh, fk, fmu);
    } else if (A.policy == ORGYM_NV_POLICY_SS)  // benchmark_newsvendor_sb3_rllib.py:363-371
        level = A.level_in ? (valid ? A.level_in[e] : 0.0) : nv_policy_level(P, A.policy, A.param0, L, fh, fk, fmu);
    const PoisSplit ps = poisson_split(P.pt, q.mu);  // per-episode constants of the demand sampler
    uint4 dw = make_uint4(0, 0, 0, 0);
    __shared__ double pcdf[ORGYM_PT_CDF * NV_ROLL_THREADS];  // cdf of the Poisson(r) remainder, [k][thread]
    if (ps.i0 >= 0 && !A.demand) poisson_small_table(ps.r, ps.p0, P.rcp, pcdf + tid, NV_ROLL_THREADS);
    int head = 0;
    double ret = 0.0, s_sales = 0.0, s_dem = 0.0, s_lost = 0.0, s_ex = 0.0;
    // one period given the pipeline sum and the arriving order; returns the order placed (the new last element)
    auto period = [&](const int t, const float psum, const float pipe0) -> float {
        float act;
        if (A.policy == ORGYM_NV_POLICY_ACTIONS)
            act = valid ? A.actions[e * A.a_se + (int64_t)t * A.a_st] : 0.0f;
        else if (A.policy == ORGYM_NV_POLICY_ORDER_UP_TO || (A.policy == ORGYM_NV_POLICY_CLASSIC && fallback)) {
            // benchmark_newsvendor.py:103-111 -- all float32
            float target = fmu * (float)(L + 1);
            if (A.policy == ORGYM_NV_POLICY_ORDER_UP_TO) target = target * (float)A.param0;
            float x = target - psum;
            act = clipf(x > 0.0f ? x : 0.0f, hi);
        } else if (A.policy == ORGYM_NV_POLICY_CLASSIC) {
            double x = level - (double)psum;  // np.float64 - np.float32
            x = x > 0.0 ? x : 0.0;
            x = x > (double)hi ? (double)hi : x;
            act = (float)x;
        } else {  // (s,S)
            double x = 0.0;
            if ((double)psum < level) {
                x = level * A.param0 - (double)psum;
                x = x > 0.0 ? x : 0.0;
            }
            x = x > (double)hi ? (double)hi : x;
            act = (float)x;
        }
        const long long d = nv_roll_demand(P, A, q, ps, key, e, valid, t, dw, pcdf + tid, NV_ROLL_THREADS);
        float oq;
        double su, ex, sh;
        double r;
        if (LT > 0 || L > 0)
            r = nv_period_lt(P, q, qf, act, d, pipe0, psum, &oq, nullptr, &su, &ex, &sh);
        else
            r = nv_period(P, q, act, d, pipe0, psum, &oq, nullptr, &su, &ex, &sh);
        ret += r;
        s_sales += su; s_dem += (double)d; s_lost += sh; s_ex += ex;
        if (valid && A.reward_traj) A.reward_traj[e * P.T + t] = r;
        if (valid && A.action_traj) A.action_traj[e * P.T + t] = act;
        return oq;
    };
    float pv[LT > 0 ? LT : 1];
#pragma unroll
    for (int j = 0; j < (LT > 0 ? LT : 1); j++) pv[j] = 0.0f;
    if (LT > 0) {
        for (int t = 0; t < P.T; t++) {
            float r = 0.0f;  // np.sum over fewer than 8 float32 values: sequential, oldest first
#pragma unroll
            for (int j = 0; j < LT; j++) r = r + pv[j];
            const float oq = period(t, r, pv[0]);
#pragma unroll
            for (int j = 0; j + 1 < LT; j++) pv[j] = pv[j + 1];  // shift left, append (:177-179): LT - 1 register moves
            pv[LT - 1] = oq;
        }
    } else {
        for (int t = 0; t < P.T; t++) {
            auto get = [&](int j) {
                int s = head + j;
                s = s >= L ? s - L : s;
                return ring[s * NV_ROLL_THREADS + tid];
            };
            const float psum = nv_pipe_sum(L, get);
            const float pipe0 = L > 0 ? ring[head * NV_ROLL_THREADS + tid] : 0.0f;
            const float oq = period(t, psum, pipe0);
            if (L > 0) {  // shift left, append: overwrite the slot that just arrived and advance the head
                ring[head * NV_ROLL_THREADS + tid] = oq;
                head = head + 1 == L ? 0 : head + 1;
            }
        }
    }
    if (valid) {
        if (A.ep_return) A.ep_return[e] = ret;
        if (A.stats) {
            A.stats[e * 4 + 0] = s_sales; A.stats[e * 4 + 1] = s_dem; A.stats[e * 4 + 2] = s_lost; A.stats[e * 4 + 3] = s_ex;
        }
        if (A.final_obs) {
            float* o = A.final_obs + e * P.obs_dim;
            o[0] = (float)q.price; o[1] = (float)q.cost; o[2] = fh; o[3] = fk; o[4] = fmu;
            if (LT > 0) {
#pragma unroll
                for (int j = 0; j < LT; j++) o[5 + j] = pv[j];
            } else {
                for (int j = 0; j < L; j++) {
                    int s = head + j;
                    s = s >= L ? s - L : s;
                    o[5 + j] = ring[s * NV_ROLL_THREADS + tid];
                }
            }
        }
    }
    if (A.partials) {
        double v[7] = {valid ? 1.0 : 0.0, valid ? ret : 0.0, valid ? ret * ret : 0.0, valid ? s_sales : 0.0,
                       valid ? s_dem : 0.0, valid ? s_lost : 0.0, valid ? s_ex : 0.0};
        __shared__ double red[NV_ROLL_THREADS / 32][7];
#pragma unroll
        for (int z = 0; z < 7; z++) {
            double x = v[z];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if ((tid & 31) == 0) red[tid >> 5][z] = x;
        }
        __syncthreads();
        if (tid < 7) {
            double x = 0.0;
            for (int wv = 0; wv < NV_ROLL_THREADS / 32; wv++) x += red[wv][tid];
            A.partials[(size_t)blockIdx.x * 8 + tid] = x;
        }
    }
}


// The Poisson quantile behind that level is a serial float64 recurrence of a few hundred terms per episode.  Inside the
// rollout kernel (96 registers, 5 warps per scheduler) its latency is exposed: 19 % of the instructions but ~40 % of the
// time of a classic-policy rollout.  As a kernel of its own -- nothing else live -- it runs at several times the
// occupancy and hides that latency; the level travels to the rollout kernel through the episode's
// slot of the ep_return output array (written here, read at the start of the rollout, overwritten with the return at
// its end), so no extra memory is needed.  Same arithmetic, same value.
struct NvLevelArgs {
    int64_t N, env_offset;
    uint64_t seed;
    uint32_t episode;
    int policy;
    double param0;
    const double* fixed;
    double* level_out;
};
// One thread per episode.  The searches differ in length (a few to ~110 blocks of eight terms, by the episode's demand
// mean and critical ratio), so 19 of a warp's 32 lanes are active on average.  Measured alternative (round 2, in the
// history of this file): a warp prepares 256 episodes, parks the search states in shared memory and drains them as a
// queue, a lane fetching the next state when its own search ends (refills batched, results stored coalesced at the
// end) -- 23 lanes active, but 44 % more thread-instructions for the queue handling: 0.755 ms against 0.685 ms.
__global__ void __launch_bounds__(256, 4) nv_level_kernel(const __grid_constant__ NvDev P, const __grid_constant__ NvLevelArgs A) {
    const int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (e >= A.N) return;
    NvParams q;
    if (A.fixed) {
        q.h = A.fixed[e * 5 + 2]; q.k = A.fixed[e * 5 + 3]; q.mu = A.fixed[e * 5 + 4];
    } else
        q = nv_draw_params(P, A.seed + (uint64_t)(A.env_offset + e), A.episode);
    A.level_out[e] = nv_policy_level(P, A.policy, A.param0, P.L, (float)q.h, (float)q.k, (float)q.mu);
}

// ---- fused rollout driven by an MLP actor (ORGYM_NV_POLICY_MLP) -----------------------------------------------------
// One CTA of MLP_THREADS threads = 128 consecutive envs (one row of the partial sums, like nv_rollout_kernel), run as 128/E
// sub-tiles of E envs one after the other; weights and biases are staged in shared memory once per CTA (mlp.cuh).
// Thread tid < E owns env e0 + tid of the current sub-tile: its parameters, demand sampler constants, Philox words and
// accumulators live in its registers, the CDF of its Poisson remainder in column tid of a [ORGYM_PT_CDF][E] tile.
// The float32 observation tile [obs_dim][E] is the network's input and the env's pipeline at once: rows 0-4 hold
// price, cost, h, k, mu for the episode, rows 5.. the pipeline oldest first, shifted left and appended in place.
// Per period the whole CTA runs the hidden layers (one barrier each); the owner threads then evaluate the single output
// (K ascending FMAs on their own column), take the period through the env's own device functions and append the order.
struct NvMlpPlan {
    MlpNet net;
    int E, log2E;
    int obs_off, buf_off[2];  // float offsets in dynamic shared memory (the weights start at 0)
    int pcdf_off;             // byte offset of the Poisson-remainder CDF tile
};

__global__ void __launch_bounds__(MLP_THREADS, 2) nv_mlp_rollout_kernel(const __grid_constant__ NvDev P,
                                                                       const __grid_constant__ NvRolloutArgs A,
                                                                       const __grid_constant__ NvMlpPlan M) {
    static_assert(MLP_THREADS >= NV_ROLL_THREADS, "one CTA covers a partial-sum row");
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ double red[NV_ROLL_THREADS / 32][7];
    const int tid = threadIdx.x, E = M.E, NL = M.net.L, L = P.L, od = P.obs_dim;
    float* fs = (float*)smem;
    float* obs = fs + M.obs_off;
    double* pcdf = (double*)(smem + M.pcdf_off) + tid;
    mlp_stage_weights(M.net, fs);
    const int Klast = M.net.K[NL - 1];
    const float* Wlast = fs + M.net.w_off[NL - 1];
    const float* blast = fs + M.net.b_off[NL - 1];
    const float* hin = NL == 1 ? obs : fs + M.buf_off[(NL - 2) & 1];  // input of the last layer
    const float hi = (float)P.max_q;
    const bool owner = tid < E;
    const int nsub = NV_ROLL_THREADS / E;
    for (int sub = 0; sub < nsub; sub++) {
        const int64_t e0 = (int64_t)blockIdx.x * NV_ROLL_THREADS + (int64_t)sub * E;
        const int64_t e = e0 + tid;
        const bool valid = owner && e < A.N;
        if (e0 >= A.N) {  // CTA-uniform: the sums of the missing warps are zero, like idle lanes of nv_rollout_kernel
            if (tid < 7 * (E / 32)) red[sub * (E / 32) + tid / 7][tid % 7] = 0.0;
            continue;
        }
        const uint64_t key = A.seed + (uint64_t)(A.env_offset + e);
        NvParams q = {0.0, 0.0, 0.0, 0.0, 0.0};
        NvPar32 qf = {0.f, 0.f, 0.f, 0.f};
        PoisSplit ps;
        uint4 dw = make_uint4(0, 0, 0, 0);
        double ret = 0.0, s_sales = 0.0, s_dem = 0.0, s_lost = 0.0, s_ex = 0.0;
        if (owner) {
            if (A.fixed && valid) {
                q.price = A.fixed[e * 5 + 0]; q.cost = A.fixed[e * 5 + 1]; q.h = A.fixed[e * 5 + 2];
                q.k = A.fixed[e * 5 + 3]; q.mu = A.fixed[e * 5 + 4];
            } else
                q = nv_draw_params(P, key, A.episode);
            qf = {(float)q.price, (float)q.cost, (float)q.h, (float)q.k};
            ps = poisson_split(P.pt, q.mu);
            if (ps.i0 >= 0 && !A.demand) poisson_small_table(ps.r, ps.p0, P.rcp, pcdf, E);
            // first observation [price, cost, h, k, mu, 0 ...] (:115, :122)
            obs[0 * E + tid] = (float)q.price; obs[1 * E + tid] = (float)q.cost; obs[2 * E + tid] = (float)q.h;
            obs[3 * E + tid] = (float)q.k; obs[4 * E + tid] = (float)q.mu;
            for (int j = 0; j < L; j++) obs[(5 + j) * E + tid] = 0.0f;
        }
        __syncthreads();
        for (int t = 0; t < P.T; t++) {
            const float* in = obs;
            for (int l = 0; l < NL - 1; l++) {
                float* out = fs + M.buf_off[l & 1];
                mlp_hidden_layer(in, out, fs + M.net.w_off[l], fs + M.net.b_off[l], M.net.K[l], M.net.Np[l], E, M.log2E,
                                 M.net.act);
                __syncthreads();
                in = out;
            }
            if (owner) {
                float y = blast[0];  // last layer: acc = b, then K ascending FMAs, no activation
                for (int k = 0; k < Klast; k++) y = __fmaf_rn(Wlast[k], hin[k * E + tid], y);
                float act = y > 0.0f ? y : 0.0f;  // np.clip to the action Box in float32, NaN kept
                act = act < hi ? act : hi;
                act = y != y ? y : act;
                const long long d = nv_roll_demand(P, A, q, ps, key, e, valid, t, dw, pcdf, E);
                const float psum = nv_pipe_sum(L, [&](int j) { return obs[(5 + j) * E + tid]; });
                const float pipe0 = L > 0 ? obs[5 * E + tid] : 0.0f;
                float oq;
                double su, ex, sh;
                double r;
                if (L > 0)
                    r = nv_period_lt(P, q, qf, act, d, pipe0, psum, &oq, nullptr, &su, &ex, &sh);
                else
                    r = nv_period(P, q, act, d, pipe0, psum, &oq, nullptr, &su, &ex, &sh);
                ret += r;
                s_sales += su; s_dem += (double)d; s_lost += sh; s_ex += ex;
                if (valid && A.reward_traj) A.reward_traj[e * P.T + t] = r;
                if (valid && A.action_traj) A.action_traj[e * P.T + t] = act;
                for (int j = 0; j < L; j++)  // shift left, append the order placed (:177-179)
                    obs[(5 + j) * E + tid] = j + 1 < L ? obs[(6 + j) * E + tid] : oq;
            }
            __syncthreads();
        }
        if (valid) {
            if (A.ep_return) A.ep_return[e] = ret;
            if (A.stats) {
                A.stats[e * 4 + 0] = s_sales; A.stats[e * 4 + 1] = s_dem; A.stats[e * 4 + 2] = s_lost; A.stats[e * 4 + 3] = s_ex;
            }
            if (A.final_obs)
                for (int z = 0; z < od; z++) A.final_obs[e * od + z] = obs[z * E + tid];
        }
        if (A.partials && owner) {  // warp of 32 consecutive envs: the xor tree of nv_rollout_kernel
            const double v[7] = {valid ? 1.0 : 0.0, valid ? ret : 0.0, valid ? ret * ret : 0.0, valid ? s_sales : 0.0,
                                 valid ? s_dem : 0.0, valid ? s_lost : 0.0, valid ? s_ex : 0.0};
#pragma unroll
            for (int z = 0; z < 7; z++) {
                double x = v[z];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
                if ((tid & 31) == 0) red[sub * (E / 32) + (tid >> 5)][z] = x;
            }
        }
    }
    if (A.partials) {
        __syncthreads();
        if (tid < 7) {  // the four warps in order, as nv_rollout_kernel
            double x = 0.0;
            for (int wv = 0; wv < NV_ROLL_THREADS / 32; wv++) x += red[wv][tid];
            A.partials[(size_t)blockIdx.x * 8 + tid] = x;
        }
    }
}

// Checks an orgym_mlp_t against the handle (ORGYM_E_INVALID) and lays out one CTA's shared memory for it: the largest
// sub-tile of E in {64, 32} envs whose working set fits (ORGYM_E_UNSUPPORTED, with the sizes, when none does).
static int nv_mlp_plan(const NvDev& P, const orgym_mlp_t* mlp, NvMlpPlan* M, size_t* smem_out) {
    ORGYM_REQUIRE(mlp, "policy ORGYM_NV_POLICY_MLP needs in->mlp");
    memset(M, 0, sizeof(*M));
    if (int rc = mlp_net_plan(mlp, P.obs_dim, 1, "the action dimension", &M->net)) return rc;
    const int L = M->net.L, hmax = M->net.hmax;
    const int nbuf = L >= 3 ? 2 : (L == 2 ? 1 : 0);
    size_t smem = 0;
    for (int E = 64; E >= 32; E /= 2) {
        int g = M->net.wfloats;
        M->obs_off = g;
        g += P.obs_dim * E;
        M->buf_off[0] = g;
        g += nbuf >= 1 ? hmax * E : 0;
        M->buf_off[1] = g;
        g += nbuf >= 2 ? hmax * E : 0;
        M->pcdf_off = (int)round_up((int64_t)g * 4, 16);
        smem = (size_t)M->pcdf_off + (size_t)ORGYM_PT_CDF * E * sizeof(double);
        M->E = E;
        M->log2E = E == 64 ? 6 : 5;
        if (smem <= MLP_SMEM_BUDGET) break;
    }
    if (smem > MLP_SMEM_BUDGET) {
        orgym_set_error("mlp: one CTA of 32 envs needs %zu bytes of shared memory (weights and biases %d floats, observation "
                        "tile %d x 32, %d activation tile(s) %d x 32, Poisson CDF tile %d x 32 doubles); this build's limit "
                        "is %d",
                        smem, M->net.wfloats, P.obs_dim, nbuf, hmax, ORGYM_PT_CDF, MLP_SMEM_BUDGET);
        return ORGYM_E_UNSUPPORTED;
    }
    *smem_out = smem;
    return ORGYM_OK;
}

// ------------------------------------------------------------------------------------------------
// host side of the C ABI
// ------------------------------------------------------------------------------------------------
extern "C" int orgym_newsvendor_create(const orgym_newsvendor_config_t* cfg, int64_t num_envs, int device,
                                       orgym_handle_t* out) {
    ORGYM_REQUIRE(cfg && out, "null argument");
    ORGYM_REQUIRE(cfg->lead_time >= 0, "lead_time must be >= 0 (the reference clamps it, newsvendor.py:65)");
    ORGYM_REQUIRE(cfg->step_limit > 0, "step_limit must be positive");
    if (cfg->lead_time > NV_MAXL) {
        orgym_set_error("lead_time %d exceeds this build's limit of %d", cfg->lead_time, NV_MAXL);
        return ORGYM_E_UNSUPPORTED;
    }
    NvHandle* H = new NvHandle();
    NvDev& P = H->dev;
    P.L = cfg->lead_time;
    P.T = cfg->step_limit;
    P.obs_dim = P.L + 5;
    P.max_inv = cfg->max_inventory;
    P.max_q = cfg->max_order_quantity;
    P.p_max = cfg->p_max; P.h_max = cfg->h_max; P.k_max = cfg->k_max; P.mu_max = cfg->mu_max;
    int rc = orgym_handle_base_init(&H->base, FAM_NEWSVENDOR, device, num_envs);
    if (rc == ORGYM_OK) rc = orgym_rcp_table(device, &P.rcp);
    if (rc == ORGYM_OK) rc = orgym_poisson_tables(device, cfg->mu_max, &P.pt);
    if (rc != ORGYM_OK) {
        delete H;
        return rc;
    }
    DeviceGuard g(device);
    H->npad = round_up(num_envs, 32);
    int nblocks = (int)((num_envs + NV_ROLL_THREADS - 1) / NV_ROLL_THREADS);
    H->partials = nullptr;
    size_t pbytes = sizeof(double) * (8 * (size_t)nblocks + ORGYM_REDUCE_EXTRA);
    cudaError_t ce = cudaMalloc(&H->partials, pbytes);
    if (ce == cudaSuccess) ce = cudaMemset(H->partials, 0, pbytes);
    if (ce != cudaSuccess) {
        orgym_set_error("device allocation failed: %s", cudaGetErrorString(ce));
        orgym_handle_base_free(&H->base);
        delete H;
        return ORGYM_E_CUDA;
    }
    H->allocs.push_back(H->partials);
    *out = (orgym_handle_t)H;
    return ORGYM_OK;
}

extern "C" int orgym_newsvendor_destroy(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_NEWSVENDOR)) return ORGYM_E_INVALID;
    NvHandle* H = (NvHandle*)h;
    {
        DeviceGuard g(H->base.device);
        for (void* p : H->allocs) cudaFree(p);
    }
    orgym_handle_base_free(&H->base);
    delete H;
    return ORGYM_OK;
}

extern "C" int64_t orgym_newsvendor_state_bytes(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_NEWSVENDOR)) return -1;
    NvHandle* H = (NvHandle*)h;
    return nv_state_bytes(H->npad, H->dev.L);
}
extern "C" int32_t orgym_newsvendor_obs_dim(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_NEWSVENDOR)) return -1;
    return ((NvHandle*)h)->dev.obs_dim;
}

extern "C" int orgym_newsvendor_reset(orgym_handle_t h, void* state_dev, int reseed, uint64_t seed, int64_t env_offset,
                                      const uint8_t* mask_dev, const double* fixed_params_dev, float* obs_dev,
                                      void* stream) {
    if (orgym_check_handle(h, FAM_NEWSVENDOR)) return ORGYM_E_INVALID;
    NvHandle* H = (NvHandle*)h;
    ORGYM_REQUIRE(state_dev && obs_dev, "state_dev and obs_dev are required");
    DeviceGuard g(H->base.device);
    int64_t N = H->base.num_envs;
    nv_reset_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        H->dev, N, H->npad, state_dev, reseed, seed, env_offset, mask_dev, fixed_params_dev, obs_dev);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

extern "C" int orgym_newsvendor_step(orgym_handle_t h, void* state_dev, const float* actions_dev,
                                     const int64_t* demand_override_dev, int autoreset_mode, float* obs_dev,
                                     double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                                     const orgym_newsvendor_info_t* info, void* stream) {
    if (orgym_check_handle(h, FAM_NEWSVENDOR)) return ORGYM_E_INVALID;
    NvHandle* H = (NvHandle*)h;
    ORGYM_REQUIRE(state_dev && actions_dev && obs_dev && reward_dev && terminated_dev && truncated_dev,
                  "state, actions, obs, reward, terminated and truncated pointers are required");
    ORGYM_REQUIRE(autoreset_mode >= 0 && autoreset_mode <= 2, "bad autoreset mode");
    DeviceGuard g(H->base.device);
    NvStepArgs A;
    memset(&A, 0, sizeof(A));
    A.N = H->base.num_envs;
    A.npad = H->npad;
    A.state = state_dev;
    A.actions = actions_dev;
    A.demand = demand_override_dev;
    A.autoreset = autoreset_mode;
    A.obs = obs_dev;
    A.reward = reward_dev;
    A.terminated = terminated_dev;
    A.truncated = truncated_dev;
    if (info) {
        A.info_demand = info->demand_dev;
        A.info_parts = info->parts_dev;
        ORGYM_REQUIRE(info->info_ld == 0 || info->info_ld >= H->base.num_envs, "info_ld must be 0 (row-major) or >= num_envs");
        A.info_ld = info->info_ld;
        A.final_obs = info->final_obs_dev;
    }
    A.err = H->base.err_dev;
    A.use_bulk = (uintptr_t)obs_dev % 16 == 0;
    size_t smem = (size_t)ORGYM_TILE * (H->dev.obs_dim + 1) * 4;
    orgym_ensure_dyn_smem<nv_step_kernel>(smem);
    nv_step_kernel<<<(unsigned)((A.N + ORGYM_TILE - 1) / ORGYM_TILE), ORGYM_TILE, smem, (cudaStream_t)stream>>>(H->dev, A);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

extern "C" int orgym_newsvendor_export_params(orgym_handle_t h, const void* state_dev, double* params_dev, void* stream) {
    if (orgym_check_handle(h, FAM_NEWSVENDOR)) return ORGYM_E_INVALID;
    NvHandle* H = (NvHandle*)h;
    ORGYM_REQUIRE(state_dev && params_dev, "null argument");
    DeviceGuard g(H->base.device);
    int64_t N = H->base.num_envs;
    nv_export_params_kernel<<<(unsigned)((N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(N, H->npad, H->dev.L, state_dev,
                                                                                         params_dev);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

extern "C" int orgym_newsvendor_rollout(orgym_handle_t h, uint64_t seed, int64_t env_offset, uint32_t episode,
                                        const orgym_newsvendor_rollout_in_t* in,
                                        const orgym_newsvendor_rollout_out_t* out, void* stream) {
    if (orgym_check_handle(h, FAM_NEWSVENDOR)) return ORGYM_E_INVALID;
    NvHandle* H = (NvHandle*)h;
    ORGYM_REQUIRE(in && out, "null argument");
    ORGYM_REQUIRE(in->policy >= 0 && in->policy <= ORGYM_NV_POLICY_MLP, "unknown policy %d", in->policy);
    ORGYM_REQUIRE(in->policy != ORGYM_NV_POLICY_ACTIONS || in->actions_dev, "policy ACTIONS needs actions_dev");
    DeviceGuard g(H->base.device);
    NvRolloutArgs A;
    memset(&A, 0, sizeof(A));
    A.N = H->base.num_envs;
    A.env_offset = env_offset;
    A.seed = seed;
    A.episode = episode;
    A.policy = in->policy;
    A.param0 = in->param[0];
    A.actions = in->actions_dev;
    A.a_se = in->act_stride_env;
    A.a_st = in->act_stride_t;
    A.demand = in->demand_dev;
    A.d_se = in->dem_stride_env;
    A.d_st = in->dem_stride_t;
    A.fixed = in->fixed_params_dev;
    A.ep_return = out->ep_return_dev;
    A.stats = out->stats_dev;
    A.reward_traj = out->reward_traj_dev;
    A.action_traj = out->action_traj_dev;
    A.final_obs = out->final_obs_dev;
    A.partials = out->summary_dev ? H->partials : nullptr;
    if ((in->policy == ORGYM_NV_POLICY_CLASSIC || in->policy == ORGYM_NV_POLICY_SS) && A.ep_return) {
        NvLevelArgs LA;
        memset(&LA, 0, sizeof(LA));
        LA.N = A.N; LA.env_offset = env_offset; LA.seed = seed; LA.episode = episode; LA.policy = in->policy;
        LA.param0 = in->param[0]; LA.fixed = in->fixed_params_dev; LA.level_out = A.ep_return;
        nv_level_kernel<<<(unsigned)((A.N + 255) / 256), 256, 0, (cudaStream_t)stream>>>(H->dev, LA);
        A.level_in = A.ep_return;
    }
    size_t smem = (size_t)H->dev.L * NV_ROLL_THREADS * 4 + 16;
    int nblocks = (int)((A.N + NV_ROLL_THREADS - 1) / NV_ROLL_THREADS);
#define NV_ROLL_CASE(LTV)                                                                          \
    case LTV:                                                                                      \
        orgym_ensure_dyn_smem<nv_rollout_kernel<LTV>>(16);                                         \
        nv_rollout_kernel<LTV><<<nblocks, NV_ROLL_THREADS, 16, (cudaStream_t)stream>>>(H->dev, A); \
        break;
    if (in->policy == ORGYM_NV_POLICY_MLP) {
        NvMlpPlan M;
        if (int rc = nv_mlp_plan(H->dev, in->mlp, &M, &smem)) return rc;
        orgym_ensure_dyn_smem<nv_mlp_rollout_kernel>(smem);
        nv_mlp_rollout_kernel<<<nblocks, MLP_THREADS, smem, (cudaStream_t)stream>>>(H->dev, A, M);
    } else
        switch (H->dev.L) {  // lead times 1..7: register-resident pipeline (see the kernel)
            NV_ROLL_CASE(1) NV_ROLL_CASE(2) NV_ROLL_CASE(3) NV_ROLL_CASE(4) NV_ROLL_CASE(5) NV_ROLL_CASE(6) NV_ROLL_CASE(7)
            default:
                orgym_ensure_dyn_smem<nv_rollout_kernel<0>>(smem);  // + 17 KB static
                nv_rollout_kernel<0><<<nblocks, NV_ROLL_THREADS, smem, (cudaStream_t)stream>>>(H->dev, A);
        }
#undef NV_ROLL_CASE
    ORGYM_CUDA(cudaGetLastError());
    if (out->summary_dev) {
        int rr = orgym_launch_reduce(H->partials, nblocks, out->summary_dev, (cudaStream_t)stream);
        if (rr != ORGYM_OK) return rr;
    }
    return ORGYM_OK;
}
