// invmgmt.cu -- serial multi-echelon env (reference: inventory_management.py).
//
// Kernels (one env instance per thread, all instances independent):
//   inv_reset_kernel    reset (inventory_management.py:186-222) + first observation (:354-391)
//   inv_step_kernel     one period (:224-352) + observation; HBM-bound: struct-of-arrays state is read and
//                       written coalesced, the row-major [env][obs_dim] observation tile and the [env][n] action
//                       tile go through shared memory and the TMA engine (cp.async.bulk)
//   inv_rollout_kernel  fused reset + `periods` steps with on-device policy and Philox demand; on-hand
//                       inventory / backlog in registers, lead-time rings in shared memory; issue-bound
//   inv_mlp_rollout_kernel  the same fused rollout with an MLP actor evaluated on the device every period
//   inv_export_kernel   state export to int64 I / B / period arrays
//
// The rollout kernels write one row of partial sums per 128 envs; orgym_launch_reduce (api.cu) reduces them
// deterministically into the episode summary.  invmgmt_jit.cu generates the specialised rollout kernels.
//
// Integer state is exact (int64, or int32 with a range guard); rewards are float64 evaluated in the reference's
// operation order (no FMA contraction: the library is built with --fmad=false).
#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "launch_util.cuh"
#include "mlp.cuh"
#include <type_traits>

#include "invmgmt_jit.cuh"
#include "jit.cuh"

#define MAXN ORGYM_INV_MAX_STAGES

struct InvDev {
    int n, m, T, backlog, lt_max, obs_dim, sumL;
    int L[MAXN], roff[MAXN];
    uint32_t Lmagic[MAXN], Lm_magic;  // ceil(2^32 / d): t % d without a division (mod_small)
    long long c[MAXN], I0[MAXN];
    double up[MAXN + 1], uc[MAXN + 1], kc[MAXN + 1], hc[MAXN + 1];
    const double* disc;  // [T] alpha**t, computed on the host with libm pow like CPython's float.__pow__
    AliasDev dem;
};

struct InvHandle {
    HandleBase base;
    InvDev dev;
    int wide;
    int64_t npad;
    std::vector<void*> allocs;
    double* partials;  // [max_blocks][8] rollout block partial sums
    int max_blocks;
    // lock-step period of the batch living in `hint_state` (host-side bookkeeping for speculative ring loads;
    // a wrong hint only costs the speculation, never correctness): -1 = unknown
    const void* hint_state;
    int hint_t;
    long long user_dmax;  // largest value of a user_D trace (0 for sampled demand)
    // run-time specialised rollout kernels (invmgmt_jit.cu): one per (policy, base-stock levels), built by
    // orgym_invmgmt_specialise or on the first eligible rollout
    std::vector<double> disc_host;
    struct JitVariant {
        int policy;                 // 0 = base-stock, 1 = random
        long long target[MAXN];     // base-stock levels baked into the kernel
        JitKernel k;
        int failed;                 // compile failed (reason in err): not retried
        std::string err;
    };
    std::vector<JitVariant> jit_variants;
    int last_rollout_jit = 0;       // the most recent rollout (or specialise call) used / built a specialised kernel
};

// ---- state layout: field[slot][env], env stride npad -------------------------------------------------------
// [key u64][S slots: I n | B m | Rring sumL | Aring lt_max*n][period i32][episode u32]
template <typename S>
struct InvState {
    uint64_t* key;
    S* f;
    int32_t* period;
    uint32_t* episode;
    int64_t npad;
    int oI, oB, oR, oA;
    __host__ __device__ InvState(void* base, int64_t npad_, const InvDev& P) : npad(npad_) {
        char* p = (char*)base;
        key = (uint64_t*)p;
        p += 8 * npad;
        f = (S*)p;
        oI = 0;
        oB = P.n;
        oR = P.n + P.m;
        oA = P.n + P.m + P.sumL;
        p += sizeof(S) * npad * (size_t)(oA + P.lt_max * P.n);
        period = (int32_t*)p;
        p += 4 * npad;
        episode = (uint32_t*)p;
    }
    __device__ __forceinline__ S& at(int slot, int64_t e) const { return f[(size_t)slot * npad + e]; }
};
static int64_t inv_state_bytes(const InvDev& P, int64_t npad, int wide) {
    int64_t slots = P.n + P.m + P.sumL + (int64_t)P.lt_max * P.n;
    return npad * (8 + (wide ? 8 : 4) * slots + 8);
}

#define INT32_GUARD (1 << 29)

struct InvStepArgs {
    int64_t N, npad;
    void* state;
    const void* actions;
    int act_f64;
    const int64_t* demand;
    int autoreset;
    int64_t* obs;
    double* reward;
    uint8_t* terminated;
    uint8_t* truncated;
    int64_t* info_demand;
    int64_t* info_sales;
    int64_t* info_unf;
    double* info_profit;
    int direct_obs;  // observation rows too long for a shared-memory tile: write them straight to global memory
    int64_t info_ld;  // 0: sales / unfulfilled row-major [N][m]; > 0: column-major [m][info_ld]
    int64_t* final_obs;
    uint32_t* err;
    int use_bulk;
    int t_hint;  // period every env is expected to be in (lock-step batches), or -1
};

// ---- one period of one env: shared by the step and rollout kernels --------------------------------------------
// in:  t, req[i] (requested order, already max(a,0) truncated), arr[i] = R[t-L_i] for L_i > 0 (0 before t = L_i),
//      d = demand sample.   state: I[], B[] (B[] all-zero in lost-sales mode).
// out: Rf[] fulfilled orders, s0 retail sales, U0 unfulfilled retail demand, profit (undiscounted).
template <int NS, bool EXACT, typename S>
__device__ __forceinline__ double inv_period(const InvDev& P, const S (&req)[NS], const S (&arr)[NS], S d, S (&I)[NS],
                                             S (&B)[NS + 1], S (&Rf)[NS], S& s0_out, S (&U)[NS + 1]) {
    const int n = EXACT ? NS : P.n;
    S cur[NS];
#pragma unroll
    for (int i = 0; i < NS; i++) {
        if (EXACT || i < n) {
            cur[i] = req[i] + B[i + 1];                   // :253-255 (B is zero at t = 0)
            S r = cur[i] < (S)P.c[i] ? cur[i] : (S)P.c[i];  // :263
            if (i + 1 < n) r = I[i + 1] < r ? I[i + 1] : r; // :265 supplier's start-of-period on-hand (may be < 0)
            Rf[i] = r;
        }
    }
    S Ic[NS];
#pragma unroll
    for (int i = 0; i < NS; i++)
        if (EXACT || i < n) Ic[i] = I[i] + (P.L[i] == 0 ? Rf[i] : arr[i]);  // :271-277
    d = d > 0 ? d : 0;                                                      // :280
    S fill = d + B[0];                                                      // :284-286
    S s0 = Ic[0] < fill ? Ic[0] : fill;                                     // :288
    Ic[0] -= s0;
#pragma unroll
    for (int i = 1; i < NS; i++)
        if (EXACT || i < n) Ic[i] -= Rf[i];  // :300 (the stage's own inbound order -- reference quirk)
    U[0] = fill - s0;                        // :303
#pragma unroll
    for (int i = 0; i < NS; i++)
        if (EXACT || i < n) U[i + 1] = cur[i] - Rf[i];  // :304
    // profit :315-321: elementwise float64, then np.sum over the m stages
    double term[NS + 1];
#pragma unroll
    for (int j = 0; j <= NS; j++) {
        if (EXACT || j <= n) {
            S sj = j == 0 ? s0 : Rf[j - 1];
            S inv = 0;
            if (j < n) inv = Ic[j] > 0 ? Ic[j] : 0;
            double s = (double)sj;
            double rev = P.up[j] * s, pc = P.uc[j] * s;
            double pen = P.kc[j] * (double)U[j];
            if (EXACT && j == NS)  // last stage holds no inventory: hc = 0 (:92), x - 0.0 == x
                term[j] = (rev - pc) - pen;
            else {
                double hold = P.hc[j] * (double)inv;
                term[j] = ((rev - pc) - hold) - pen;
            }
        } else
            term[j] = 0.0;
    }
    double profit = np_sum_reg<double, NS + 1>(term, n + 1);
#pragma unroll
    for (int i = 0; i < NS; i++)
        if (EXACT || i < n) I[i] = Ic[i];  // :326
#pragma unroll
    for (int j = 0; j <= NS; j++)
        if (EXACT || j <= n) B[j] = P.backlog ? U[j] : (S)0;  // :307-312
    s0_out = s0;
    return profit;
}

// ---- reset ------------------------------------------------------------------------------------------------------
template <typename S>
__device__ __forceinline__ void inv_reset_env(const InvDev& P, const InvState<S>& st, int64_t e) {
    for (int i = 0; i < P.n; i++) st.at(st.oI + i, e) = (S)P.I0[i];
    for (int j = 0; j < P.m; j++) st.at(st.oB + j, e) = 0;
    for (int k = 0; k < P.sumL; k++) st.at(st.oR + k, e) = 0;
    for (int k = 0; k < P.lt_max * P.n; k++) st.at(st.oA + k, e) = 0;
    st.period[e] = 0;
}

template <typename S>
__global__ void __launch_bounds__(256) inv_reset_kernel(const __grid_constant__ InvDev P, int64_t N, int64_t npad,
                                                        void* state, int reseed, uint64_t seed, int64_t env_offset,
                                                        const uint8_t* __restrict__ mask, int64_t* __restrict__ obs) {
    const int64_t e0 = (int64_t)blockIdx.x * 256, e = e0 + threadIdx.x;
    if (e < N && (!mask || mask[e])) {
        InvState<S> st(state, npad, P);
        inv_reset_env(P, st, e);
        if (reseed) {
            st.key[e] = seed + (uint64_t)(env_offset + e);  // gymnasium vector convention: env i <- seed + i
            st.episode[e] = 0;
        } else
            st.episode[e] += 1;
    }
    // first observation [I0, 0, ...] (:354-391): the CTA fills its 256 rows of the row-major block cooperatively, so the
    // stores are coalesced (a thread writing its own 264-byte row would touch 33 different cache lines per warp store)
    const int W = P.obs_dim;
    const int nrows = (int)((N - e0) < 256 ? (N - e0) : 256);
    int r = 0, c = threadIdx.x;
    while (c >= W) { c -= W; r++; }
    for (int i = threadIdx.x; i < nrows * W; i += 256) {
        if (!mask || mask[e0 + r]) obs[e0 * W + i] = c < P.n ? P.I0[c] : 0;
        c += 256;
        while (c >= W) { c -= W; r++; }
    }
}

// ---- step ------------------------------------------------------------------------------------------------------
#define ORGYM_STEP_MIN_BLOCKS 6
// t % d for 0 <= t < 2^20 and 1 <= d <= 64 without a division: q = mulhi(t, ceil(2^32 / d)) is exact in that range
__device__ __forceinline__ int mod_small(int t, int d, uint32_t magic) {
    return magic ? t - (int)__umulhi((uint32_t)t, magic) * d : 0;  // magic == 0 encodes d == 1
}

// Shared-memory staging tile of the [env][obs_dim] int64 observation block.  With the compact int32 state the tile
// is kept in int32 (half the shared memory -> twice the resident CTAs) and widened to int64 on the way out with
// 16-byte coalesced stores; with the wide state the dense int64 tile leaves through one TMA bulk copy.
template <typename S>
__device__ __forceinline__ void obs_tile_store(int64_t* __restrict__ g, const S* tile, int width, int stride, int nvalid,
                                               bool bulk) {
    if (sizeof(S) == 8 && bulk) {
        fence_async_smem();
        __syncthreads();
        if (threadIdx.x == 0) {
            bulk_s2g(g, tile, (uint32_t)(nvalid * width * 8));
            bulk_commit();
            bulk_wait_read0();
        }
        return;
    }
    __syncthreads();
    const int total = nvalid * width;
    if (stride == width) {  // dense tile: element i of the block is tile[i]
        if (sizeof(S) == 4) {
            const int pairs = total >> 1;
            for (int i = threadIdx.x; i < pairs; i += ORGYM_TILE) {
                int2 v = reinterpret_cast<const int2*>(tile)[i];
                longlong2 w = make_longlong2((long long)v.x, (long long)v.y);
                __stcs(reinterpret_cast<longlong2*>(g) + i, w);
            }
            if ((total & 1) && threadIdx.x == 0) g[total - 1] = (int64_t)tile[total - 1];
        } else {
            for (int i = threadIdx.x; i < total; i += ORGYM_TILE) g[i] = (int64_t)tile[i];
        }
    } else {
        for (int i = threadIdx.x; i < total; i += ORGYM_TILE) {
            int r = i / width, c = i - r * width;
            g[i] = (int64_t)tile[r * stride + c];
        }
    }
}

// One env's observation row: normally a row of the shared-memory staging tile (stored coalesced afterwards); for rows
// that do not fit in shared memory (e.g. 16 stages x lead time 64 = 1040 entries) the row in global memory itself.
template <typename S>
struct ObsRow {
    S* s;
    int64_t* g;  // non-null: direct mode
    __device__ __forceinline__ void put(int k, S v) const {
        if (g)
            g[k] = (int64_t)v;
        else
            s[k] = v;
    }
    __device__ __forceinline__ int64_t get(int k) const { return g ? g[k] : (int64_t)s[k]; }
};

// Lead-time ring slots and the action window of one env for period t (the second group of loads of a step).
// arr[i] = R[t - L_i] (ring slot t % L_i); window positions 0..k-2 of the observation at t+1 go straight into the
// env's row of the staging tile (position k-1 is the current period's request, filled in by the caller).
// All loads of up to CH periods are issued before the first store so that their latencies overlap.
template <int NS, bool EXACT, typename S, int CH>
__device__ __forceinline__ void inv_load_rings(const InvDev& P, const InvState<S>& st, int64_t e, int t, int n,
                                               S (&arr)[NS], const ObsRow<S>& orow) {
    const int Lm = P.lt_max;
    const int tn = t + 1;
    const int k = tn < Lm ? tn : Lm;  // window length at t+1 (:378)
#pragma unroll
    for (int i = 0; i < NS; i++) {
        arr[i] = 0;
        if ((EXACT || i < n) && P.L[i] > 0)
            arr[i] = st.at(st.oR + P.roff[i] + mod_small(t, P.L[i], P.Lmagic[i]), e);  // slot holds R[t-L_i]
    }
    if (Lm > 0) {
        const int slot = mod_small(tn - k, Lm, P.Lm_magic);
        for (int q0 = 0; q0 < Lm; q0 += CH) {
            S v[CH][NS];
#pragma unroll
            for (int u = 0; u < CH; u++) {
                const int q = q0 + u;
                const bool in = q < k - 1;
                int sl = slot + q;
                sl = sl >= Lm ? sl - Lm : sl;
#pragma unroll
                for (int i = 0; i < NS; i++) {
                    v[u][i] = 0;
                    if ((EXACT || i < n) && in) v[u][i] = st.at(st.oA + sl * n + i, e);
                }
            }
#pragma unroll
            for (int u = 0; u < CH; u++) {
                const int q = q0 + u;
                if (q < Lm && q != k - 1) {
#pragma unroll
                    for (int i = 0; i < NS; i++)
                        if (EXACT || i < n) orow.put(n + q * n + i, v[u][i]);
                }
            }
        }
    }
}

template <int NS, bool EXACT, typename S>
__global__ void __launch_bounds__(ORGYM_TILE, (NS <= 4 && sizeof(S) == 4) ? ORGYM_STEP_MIN_BLOCKS : 1)
    inv_step_kernel(const __grid_constant__ InvDev P, const InvStepArgs A) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int CH = NS <= 3 ? 12 : (NS <= 6 ? 6 : 3);  // window periods loaded per batch (<= 36 loads in flight)
    const int n = EXACT ? NS : P.n, m = n + 1;
    const int tid = threadIdx.x;
    const int64_t e0 = (int64_t)blockIdx.x * ORGYM_TILE, e = e0 + tid;
    const int nvalid = (int)((A.N - e0) < ORGYM_TILE ? (A.N - e0) : ORGYM_TILE);
    const bool valid = tid < nvalid;
    const bool full = nvalid == ORGYM_TILE;
    const bool obs_dense = (P.obs_dim & 1) != 0;  // odd row length: conflict-free dense tile
    const int ostride = obs_dense ? P.obs_dim : P.obs_dim + 1;
    const bool bulk_out = A.use_bulk && full && obs_dense;
    const bool bulk_in = A.use_bulk && full;
    // shared: obs tile (S) | action tile (8 B / element) | mbarrier | alias table
    S* obs_tile = (S*)smem;
    size_t off = (!EXACT && A.direct_obs) ? 0 : (((size_t)ORGYM_TILE * ostride * sizeof(S) + 15) & ~(size_t)15);
    unsigned char* act_tile = smem + off;
    off += (size_t)ORGYM_TILE * n * 8;
    uint64_t* bar = (uint64_t*)(smem + off);
    off += 16;
    uint2* tab = (uint2*)(smem + off);

    if (bulk_in && tid == 0) mbar_init(bar, 1);
    __syncthreads();
    if (bulk_in) {
        if (tid == 0) {
            uint32_t bytes = (uint32_t)(ORGYM_TILE * n * 8);
            mbar_expect_tx(bar, bytes);
            bulk_g2s(act_tile, (const char*)A.actions + (size_t)e0 * n * 8, bytes, bar);
        }
    } else {
        const int64_t* src = (const int64_t*)A.actions + (size_t)e0 * n;
        for (int i = tid; i < nvalid * n; i += ORGYM_TILE) ((int64_t*)act_tile)[i] = src[i];
    }
    const bool sample = A.demand == nullptr && P.dem.kind != ORGYM_DIST_USER;
    if (sample)
        for (int i = tid; i < (1 << P.dem.log2k); i += ORGYM_TILE) tab[i] = P.dem.table[i];

    InvState<S> st(A.state, A.npad, P);
    S I[NS], B[NS + 1];
    int t = 0;
    uint32_t episode = 0;
    uint64_t key = 0;
    bool do_step = valid;
    // only the generic instantiation carries the direct mode (the specialised ones keep a compile-time null pointer)
    const bool direct = !EXACT && A.direct_obs;
    const ObsRow<S> orow{obs_tile + tid * ostride, direct ? A.obs + e * P.obs_dim : nullptr};
    S arr[NS];
    const int Lm = P.lt_max;
    // The ring / window addresses depend on the env's period, which itself has to be loaded: two dependent round trips
    // to HBM.  When the batch runs in lock-step the host-side handle knows the period (A.t_hint), so the second group
    // of loads is issued speculatively together with the first; an env whose period differs simply reloads.  Rows in
    // direct mode are not speculated: there the window lands in the caller's row itself, which an env already past
    // the end (autoreset disabled) has to return unchanged.
    const int t_spec = A.t_hint;
    const bool spec = valid && !direct && t_spec >= 0 && t_spec < P.T;
    if (valid) {  // loads that do not depend on the period
        t = st.period[e];
        episode = st.episode[e];
        if (sample) key = st.key[e];
#pragma unroll
        for (int i = 0; i < NS; i++)
            if (EXACT || i < n) I[i] = st.at(st.oI + i, e);
#pragma unroll
        for (int j = 0; j <= NS; j++)
            if (EXACT || j <= n) B[j] = st.at(st.oB + j, e);
    }
    if (spec) inv_load_rings<NS, EXACT, S, CH>(P, st, e, t_spec, n, arr, orow);
    if (valid) {
        if (t >= P.T) {  // episode already over
            do_step = false;
            if (A.autoreset == ORGYM_AUTORESET_NEXT_STEP) {
                inv_reset_env(P, st, e);
                st.episode[e] = episode + 1;
                for (int k = 0; k < P.obs_dim; k++) orow.put(k, k < n ? (S)P.I0[k] : (S)0);
                A.reward[e] = 0.0;
                A.terminated[e] = 0;
                A.truncated[e] = 0;
            } else {  // reference: IndexError on R[t] (inventory_management.py:267)
                atomicOr(A.err, ORGYM_ERR_STEP_PAST_END);
                const int64_t* old = A.obs + e * P.obs_dim;
                if (!direct)
                    for (int k = 0; k < P.obs_dim; k++) orow.put(k, (S)old[k]);
                A.reward[e] = 0.0;
                A.terminated[e] = 0;
                A.truncated[e] = 1;
            }
        }
    }
    if (do_step && !(spec && t == t_spec)) inv_load_rings<NS, EXACT, S, CH>(P, st, e, t, n, arr, orow);
    const int tn = t + 1;
    const int k = tn < Lm ? tn : Lm;  // window length at t+1 (:378)
    if (bulk_in) mbar_wait(bar, 0);
    __syncthreads();  // action tile (cooperative path) and alias table visible

    if (do_step) {
        S req[NS], Rf[NS], U[NS + 1];
        bool range_bad = false;
#pragma unroll
        for (int i = 0; i < NS; i++) {
            if (EXACT || i < n) {
                long long a;
                if (A.act_f64) {
                    double x = ((const double*)act_tile)[tid * n + i];
                    x = x > 0.0 ? x : 0.0;  // np.maximum(action, 0) :250
                    a = (long long)x;       // astype(int64): truncation
                } else {
                    a = ((const long long*)act_tile)[tid * n + i];
                    a = a > 0 ? a : 0;
                }
                if (sizeof(S) == 4 && a > INT32_GUARD) {
                    range_bad = true;
                    a = INT32_GUARD;
                }
                req[i] = (S)a;
            }
        }
        long long dl;
        if (A.demand)
            dl = A.demand[e];
        else
            dl = sample_fixed(P.dem, tab, key, episode, t, 0u);
        if (sizeof(S) == 4 && dl > INT32_GUARD) {
            range_bad = true;
            dl = INT32_GUARD;
        }
        S d = (S)dl, s0;
        double profit = inv_period<NS, EXACT, S>(P, req, arr, d, I, B, Rf, s0, U);
        double reward = P.disc[t] * profit;  // :322
        if (sizeof(S) == 4) {
#pragma unroll
            for (int i = 0; i < NS; i++)
                if (EXACT || i < n) range_bad |= (I[i] > INT32_GUARD) | (I[i] < -INT32_GUARD);
#pragma unroll
            for (int j = 0; j <= NS; j++)
                if (EXACT || j <= n) range_bad |= (U[j] > INT32_GUARD) | (U[j] < -INT32_GUARD);
            if (range_bad) atomicOr(A.err, ORGYM_ERR_INT32_RANGE);
        }
        const bool trunc = tn >= P.T;  // :350
        const bool reset_now = trunc && A.autoreset == ORGYM_AUTORESET_SAME_STEP;
        // finish the observation row: on-hand inventory and the current period's requested order
#pragma unroll
        for (int i = 0; i < NS; i++)
            if (EXACT || i < n) {
                orow.put(i, I[i]);
                if (Lm > 0) orow.put(n + (k - 1) * n + i, req[i]);
            }
        if (!reset_now) {
            const int aslot = Lm > 0 ? mod_small(t, Lm, P.Lm_magic) : 0;
#pragma unroll
            for (int i = 0; i < NS; i++)
                if (EXACT || i < n) {
                    st.at(st.oI + i, e) = I[i];
                    if (P.L[i] > 0) st.at(st.oR + P.roff[i] + mod_small(t, P.L[i], P.Lmagic[i]), e) = Rf[i];
                    if (Lm > 0) st.at(st.oA + aslot * n + i, e) = req[i];
                }
#pragma unroll
            for (int j = 0; j <= NS; j++)
                if (EXACT || j <= n) st.at(st.oB + j, e) = B[j];
            st.period[e] = tn;
        } else {
            // SAME_STEP autoreset: the terminal observation goes to final_obs, the env restarts immediately
            if (A.final_obs) {
                int64_t* fo = A.final_obs + e * P.obs_dim;
                for (int q = 0; q < P.obs_dim; q++) fo[q] = orow.get(q);
            }
            inv_reset_env(P, st, e);
            st.episode[e] = episode + 1;
            for (int q = 0; q < P.obs_dim; q++) orow.put(q, q < n ? (S)P.I0[q] : (S)0);
        }
        A.reward[e] = reward;
        A.terminated[e] = 0;  // :349
        A.truncated[e] = trunc ? 1 : 0;
        if (A.info_demand) A.info_demand[e] = (int64_t)(d > 0 ? d : 0);
        if (A.info_profit) A.info_profit[e] = profit;
        if (A.info_sales || A.info_unf) {
            // each env owns m consecutive int64: pairs go out as 16-byte stores when the row is 16-byte aligned
            long long sv[NS + 1];
            sv[0] = (long long)s0;
#pragma unroll
            for (int i = 0; i < NS; i++) sv[i + 1] = (EXACT || i < n) ? (long long)Rf[i] : 0;
            if (A.info_ld) {  // column-major: one coalesced 8-byte store per stage
#pragma unroll
                for (int j = 0; j <= NS; j++)
                    if (EXACT || j <= n) {
                        if (A.info_sales) A.info_sales[(int64_t)j * A.info_ld + e] = sv[j];
                        if (A.info_unf) A.info_unf[(int64_t)j * A.info_ld + e] = (long long)U[j];
                    }
            } else {
                if (A.info_sales) {
                    int64_t* row = A.info_sales + e * m;
                    if (EXACT && (((NS + 1) & 1) == 0)) {
#pragma unroll
                        for (int j = 0; j < NS + 1; j += 2)
                            *reinterpret_cast<longlong2*>(row + j) = make_longlong2(sv[j], sv[j + 1 <= NS ? j + 1 : NS]);
                    } else {
#pragma unroll
                        for (int j = 0; j <= NS; j++)
                            if (EXACT || j <= n) row[j] = sv[j];
                    }
                }
                if (A.info_unf) {
                    int64_t* row = A.info_unf + e * m;
                    if (EXACT && (((NS + 1) & 1) == 0)) {
#pragma unroll
                        for (int j = 0; j < NS + 1; j += 2)
                            *reinterpret_cast<longlong2*>(row + j) =
                                make_longlong2((long long)U[j], (long long)U[j + 1 <= NS ? j + 1 : NS]);
                    } else {
#pragma unroll
                        for (int j = 0; j <= NS; j++)
                            if (EXACT || j <= n) row[j] = (long long)U[j];
                    }
                }
            }
        }
    }
    if (!direct) obs_tile_store<S>(A.obs + (size_t)e0 * P.obs_dim, obs_tile, P.obs_dim, ostride, nvalid, bulk_out);
}

// ---- export -----------------------------------------------------------------------------------------------------
template <typename S>
__global__ void inv_export_kernel(const __grid_constant__ InvDev P, int64_t N, int64_t npad, const void* state,
                                  int64_t* __restrict__ I, int64_t* __restrict__ B, int32_t* __restrict__ period) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    InvState<S> st((void*)state, npad, P);
    if (I)
        for (int i = 0; i < P.n; i++) I[e * P.n + i] = (int64_t)st.at(st.oI + i, e);
    if (B)
        for (int j = 0; j < P.m; j++) B[e * P.m + j] = (int64_t)st.at(st.oB + j, e);
    if (period) period[e] = st.period[e];
}

// ---- fused rollout ----------------------------------------------------------------------------------------------
struct InvRolloutArgs {
    int64_t N, env_offset;
    uint64_t seed;
    uint32_t episode;
    int policy;
    double target[MAXN];  // base-stock levels (L_i+1)*mu*sf as float64
    long long target_int[MAXN];
    int target_is_int;    // every level is an integer below 2^30: the policy is evaluated in integers (same result)
    int rroff[MAXN], rslots;  // rollout ring layout: stage i owns max(L_i, 1) slots starting at rroff[i]
    const int64_t* actions;
    int64_t a_se, a_st;
    const int64_t* demand;
    int64_t d_se, d_st;
    double* ep_return;
    int64_t* stats;
    double* reward_traj;
    int64_t* final_I;
    int64_t* final_B;
    int32_t* stats32;
    int64_t* action_traj;  // [N][T][n]
    double* partials;  // [ceil(N / ROLL_THREADS)][8]: one row per 128 envs, whatever the CTA size
    void* ring_scratch;    // non-null: the rings do not fit in shared memory and live here as [slot][ring_stride]
    int64_t ring_stride;   // >= round_up(N, ROLL_THREADS)
};

#define ROLL_THREADS 128

// ---- pieces shared by the fused rollout kernels (inv_rollout_kernel, inv_mlp_rollout_kernel) --------------------------
// per-episode accumulators of one env; the statistics are kept in the state type: the int32 instantiations are only
// launched when the host has bounded every per-episode sum below 2^31 (orgym_invmgmt_rollout), otherwise S = int64
template <typename S>
struct InvRollAcc {
    double ret;
    S sales, dem, stock, inv;
};

// one period after the policy has chosen req[]: lead-time ring slot rbase + rpos holds R[t - L_i] (zero before t = L_i)
// and receives this period's fulfilled order; demand is replayed, a user trace or one Philox block per four periods
// through the alias table.  The caller advances the ring positions.
template <int NS, bool EXACT, typename S, typename RI>
__device__ __forceinline__ void inv_roll_period(const InvDev& P, const InvRolloutArgs& A, const uint2* tab, uint64_t key,
                                                int64_t e, bool valid, int t, int n, const S (&req)[NS], S* rring,
                                                const RI (&rbase)[NS], const RI (&rpos)[NS], S (&I)[NS], S (&B)[NS + 1],
                                                uint4& w, InvRollAcc<S>& acc, double* rtraj) {
    S arr[NS], Rf[NS], U[NS + 1];
#pragma unroll
    for (int i = 0; i < NS; i++)
        if (EXACT || i < n) arr[i] = rring[rbase[i] + rpos[i]];
    long long dl;
    if (A.demand)
        dl = valid ? A.demand[e * A.d_se + (int64_t)t * A.d_st] : 0;
    else if (P.dem.kind == ORGYM_DIST_USER)
        dl = t < P.dem.user_D_len ? P.dem.user_D[t] : 0;
    else {
        if ((t & 3) == 0) w = philox_block(key, (uint32_t)t >> 2, A.episode, STREAM_DEMAND, 0u);
        dl = alias_draw(tab, P.dem.log2k, P.dem.base, pick_word(w, t & 3));
    }
    S s0;
    double profit = inv_period<NS, EXACT, S>(P, req, arr, (S)dl, I, B, Rf, s0, U);
    double reward = P.disc[t] * profit;
    acc.ret += reward;  // Python: total += reward, in period order
    if (rtraj) rtraj[t] = reward;
    acc.sales += s0;
    acc.dem += (S)dl > 0 ? (S)dl : (S)0;
    acc.stock += U[0];
#pragma unroll
    for (int i = 0; i < NS; i++)
        if (EXACT || i < n) acc.inv += I[i] > 0 ? I[i] : (S)0;
#pragma unroll
    for (int i = 0; i < NS; i++)
        if (EXACT || i < n) rring[rbase[i] + rpos[i]] = Rf[i];
}

// per-episode outputs of one env
template <int NS, typename S>
__device__ __forceinline__ void inv_roll_outputs(const InvRolloutArgs& A, int64_t e, int n, const InvRollAcc<S>& acc,
                                                 const S (&I)[NS], const S (&B)[NS + 1]) {
    if (A.ep_return) A.ep_return[e] = acc.ret;
    if (A.stats) {
        longlong4 v = make_longlong4((long long)acc.sales, (long long)acc.dem, (long long)acc.stock, (long long)acc.inv);
        *reinterpret_cast<longlong4*>(A.stats + e * 4) = v;
    }
    if (A.stats32) {
        auto sat = [](long long v) { return (int)(v > 2147483647LL ? 2147483647LL : (v < -2147483648LL ? -2147483648LL : v)); };
        *reinterpret_cast<int4*>(A.stats32 + e * 4) =
            make_int4(sat((long long)acc.sales), sat((long long)acc.dem), sat((long long)acc.stock), sat((long long)acc.inv));
    }
    if (A.final_I)
        for (int i = 0; i < n; i++) A.final_I[e * n + i] = (int64_t)I[i];
    if (A.final_B)
        for (int j = 0; j <= n; j++) A.final_B[e * (n + 1) + j] = (int64_t)B[j];
}

// batch summary, first stage: the 7 sums of one warp of 32 consecutive envs (butterfly shuffles) into red[7]
template <typename S>
__device__ __forceinline__ void inv_roll_warp_sums(bool valid, const InvRollAcc<S>& acc, double* red) {
    double v[7];
    v[0] = valid ? 1.0 : 0.0;
    v[1] = valid ? acc.ret : 0.0;
    v[2] = valid ? acc.ret * acc.ret : 0.0;
    v[3] = valid ? (double)acc.sales : 0.0;
    v[4] = valid ? (double)acc.dem : 0.0;
    v[5] = valid ? (double)acc.stock : 0.0;
    v[6] = valid ? (double)acc.inv : 0.0;
#pragma unroll
    for (int q = 0; q < 7; q++) {
        double x = v[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if ((threadIdx.x & 31) == 0) red[q] = x;
    }
}

// second stage (threads 0..6, after a barrier): the four warp rows of 128 envs, in warp order, into one partials row
__device__ __forceinline__ void inv_roll_partials_row(const double (*red)[7], double* row) {
    const int q = threadIdx.x;
    if (q < 7) {
        double x = 0.0;
        for (int wv = 0; wv < ROLL_THREADS / 32; wv++) x += red[wv][q];
        row[q] = x;
    }
}

template <int NS, bool EXACT, typename S>
__global__ void __launch_bounds__(ROLL_THREADS) inv_rollout_kernel(const __grid_constant__ InvDev P,
                                                                   const __grid_constant__ InvRolloutArgs A) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int n = EXACT ? NS : P.n;
    const int tid = threadIdx.x;
    const int64_t e = (int64_t)blockIdx.x * ROLL_THREADS + tid;
    const bool valid = e < A.N;
    const bool need_aring = A.policy == ORGYM_POLICY_BASE_STOCK;
    // shared: alias table | R rings [rslots][threads] | request rings [rslots][threads] (base-stock only).
    // Every stage owns max(L_i, 1) ring slots so that the ring traffic below is branch-free (a stage with L_i = 0
    // reads and writes a dummy slot whose value is never used).
    uint2* tab = (uint2*)smem;
    const int K = (P.dem.kind == ORGYM_DIST_USER) ? 0 : (1 << P.dem.log2k);
    // Rings too long for shared memory (sum of lead times in the hundreds) fall back to a global scratch buffer with
    // the same [slot][lane] indexing; only the generic instantiation carries that mode.
    const bool gring = !EXACT && A.ring_scratch != nullptr;
    typedef typename std::conditional<EXACT, int, long long>::type RI;  // ring offsets (elements)
    const RI rstride = gring ? (RI)A.ring_stride : (RI)ROLL_THREADS;
    const RI lane = gring ? (RI)e : (RI)tid;
    S* rring = gring ? (S*)A.ring_scratch : (S*)(smem + (size_t)K * 8);
    S* aring = rring + (size_t)A.rslots * (size_t)rstride;
    for (int i = tid; i < K; i += ROLL_THREADS) tab[i] = P.dem.table[i];
    for (int k = 0; k < A.rslots; k++) {
        rring[k * rstride + lane] = 0;
        if (need_aring) aring[k * rstride + lane] = 0;
    }
    __syncthreads();

    const uint64_t key = A.seed + (uint64_t)(A.env_offset + e);
    S I[NS], B[NS + 1], psum[NS], lmask[NS];
    RI rbase[NS], rpos[NS], rlen[NS];  // ring base / position / length in elements of the [slot][lane] layout
#pragma unroll
    for (int i = 0; i < NS; i++) {
        I[i] = (EXACT || i < n) ? (S)P.I0[i] : (S)0;
        psum[i] = 0;
        rbase[i] = A.rroff[i] * rstride + lane;
        rpos[i] = 0;
        rlen[i] = (P.L[i] > 0 ? P.L[i] : 1) * rstride;
        lmask[i] = P.L[i] > 0 ? (S)-1 : (S)0;
    }
#pragma unroll
    for (int j = 0; j <= NS; j++) B[j] = 0;
    InvRollAcc<S> acc = {0.0, 0, 0, 0, 0};
    uint4 w = make_uint4(0, 0, 0, 0);
    double* const rtraj = (A.reward_traj && valid) ? A.reward_traj + e * P.T : nullptr;
    int64_t* const atraj = (A.action_traj && valid) ? A.action_traj + e * P.T * n : nullptr;

    for (int t = 0; t < P.T; t++) {
        S req[NS];
        // ---- policy ---------------------------------------------------------------------------------------
        if (A.policy == ORGYM_POLICY_BASE_STOCK) {
            // benchmark_InvManagementBacklogEnv.py:152-198: position = on-hand + requested orders of the last L_i
            // periods; q = clip(max(0, target - position), 0, c) in float64, truncated to int64.  With an
            // integer-valued target the float64 expression is exact, so it is evaluated in integers.
            if (A.target_is_int) {
#pragma unroll
                for (int i = 0; i < NS; i++)
                    if (EXACT || i < n) {  // |target|, |I + psum| < 2^30 (range guard): no overflow in S
                        S q = (S)A.target_int[i] - (I[i] + psum[i]);
                        q = q > 0 ? q : 0;
                        q = q < (S)P.c[i] ? q : (S)P.c[i];
                        req[i] = q;
                    }
            } else {
#pragma unroll
                for (int i = 0; i < NS; i++)
                    if (EXACT || i < n) {
                        double q = A.target[i] - (double)(I[i] + psum[i]);
                        q = q > 0.0 ? q : 0.0;
                        double cap = (double)P.c[i];
                        q = q < cap ? q : cap;
                        req[i] = (S)(long long)q;
                    }
            }
        } else if (A.policy == ORGYM_POLICY_RANDOM) {
            uint4 a4 = make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int i = 0; i < NS; i++)
                if (EXACT || i < n) {
                    if ((i & 3) == 0) a4 = philox_block(key, (uint32_t)t, A.episode, STREAM_ACTION, (uint32_t)(i >> 2));
                    uint32_t u = (i & 3) == 0 ? a4.x : (i & 3) == 1 ? a4.y : (i & 3) == 2 ? a4.z : a4.w;
                    req[i] = (S)mulhi32(u, (uint32_t)P.c[i] + 1u);  // uniform on {0..c_i}
                }
        } else {
#pragma unroll
            for (int i = 0; i < NS; i++)
                if (EXACT || i < n) {
                    long long a = valid ? A.actions[e * A.a_se + (int64_t)t * A.a_st + i] : 0;
                    a = a > 0 ? a : 0;
                    req[i] = (S)a;
                }
        }
        if (atraj)
#pragma unroll
            for (int i = 0; i < NS; i++)
                if (EXACT || i < n) atraj[t * n + i] = (int64_t)req[i];
        inv_roll_period<NS, EXACT, S, RI>(P, A, tab, key, e, valid, t, n, req, rring, rbase, rpos, I, B, w, acc, rtraj);
        // ---- request ring (base-stock position) and ring advance (branch-free) ----------------------------------
#pragma unroll
        for (int i = 0; i < NS; i++)
            if (EXACT || i < n) {
                if (need_aring) {
                    const RI slot = rbase[i] + rpos[i];
                    S old = aring[slot];
                    aring[slot] = req[i];
                    psum[i] = (psum[i] + req[i] - old) & lmask[i];  // stays 0 for a stage without lead time
                }
                const RI np1 = rpos[i] + rstride;
                rpos[i] = np1 == rlen[i] ? 0 : np1;
            }
    }
    // ---- per-episode outputs --------------------------------------------------------------------------------------
    if (valid) inv_roll_outputs<NS, S>(A, e, n, acc, I, B);
    // ---- batch summary: warp shuffles -> one row of partials per CTA (summed in fixed order afterwards) -------
    if (A.partials) {
        __shared__ double red[ROLL_THREADS / 32][7];
        inv_roll_warp_sums<S>(valid, acc, red[tid >> 5]);
        __syncthreads();
        inv_roll_partials_row(red, A.partials + (size_t)blockIdx.x * 8);
    }
}

// ---- fused rollout driven by an MLP actor (ORGYM_POLICY_MLP) ----------------------------------------------------------
// One CTA = 128 consecutive envs (one row of the partial sums, like inv_rollout_kernel), run as 128/E sub-tiles of E
// envs one after the other; weights and biases are staged in shared memory once per CTA.  Thread tid < E owns env
// e0 + tid of the current sub-tile (integer state in registers, lead-time ring in shared memory).  Per period the whole
// CTA evaluates the network on the sub-tile's observations (mlp.cuh: register-tiled SGEMM on feature-major tiles).  The
// observation tile itself is the request window (shifted in place).
struct InvMlpPlan {
    int L, act, E, log2E;
    int K[ORGYM_MLP_MAX_LAYERS + 1];   // widths
    int Np[ORGYM_MLP_MAX_LAYERS];      // output widths of the hidden layers padded to MLP_TN (zero weights and biases)
    const float* W[ORGYM_MLP_MAX_LAYERS];
    const float* b[ORGYM_MLP_MAX_LAYERS];
    // shared memory: alias table at 0 | float area at fbase (offsets in floats) | lead-time ring at ring_off (bytes)
    int w_off[ORGYM_MLP_MAX_LAYERS], b_off[ORGYM_MLP_MAX_LAYERS], obs_off, buf_off[2], y_off;
    int fbase, ring_off;
};

template <int NS, bool EXACT, typename S>
__global__ void __launch_bounds__(MLP_THREADS, (EXACT && NS <= 4 && sizeof(S) == 4) ? 3 : 2) inv_mlp_rollout_kernel(const __grid_constant__ InvDev P,
                                                                      const __grid_constant__ InvRolloutArgs A,
                                                                      const __grid_constant__ InvMlpPlan M) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ double red[ROLL_THREADS / 32][7];
    const int n = EXACT ? NS : P.n;
    const int tid = threadIdx.x;
    const int E = M.E, L = M.L;
    uint2* tab = (uint2*)smem;
    float* fs = (float*)(smem + M.fbase);
    S* rring = (S*)(smem + M.ring_off);
    float* obs = fs + M.obs_off;
    float* y = fs + M.y_off;
    const int K = (P.dem.kind == ORGYM_DIST_USER) ? 0 : (1 << P.dem.log2k);
    for (int i = tid; i < K; i += MLP_THREADS) tab[i] = P.dem.table[i];
    // weights: hidden layers transposed to [k][Np] (zero-padded columns), the last layer as given ([n][K] row-major)
    mlp_stage_weights(M, fs);
    const int Lm = P.lt_max, od = P.obs_dim;
    const int Klast = M.K[L - 1];
    const float* Wlast = fs + M.w_off[L - 1];
    const float* blast = fs + M.b_off[L - 1];
    const float* hin = L == 1 ? obs : fs + M.buf_off[(L - 2) & 1];  // input of the last layer
    const int nsub = ROLL_THREADS / E;
    for (int sub = 0; sub < nsub; sub++) {
        const int64_t e0 = (int64_t)blockIdx.x * ROLL_THREADS + (int64_t)sub * E;
        const bool owner = tid < E;
        const int64_t e = e0 + tid;
        const bool valid = owner && e < A.N;
        if (e0 >= A.N) {  // CTA-uniform: the sums of the missing warps are zero, like idle lanes of inv_rollout_kernel
            if (tid < 7 * (E / 32)) red[sub * (E / 32) + tid / 7][tid % 7] = 0.0;
            continue;
        }
        const uint64_t key = A.seed + (uint64_t)(A.env_offset + e);
        S I[NS], B[NS + 1];
        int rbase[NS], rpos[NS], rlen[NS];
#pragma unroll
        for (int i = 0; i < NS; i++) {
            I[i] = (EXACT || i < n) ? (S)P.I0[i] : (S)0;
            rbase[i] = A.rroff[i] * E + tid;
            rpos[i] = 0;
            rlen[i] = (P.L[i] > 0 ? P.L[i] : 1) * E;
        }
#pragma unroll
        for (int j = 0; j <= NS; j++) B[j] = 0;
        InvRollAcc<S> acc = {0.0, 0, 0, 0, 0};
        uint4 w = make_uint4(0, 0, 0, 0);
        double* const rtraj = (A.reward_traj && valid) ? A.reward_traj + e * P.T : nullptr;
        int64_t* const atraj = (A.action_traj && valid) ? A.action_traj + e * P.T * n : nullptr;
        if (owner) {  // first observation [I0, 0, ...] and empty rings
            for (int k = 0; k < od; k++) obs[k * E + tid] = k < n ? (float)(S)P.I0[k] : 0.f;
            for (int k = 0; k < A.rslots; k++) rring[k * E + tid] = 0;
        }
        __syncthreads();
        for (int t = 0; t < P.T; t++) {
            // ---- policy: the network on the observation tile ------------------------------------------------------
            const float* in = obs;
            for (int l = 0; l < L - 1; l++) {
                float* out = fs + M.buf_off[l & 1];
                mlp_hidden_layer(in, out, fs + M.w_off[l], fs + M.b_off[l], M.K[l], M.Np[l], E, M.log2E, M.act);
                __syncthreads();
                in = out;
            }
            for (int idx = tid; idx < n * E; idx += MLP_THREADS) {  // last layer: one output of one env per thread
                const int i = idx >> M.log2E, ee = idx & (E - 1);
                const float* wr = Wlast + i * Klast;
                float a = blast[i];
                for (int k = 0; k < Klast; k++) a = __fmaf_rn(wr[k], hin[k * E + ee], a);
                y[idx] = a;
            }
            __syncthreads();
            if (owner) {
                S req[NS];
#pragma unroll
                for (int i = 0; i < NS; i++)
                    if (EXACT || i < n) {  // clip to [0, c_i] in float64 (NaN -> 0), truncate (:250)
                        double v = (double)y[i * E + tid];
                        v = v > 0.0 ? v : 0.0;
                        const double cap = (double)P.c[i];
                        v = v < cap ? v : cap;
                        req[i] = (S)(long long)v;
                    }
                if (atraj)
#pragma unroll
                    for (int i = 0; i < NS; i++)
                        if (EXACT || i < n) atraj[t * n + i] = (int64_t)req[i];
                inv_roll_period<NS, EXACT, S, int>(P, A, tab, key, e, valid, t, n, req, rring, rbase, rpos, I, B, w, acc,
                                                   rtraj);
#pragma unroll
                for (int i = 0; i < NS; i++)
                    if (EXACT || i < n) {
                        const int np1 = rpos[i] + E;
                        rpos[i] = np1 == rlen[i] ? 0 : np1;
                    }
                // ---- observation of period t+1: I, then the window of the last min(t+1, lt_max) requests -----------
#pragma unroll
                for (int i = 0; i < NS; i++)
                    if (EXACT || i < n) obs[i * E + tid] = (float)I[i];
                if (Lm > 0) {
                    int q = t;
                    if (t >= Lm) {  // full window: drop the oldest request
                        for (int k = n; k < od - n; k++) obs[k * E + tid] = obs[(k + n) * E + tid];
                        q = Lm - 1;
                    }
#pragma unroll
                    for (int i = 0; i < NS; i++)
                        if (EXACT || i < n) obs[(n + q * n + i) * E + tid] = (float)req[i];
                }
            }
            __syncthreads();
        }
        if (valid) inv_roll_outputs<NS, S>(A, e, n, acc, I, B);
        if (A.partials && owner) inv_roll_warp_sums<S>(valid, acc, red[sub * (E / 32) + (tid >> 5)]);
    }
    if (A.partials) {
        __syncthreads();
        inv_roll_partials_row(red, A.partials + (size_t)blockIdx.x * 8);
    }
}

// ------------------------------------------------------------------------------------------------
// host side of the C ABI
// ------------------------------------------------------------------------------------------------
// The fields of InvDev a configuration determines, without validation (orgym_invmgmt_create validates like the
// reference first).  The price arrays may be absent (orgym_invmgmt_value_bounds without profit_mag): prices stay 0.
static void inv_dev_from_config(const orgym_invmgmt_config_t* cfg, InvDev* P) {
    const int n = cfg->num_stages - 1;
    memset(P, 0, sizeof(*P));
    P->n = n;
    P->m = n + 1;
    P->T = cfg->periods;
    P->backlog = cfg->backlog ? 1 : 0;
    for (int i = 0; i < n; i++) {
        P->I0[i] = cfg->init_inv[i];
        P->c[i] = cfg->capacity[i];
        P->L[i] = (int)cfg->lead_time[i];
        P->roff[i] = P->sumL;
        P->sumL += P->L[i];
        if (P->L[i] > P->lt_max) P->lt_max = P->L[i];
    }
    if (cfg->unit_price && cfg->unit_cost && cfg->demand_cost && cfg->holding_cost)
        for (int j = 0; j <= n; j++) {
            P->up[j] = cfg->unit_price[j];
            P->uc[j] = cfg->unit_cost[j];
            P->kc[j] = cfg->demand_cost[j];
            P->hc[j] = cfg->holding_cost[j];
        }
    P->obs_dim = n * (P->lt_max + 1);
    for (int i = 0; i < n; i++) P->Lmagic[i] = P->L[i] > 1 ? (uint32_t)((0x100000000ULL + P->L[i] - 1) / P->L[i]) : 0u;
    P->Lm_magic = P->lt_max > 1 ? (uint32_t)((0x100000000ULL + P->lt_max - 1) / P->lt_max) : 0u;
}

// alpha**t for t = 0..T-1 with libm pow, like CPython's float ** int
static std::vector<double> inv_discounts(double alpha, int T) {
    std::vector<double> disc((size_t)T);
    for (int t = 0; t < T; t++) disc[(size_t)t] = std::pow(alpha, (double)t);
    return disc;
}

// log2 of the alias-table size and the support's base of a sampled demand distribution (as orgym_build_alias builds it)
static int inv_demand_table(const orgym_dist_t* d, int* log2k, int64_t* base) {
    std::vector<double> pmf;
    if (int rc = orgym_dist_pmf(d, &pmf, base)) return rc;
    *log2k = 0;
    while ((size_t(1) << *log2k) < pmf.size()) ++*log2k;
    return ORGYM_OK;
}

// shared memory of the demand's alias table staged by the step and rollout kernels (a user trace stages none)
static size_t inv_alias_smem(const InvDev& P) { return P.dem.kind == ORGYM_DIST_USER ? 0 : (size_t(8) << P.dem.log2k); }
// dynamic shared memory above which the step kernel writes observations directly and the rollout kernel keeps its
// lead-time rings in global scratch (correct, not fast)
#define INV_STAGING_SMEM_LIMIT (200 * 1024)

template <typename S>
static void launch_step(const InvHandle* H, const InvStepArgs& A, size_t smem, cudaStream_t s) {
    const InvDev& P = H->dev;
    unsigned grid = (unsigned)((A.N + ORGYM_TILE - 1) / ORGYM_TILE);
#define STEP_CASE(NSV)                                                                                              \
    case NSV:                                                                                                       \
        orgym_ensure_dyn_smem<inv_step_kernel<NSV, true, S>>(smem);                                                  \
        inv_step_kernel<NSV, true, S><<<grid, ORGYM_TILE, smem, s>>>(P, A);                                          \
        break;
    switch (A.direct_obs ? 0 : P.n) {
        STEP_CASE(1) STEP_CASE(2) STEP_CASE(3) STEP_CASE(4) STEP_CASE(5) STEP_CASE(6) STEP_CASE(7) STEP_CASE(8)
        default:
            orgym_ensure_dyn_smem<inv_step_kernel<MAXN, false, S>>(smem);
            inv_step_kernel<MAXN, false, S><<<grid, ORGYM_TILE, smem, s>>>(P, A);
    }
#undef STEP_CASE
}

template <typename S>
static void launch_rollout(const InvHandle* H, const InvRolloutArgs& A, size_t smem, cudaStream_t s) {
    const InvDev& P = H->dev;
    unsigned grid = (unsigned)((A.N + ROLL_THREADS - 1) / ROLL_THREADS);
#define ROLL_CASE(NSV)                                                                                                 \
    case NSV:                                                                                                          \
        orgym_ensure_dyn_smem<inv_rollout_kernel<NSV, true, S>>(smem);                                               \
        inv_rollout_kernel<NSV, true, S><<<grid, ROLL_THREADS, smem, s>>>(P, A);                                        \
        break;
    switch (A.ring_scratch ? 0 : P.n) {
        ROLL_CASE(1) ROLL_CASE(2) ROLL_CASE(3) ROLL_CASE(4) ROLL_CASE(5) ROLL_CASE(6) ROLL_CASE(7) ROLL_CASE(8)
        default:
            orgym_ensure_dyn_smem<inv_rollout_kernel<MAXN, false, S>>(smem);
            inv_rollout_kernel<MAXN, false, S><<<grid, ROLL_THREADS, smem, s>>>(P, A);
    }
#undef ROLL_CASE
}

template <typename S>
static void launch_mlp_rollout(const InvHandle* H, const InvRolloutArgs& A, const InvMlpPlan& M, size_t smem,
                               cudaStream_t s) {
    const InvDev& P = H->dev;
    unsigned grid = (unsigned)((A.N + ROLL_THREADS - 1) / ROLL_THREADS);
#define MLP_CASE(NSV)                                                                                                  \
    case NSV:                                                                                                          \
        orgym_ensure_dyn_smem<inv_mlp_rollout_kernel<NSV, true, S>>(smem);                                           \
        inv_mlp_rollout_kernel<NSV, true, S><<<grid, MLP_THREADS, smem, s>>>(P, A, M);                                 \
        break;
    switch (P.n) {
        MLP_CASE(1) MLP_CASE(2) MLP_CASE(3) MLP_CASE(4) MLP_CASE(5) MLP_CASE(6)
        default:
            orgym_ensure_dyn_smem<inv_mlp_rollout_kernel<MAXN, false, S>>(smem);
            inv_mlp_rollout_kernel<MAXN, false, S><<<grid, MLP_THREADS, smem, s>>>(P, A, M);
    }
#undef MLP_CASE
}

// Checks an orgym_mlp_t against the handle (ORGYM_E_INVALID) and lays out one CTA's shared memory for it: the largest
// sub-tile of E in {64, 32} envs whose working set fits (ORGYM_E_UNSUPPORTED, with the sizes, when none does).
static int inv_mlp_plan(const InvDev& P, const orgym_mlp_t* mlp, int rslots, size_t ring_elem, InvMlpPlan* M,
                        size_t* smem_out) {
    ORGYM_REQUIRE(mlp, "policy ORGYM_POLICY_MLP needs in->mlp");
    MlpNet net;
    if (int rc = mlp_net_plan(mlp, P.obs_dim, P.n, "the action dimension m-1", &net)) return rc;
    const int L = net.L;
    memset(M, 0, sizeof(*M));
    M->L = L;
    M->act = net.act;
    for (int l = 0; l <= L; l++) M->K[l] = net.K[l];
    for (int l = 0; l < L; l++) {
        M->W[l] = net.W[l];
        M->b[l] = net.b[l];
        M->Np[l] = net.Np[l];
        M->w_off[l] = net.w_off[l];
        M->b_off[l] = net.b_off[l];
    }
    auto a4 = [](int x) { return (int)round_up(x, 4); };  // float offsets stay 16-byte aligned
    const int wfloats = net.wfloats, hmax = net.hmax;
    const size_t tab = inv_alias_smem(P);
    const int nbuf = L >= 3 ? 2 : (L == 2 ? 1 : 0);
    size_t smem = 0;
    for (int E = 64; E >= 32; E /= 2) {
        int g = wfloats;
        M->obs_off = g;
        g += P.obs_dim * E;
        M->buf_off[0] = g;
        g += nbuf >= 1 ? hmax * E : 0;
        M->buf_off[1] = g;
        g += nbuf >= 2 ? hmax * E : 0;
        M->y_off = g;
        g += a4(P.n * E);
        M->fbase = (int)round_up((int64_t)tab, 16);
        M->ring_off = (int)round_up(M->fbase + (int64_t)g * 4, 16);
        smem = (size_t)M->ring_off + (size_t)rslots * E * ring_elem;
        M->E = E;
        M->log2E = E == 64 ? 6 : 5;
        if (smem <= MLP_SMEM_BUDGET) break;
    }
    if (smem > MLP_SMEM_BUDGET) {
        orgym_set_error("mlp: one CTA of 32 envs needs %zu bytes of shared memory (weights and biases %d floats, observation "
                        "tile %d x 32, %d activation tile(s) %d x 32, lead-time rings %d slots); this build's limit is %d",
                        smem, wfloats, P.obs_dim, nbuf, hmax, rslots, MLP_SMEM_BUDGET);
        return ORGYM_E_UNSUPPORTED;
    }
    *smem_out = smem;
    return ORGYM_OK;
}

extern "C" int orgym_invmgmt_create(const orgym_invmgmt_config_t* cfg, int64_t num_envs, int device,
                                    orgym_handle_t* out) {
    ORGYM_REQUIRE(cfg && out, "null argument");
    const int m = cfg->num_stages, n = m - 1;
    // the reference's input validation (inventory_management.py:144-167)
    ORGYM_REQUIRE(m >= 2, "Minimum number of stages is 2");
    ORGYM_REQUIRE(cfg->periods > 0, "Number of periods must be positive");
    ORGYM_REQUIRE(cfg->alpha > 0 && cfg->alpha <= 1, "alpha must be in the range (0, 1]");
    ORGYM_REQUIRE(cfg->init_inv && cfg->capacity && cfg->lead_time && cfg->unit_price && cfg->unit_cost &&
                      cfg->demand_cost && cfg->holding_cost,
                  "null config array");
    if (n > MAXN) {
        orgym_set_error("%d inventory stages exceed this build's limit of %d", n, MAXN);
        return ORGYM_E_UNSUPPORTED;
    }
    int rc = ORGYM_OK;
    for (int i = 0; i < n && rc == ORGYM_OK; i++) {
        if (cfg->init_inv[i] < 0) { orgym_set_error("Initial inventory cannot be negative"); rc = ORGYM_E_INVALID; }
        if (cfg->capacity[i] <= 0) { orgym_set_error("Supply capacities must be positive"); rc = ORGYM_E_INVALID; }
        if (cfg->lead_time[i] < 0) { orgym_set_error("Lead times cannot be negative"); rc = ORGYM_E_INVALID; }
        if (cfg->lead_time[i] > ORGYM_INV_MAX_LEAD) {
            orgym_set_error("lead time %lld exceeds this build's limit of %d", (long long)cfg->lead_time[i], ORGYM_INV_MAX_LEAD);
            rc = ORGYM_E_UNSUPPORTED;
        }
    }
    for (int j = 0; j < m && rc == ORGYM_OK; j++) {
        if (cfg->unit_price[j] < 0 || cfg->unit_cost[j] < 0 || cfg->demand_cost[j] < 0 || cfg->holding_cost[j] < 0) {
            orgym_set_error("prices and costs cannot be negative");
            rc = ORGYM_E_INVALID;
        }
    }
    if (rc == ORGYM_OK && !(cfg->dist.kind >= 1 && cfg->dist.kind <= 5)) {
        orgym_set_error("dist must be one of 1, 2, 3, 4, 5");
        rc = ORGYM_E_INVALID;
    }
    if (rc == ORGYM_OK && cfg->dist.kind == ORGYM_DIST_USER && cfg->dist.user_D_len != cfg->periods) {
        orgym_set_error("User specified demand length != num periods");
        rc = ORGYM_E_INVALID;
    }
    if (rc == ORGYM_OK && cfg->periods > (1 << 20)) {
        orgym_set_error("periods above 2^20 are not supported");
        rc = ORGYM_E_UNSUPPORTED;
    }
    if (rc != ORGYM_OK) return rc;
    InvHandle* H = new InvHandle();
    InvDev& P = H->dev;
    inv_dev_from_config(cfg, &P);
    long long cmax = 0;
    for (int i = 0; i < n; i++) cmax = std::max({cmax, P.c[i], P.I0[i]});
    H->wide = cfg->wide_state ? 1 : 0;
    if (!H->wide && cmax > (INT32_GUARD >> 8)) H->wide = 1;  // compact int32 state cannot hold it
    rc = orgym_handle_base_init(&H->base, FAM_INVMGMT, device, num_envs);
    if (rc != ORGYM_OK) {
        delete H;
        return rc;
    }
    DeviceGuard g(device);
    H->npad = round_up(num_envs, 32);
    const std::vector<double> disc = inv_discounts(cfg->alpha, P.T);
    double* disc_dev = nullptr;
    cudaError_t ce = cudaMalloc(&disc_dev, sizeof(double) * (size_t)P.T);
    if (ce == cudaSuccess) {
        H->allocs.push_back(disc_dev);
        ce = cudaMemcpy(disc_dev, disc.data(), sizeof(double) * (size_t)P.T, cudaMemcpyHostToDevice);
    }
    P.disc = disc_dev;
    H->disc_host = disc;
    H->max_blocks = (int)((num_envs + ROLL_THREADS - 1) / ROLL_THREADS);
    H->hint_state = nullptr;
    H->hint_t = -1;
    H->user_dmax = 0;
    if (cfg->dist.kind == ORGYM_DIST_USER)
        for (int t = 0; t < cfg->dist.user_D_len; t++) H->user_dmax = std::max<long long>(H->user_dmax, std::llabs(cfg->dist.user_D[t]));
    H->partials = nullptr;
    if (ce == cudaSuccess) {
        size_t pbytes = sizeof(double) * (8 * (size_t)H->max_blocks + ORGYM_REDUCE_EXTRA);
        ce = cudaMalloc(&H->partials, pbytes);
        if (ce == cudaSuccess) {
            H->allocs.push_back(H->partials);
            ce = cudaMemset(H->partials, 0, pbytes);  // also zeroes the reduction ticket
        }
    }
    if (ce != cudaSuccess) {
        orgym_set_error("device allocation failed: %s", cudaGetErrorString(ce));
        rc = ORGYM_E_CUDA;
    }
    if (rc == ORGYM_OK) rc = orgym_build_alias(&cfg->dist, 0, &P.dem, &H->allocs);
    if (rc != ORGYM_OK) {
        for (void* p : H->allocs) cudaFree(p);
        orgym_handle_base_free(&H->base);
        delete H;
        return rc;
    }
    *out = (orgym_handle_t)H;
    return ORGYM_OK;
}

extern "C" int orgym_invmgmt_destroy(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return ORGYM_E_INVALID;
    InvHandle* H = (InvHandle*)h;
    {
        DeviceGuard g(H->base.device);
        for (void* p : H->allocs) cudaFree(p);
        for (auto& v : H->jit_variants)
            if (v.k.lib) orgym_jit_release(&v.k);
    }
    orgym_handle_base_free(&H->base);
    delete H;
    return ORGYM_OK;
}

extern "C" int64_t orgym_invmgmt_state_bytes(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return -1;
    InvHandle* H = (InvHandle*)h;
    return inv_state_bytes(H->dev, H->npad, H->wide);
}
extern "C" int32_t orgym_invmgmt_obs_dim(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return -1;
    return ((InvHandle*)h)->dev.obs_dim;
}
extern "C" int32_t orgym_invmgmt_act_dim(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return -1;
    return ((InvHandle*)h)->dev.n;
}

extern "C" int orgym_invmgmt_reset(orgym_handle_t h, void* state_dev, int reseed, uint64_t seed, int64_t env_offset,
                                   const uint8_t* mask_dev, int64_t* obs_dev, void* stream) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return ORGYM_E_INVALID;
    InvHandle* H = (InvHandle*)h;
    ORGYM_REQUIRE(state_dev && obs_dev, "state_dev and obs_dev are required");
    DeviceGuard g(H->base.device);
    int64_t N = H->base.num_envs;
    unsigned grid = (unsigned)((N + 255) / 256);
    if (H->wide)
        inv_reset_kernel<long long><<<grid, 256, 0, (cudaStream_t)stream>>>(H->dev, N, H->npad, state_dev, reseed, seed,
                                                                           env_offset, mask_dev, obs_dev);
    else
        inv_reset_kernel<int><<<grid, 256, 0, (cudaStream_t)stream>>>(H->dev, N, H->npad, state_dev, reseed, seed,
                                                                     env_offset, mask_dev, obs_dev);
    ORGYM_CUDA(cudaGetLastError());
    H->hint_state = state_dev;
    H->hint_t = mask_dev ? -1 : 0;
    return ORGYM_OK;
}

extern "C" int orgym_invmgmt_step(orgym_handle_t h, void* state_dev, const void* actions_dev, int action_is_f64,
                                  const int64_t* demand_override_dev, int autoreset_mode, int64_t* obs_dev,
                                  double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                                  const orgym_invmgmt_info_t* info, void* stream) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return ORGYM_E_INVALID;
    InvHandle* H = (InvHandle*)h;
    ORGYM_REQUIRE(state_dev && actions_dev && obs_dev && reward_dev && terminated_dev && truncated_dev,
                  "state, actions, obs, reward, terminated and truncated pointers are required");
    ORGYM_REQUIRE(autoreset_mode >= 0 && autoreset_mode <= 2, "bad autoreset mode");
    DeviceGuard g(H->base.device);
    const InvDev& P = H->dev;
    InvStepArgs A;
    memset(&A, 0, sizeof(A));
    A.N = H->base.num_envs;
    A.npad = H->npad;
    A.state = state_dev;
    A.actions = actions_dev;
    A.act_f64 = action_is_f64;
    A.demand = demand_override_dev;
    A.autoreset = autoreset_mode;
    A.obs = obs_dev;
    A.reward = reward_dev;
    A.terminated = terminated_dev;
    A.truncated = truncated_dev;
    if (info) {
        A.info_demand = info->demand_dev;
        A.info_sales = info->sales_dev;
        A.info_unf = info->unfulfilled_dev;
        A.info_profit = info->profit_dev;
        ORGYM_REQUIRE(info->info_ld == 0 || info->info_ld >= H->base.num_envs, "info_ld must be 0 (row-major) or >= num_envs");
        A.info_ld = info->info_ld;
        A.final_obs = info->final_obs_dev;
    }
    A.err = H->base.err_dev;
    A.t_hint = (H->hint_state == state_dev) ? H->hint_t : -1;
    if (A.t_hint >= 0) {  // advance the host-side mirror of the lock-step period exactly like the kernel will
        int t = A.t_hint;
        if (t >= P.T)
            H->hint_t = autoreset_mode == ORGYM_AUTORESET_NEXT_STEP ? 0 : t;
        else
            H->hint_t = (t + 1 >= P.T && autoreset_mode == ORGYM_AUTORESET_SAME_STEP) ? 0 : t + 1;
    }
    A.use_bulk = ((uintptr_t)actions_dev % 16 == 0) && ((uintptr_t)obs_dev % 16 == 0);
    int ostride = (P.obs_dim & 1) ? P.obs_dim : P.obs_dim + 1;
    const size_t rest = (size_t)ORGYM_TILE * P.n * 8 + 16 + inv_alias_smem(P);  // action tile, mbarrier, alias table
    size_t smem = (((size_t)ORGYM_TILE * ostride * (H->wide ? 8 : 4) + 15) & ~(size_t)15) + rest;
    if (smem > INV_STAGING_SMEM_LIMIT) {  // rows too long to stage: the generic kernel writes them directly
        A.direct_obs = 1;
        smem = rest;
    }
    if (H->wide)
        launch_step<long long>(H, A, smem, (cudaStream_t)stream);
    else
        launch_step<int>(H, A, smem, (cudaStream_t)stream);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

extern "C" int orgym_invmgmt_export_state(orgym_handle_t h, const void* state_dev, int64_t* I_dev, int64_t* B_dev,
                                          int32_t* period_dev, void* stream) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return ORGYM_E_INVALID;
    InvHandle* H = (InvHandle*)h;
    ORGYM_REQUIRE(state_dev, "state_dev is required");
    DeviceGuard g(H->base.device);
    int64_t N = H->base.num_envs;
    unsigned grid = (unsigned)((N + 255) / 256);
    if (H->wide)
        inv_export_kernel<long long><<<grid, 256, 0, (cudaStream_t)stream>>>(H->dev, N, H->npad, state_dev, I_dev, B_dev,
                                                                            period_dev);
    else
        inv_export_kernel<int><<<grid, 256, 0, (cudaStream_t)stream>>>(H->dev, N, H->npad, state_dev, I_dev, B_dev,
                                                                      period_dev);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

// ---- rigorous value bounds of an episode driven by an on-device policy (requests within [0, c_i]) -------------------
// The reference's dynamics let on-hand inventory of the upstream stages go negative (a stage subtracts its own inbound
// order, :300), and a negative supplier inventory makes fulfilled orders negative (:265).  Telescoping the pipeline gives
//   I_i(t) = I0_i - sum of the <= min(L_i, T) orders of stage i still in transit          (i >= 1)
// so with  Rhi_i = c_i,  Rlo_i = min(0, Ilo_{i+1})  (Rlo_{n-1} = 0: no supplier constraint):
//   Ilo_i = I0_i - min(L_i,T) * Rhi_i,   Ihi_i = I0_i - min(L_i,T) * Rlo_i,   and for the retailer 0 <= I_0 <= I0_0 + T * c_0.
// The retailer's lower bound holds whatever it receives (a negative fulfilled order included): it sells min(on-hand,
// fill), so it keeps max(on-hand - fill, 0).  Backlogs grow by at most (request - fulfilled) <= c_i - Rlo_i per period.
// *xvar bounds every state value, order, sale and unfulfilled quantity of any period; *xsum bounds the per-episode
// statistics (sums over periods and stages).
struct InvTermBounds {  // per stage j = 0..n: |units sold|, on-hand inventory above zero, unfulfilled quantity
    double sale[MAXN + 1], inv[MAXN + 1], unf[MAXN + 1];
    bool nonneg[MAXN];  // sign fact: Ilo_j >= 0, stage j's on-hand inventory is never negative after a period
};
static void inv_value_bounds(const InvDev& P, double dmax, double* xvar, double* xsum, InvTermBounds* tb = nullptr) {
    const int n = P.n, T = P.T;
    double Ilo[MAXN + 1], Ihi[MAXN + 1], Rlo[MAXN + 1];
    double x = dmax;
    if (tb) memset(tb, 0, sizeof(*tb));
    for (int i = n - 1; i >= 0; i--) {
        Rlo[i] = (i == n - 1) ? 0.0 : std::min(0.0, Ilo[i + 1]);
        const double Lp = (double)std::min(P.L[i], T);
        if (i >= 1) {
            Ilo[i] = (double)P.I0[i] - Lp * (double)P.c[i];
            Ihi[i] = (double)P.I0[i] - Lp * Rlo[i];
        } else {
            Ilo[i] = 0.0;
            Ihi[i] = (double)P.I0[i] + (double)T * (double)P.c[i];
        }
        const double grow = (double)P.c[i] - Rlo[i];                   // request - fulfilled, per period
        const double Bmax = P.backlog ? (double)T * grow : 0.0;        // B[i+1]
        const double Umax = (double)P.c[i] + Bmax - Rlo[i];            // cur_i - r_i
        x = std::max({x, std::fabs(Ilo[i]), std::fabs(Ihi[i]), std::fabs(Rlo[i]), (double)P.c[i], Bmax, Umax});
        if (tb) {
            tb->sale[i + 1] = std::max((double)P.c[i], std::fabs(Rlo[i]));  // fulfilled order r_i in [Rlo_i, c_i]
            tb->unf[i + 1] = Umax;
            tb->inv[i] = std::max(0.0, Ihi[i]);
            tb->nonneg[i] = Ilo[i] >= 0.0;
        }
    }
    const double B0 = P.backlog ? (double)T * (dmax - Rlo[0]) : 0.0;   // retail backlog
    x = std::max({x, B0, dmax + B0 - Rlo[0]});                         // fill, U_0, s0
    if (tb) tb->sale[0] = tb->unf[0] = dmax + B0 - Rlo[0];
    *xvar = x;
    *xsum = x * (double)T * (double)std::max(n, 1);
}

// ---- run-time specialised rollout (invmgmt_jit.cu) ------------------------------------------------------------------
static void inv_jit_spec(const InvDev& P, const std::vector<double>& disc, int policy, const long long* target,
                         InvJitSpec* S) {
    {
        double xv = 0.0, xs = 0.0;
        InvTermBounds tb;
        inv_value_bounds(P, (double)P.dem.base + (double)(1LL << P.dem.log2k), &xv, &xs, &tb);
        S->xbound = xv < 9.0e15 ? (long long)xv + 1 : 0;
        for (int j = 0; j <= P.n; j++) {
            S->sale_bound[j] = tb.sale[j];
            S->inv_bound[j] = tb.inv[j];
            S->unf_bound[j] = tb.unf[j];
        }
        for (int i = 0; i < P.n; i++) S->inv_nonneg[i] = tb.nonneg[i];
    }
    S->n = P.n;
    S->T = P.T;
    S->backlog = P.backlog;
    for (int i = 0; i < P.n; i++) {
        S->L[i] = P.L[i];
        S->c[i] = P.c[i];
        S->I0[i] = P.I0[i];
        S->target[i] = target ? target[i] : 0;
    }
    for (int j = 0; j <= P.n; j++) {
        S->up[j] = P.up[j];
        S->uc[j] = P.uc[j];
        S->kc[j] = P.kc[j];
        S->hc[j] = P.hc[j];
    }
    S->disc = disc;
    S->log2k = P.dem.log2k;
    S->base = P.dem.base;
    S->policy = policy;
}

// The specialiser's range: ORGYM_E_UNSUPPORTED, with the reason, for a user-trace demand (checked alone when S is null)
// and for a kernel spec outside inv_jit_eligible.
static int inv_jit_check(const InvDev& P, const InvJitSpec* S) {
    if (P.dem.kind == ORGYM_DIST_USER) {
        orgym_set_error("user-trace demand runs the ahead-of-time kernel");
        return ORGYM_E_UNSUPPORTED;
    }
    if (S && !inv_jit_eligible(*S)) {
        orgym_set_error("configuration outside the specialiser's range (1..6 stages, <= 64 periods, sum of lead times <= 40)");
        return ORGYM_E_UNSUPPORTED;
    }
    return ORGYM_OK;
}

// base-stock levels (lead_times + 1) * mu * sf (benchmark_InvManagementBacklogEnv.py:186); *all_int = they are integers
static void inv_base_stock_targets(const InvDev& P, const double* param, double* target, long long* target_int, int* all_int) {
    *all_int = 1;
    for (int i = 0; i < P.n; i++) {
        target[i] = ((double)(P.L[i] + 1) * param[1]) * param[0];
        if (!(target[i] == std::floor(target[i]) && std::fabs(target[i]) < 1073741824.0)) *all_int = 0;
    }
    for (int i = 0; i < P.n; i++) target_int[i] = *all_int ? (long long)target[i] : 0;
}

// ORGYM_INV_JIT: 0 = ahead-of-time kernels only, 1 (default) = specialise, fall back silently, 2 = specialise and fail
// loudly when an eligible rollout cannot get its specialised kernel
static int inv_jit_mode() {
    const char* v = getenv("ORGYM_INV_JIT");
    if (!v) return 1;
    return v[0] == '0' ? 0 : (v[0] == '2' ? 2 : 1);
}

// debugging / test aid (no GPU needed): the CUDA source generated for a config; compile_check != 0 also runs it through
// NVRTC.  Returns ORGYM_E_UNSUPPORTED (with the reason) for configurations the generator does not cover.
extern "C" int orgym_invmgmt_codegen(const orgym_invmgmt_config_t* cfg, const orgym_invmgmt_rollout_in_t* in,
                                     int compile_check, char* buf, int64_t buflen, int64_t* needed) {
    ORGYM_REQUIRE(cfg && cfg->init_inv && cfg->capacity && cfg->lead_time && cfg->unit_price && cfg->unit_cost &&
                      cfg->demand_cost && cfg->holding_cost,
                  "null argument");
    const int n = cfg->num_stages - 1;
    ORGYM_REQUIRE(n >= 1 && n <= MAXN && cfg->periods > 0, "bad stage count / horizon");
    InvDev Pb;
    inv_dev_from_config(cfg, &Pb);
    Pb.dem.kind = cfg->dist.kind;
    if (int rc = inv_jit_check(Pb, nullptr)) return rc;  // a user trace has no demand table to specialise on
    int64_t base = 0;
    if (int rc = inv_demand_table(&cfg->dist, &Pb.dem.log2k, &base)) return rc;
    Pb.dem.base = (int32_t)base;
    // policy to bake in: the caller's, or the benchmark's default base-stock (levels (L+1) * p0, SF = 1)
    int policy = 0;
    double param[4] = {1.0, cfg->dist.p0, 0.0, 0.0};
    if (in && in->policy == ORGYM_POLICY_MLP) {
        orgym_set_error("the MLP policy runs the ahead-of-time kernel (inv_mlp_rollout_kernel); it is not specialised");
        return ORGYM_E_UNSUPPORTED;
    }
    if (in) {
        ORGYM_REQUIRE(in->policy == ORGYM_POLICY_BASE_STOCK || in->policy == ORGYM_POLICY_RANDOM,
                      "only the on-device base-stock and random policies are specialised");
        policy = in->policy == ORGYM_POLICY_BASE_STOCK ? 0 : 1;
        for (int k = 0; k < 4; k++) param[k] = in->param[k];
    }
    double target[MAXN];
    long long target_int[MAXN];
    int all_int = 1;
    if (policy == 0) inv_base_stock_targets(Pb, param, target, target_int, &all_int);
    if (!all_int) {
        orgym_set_error("base-stock levels are not integers: the ahead-of-time kernel evaluates them in float64");
        return ORGYM_E_UNSUPPORTED;
    }
    InvJitSpec S;
    inv_jit_spec(Pb, inv_discounts(cfg->alpha, Pb.T), policy, target_int, &S);
    if (int rc = inv_jit_check(Pb, &S)) return rc;
    std::string src = inv_jit_source(S);
    if (needed) *needed = (int64_t)src.size();
    if (buf && buflen > 0) {
        size_t k = src.size() < (size_t)buflen - 1 ? src.size() : (size_t)buflen - 1;
        memcpy(buf, src.data(), k);
        buf[k] = 0;
    }
    if (compile_check) {
        std::string err;
        if (orgym_jit_compile_only(src, &err) != 0) {
            orgym_set_error("%s", err.substr(0, 900).c_str());
            return ORGYM_E_UNSUPPORTED;
        }
    }
    return ORGYM_OK;
}

// diagnostic (no GPU needed): the rigorous bounds inv_value_bounds derives for a configuration driven by an on-device
// policy -- *xvar bounds every state value / order / sale of any period, *xsum the per-episode statistics.  They decide
// between int32 and int64 rollouts and feed the specialiser's exactness proof; the CPU suite checks them against
// brute-force simulation with the oracle.
extern "C" int orgym_invmgmt_value_bounds(const orgym_invmgmt_config_t* cfg, double* xvar, double* xsum,
                                          double* profit_mag) {
    ORGYM_REQUIRE(cfg && xvar && xsum && cfg->init_inv && cfg->capacity && cfg->lead_time, "null argument");
    const int n = cfg->num_stages - 1;
    ORGYM_REQUIRE(n >= 1 && n <= MAXN && cfg->periods > 0, "bad stage count / horizon");
    InvDev Pb;
    inv_dev_from_config(cfg, &Pb);
    double dmax = 0.0;
    if (cfg->dist.kind == ORGYM_DIST_USER) {
        for (int t = 0; t < cfg->dist.user_D_len; t++) dmax = std::max(dmax, std::fabs((double)cfg->dist.user_D[t]));
    } else {
        int log2k = 0;
        int64_t base = 0;
        if (int rc = inv_demand_table(&cfg->dist, &log2k, &base)) return rc;
        dmax = (double)base + (double)(1LL << log2k);
    }
    InvTermBounds tb;
    inv_value_bounds(Pb, dmax, xvar, xsum, &tb);
    if (profit_mag) {  // bound on the sum of |terms| of one period's profit (the specialiser's exactness proof)
        ORGYM_REQUIRE(cfg->unit_price && cfg->unit_cost && cfg->demand_cost && cfg->holding_cost, "null argument");
        double mag = 0.0;
        for (int j = 0; j <= n; j++) mag += (Pb.up[j] + Pb.uc[j]) * tb.sale[j] + Pb.hc[j] * tb.inv[j] + Pb.kc[j] * tb.unf[j];
        *profit_mag = mag;
    }
    return ORGYM_OK;
}

// 1 when the most recent rollout ran a specialised kernel (or orgym_invmgmt_specialise just built one)
extern "C" int orgym_invmgmt_is_specialised(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return ORGYM_E_INVALID;
    return ((InvHandle*)h)->last_rollout_jit ? 1 : 0;
}

// The specialised kernel for (policy, levels): looked up in the handle's small cache, else generated and compiled.
// Returns ORGYM_OK with *fn set; ORGYM_E_UNSUPPORTED when the configuration / policy is outside the specialiser's range
// and ORGYM_E_CUDA when NVRTC failed -- both with the reason (NVRTC log included) in orgym_last_error().
static int inv_jit_get(InvHandle* H, int policy, const long long* target_int, cudaKernel_t* fn) {
    const InvDev& P = H->dev;
    for (auto& v : H->jit_variants) {
        if (v.policy != policy) continue;
        bool same = true;
        if (policy == 0)
            for (int i = 0; i < P.n; i++) same = same && v.target[i] == target_int[i];
        if (!same) continue;
        if (v.failed) {
            orgym_set_error("%s", v.err.c_str());
            return ORGYM_E_CUDA;
        }
        *fn = v.k.fn;
        return ORGYM_OK;
    }
    InvJitSpec S;
    inv_jit_spec(P, H->disc_host, policy, target_int, &S);
    if (int rc = inv_jit_check(P, &S)) return rc;
    if (H->jit_variants.size() >= 16) {  // bounded: drop the oldest variant (e.g. a sweep over safety factors)
        if (H->jit_variants.front().k.lib) orgym_jit_release(&H->jit_variants.front().k);
        H->jit_variants.erase(H->jit_variants.begin());
    }
    InvHandle::JitVariant v;
    v.policy = policy;
    for (int i = 0; i < MAXN; i++) v.target[i] = (policy == 0 && i < P.n) ? target_int[i] : 0;
    v.failed = 0;
    std::string err;
    if (orgym_jit_compile(inv_jit_source(S), inv_jit_kernel_name(policy), &v.k, &err) != 0) {
        v.failed = 1;
        v.err = "specialising the rollout kernel failed: " + err.substr(0, 800);
        H->jit_variants.push_back(v);
        orgym_set_error("%s", v.err.c_str());
        return ORGYM_E_CUDA;
    }
    H->jit_variants.push_back(v);
    *fn = v.k.fn;
    return ORGYM_OK;
}

// true when this request can run a specialised kernel at all (policy, outputs, arithmetic width)
static bool inv_jit_policy_ok(const orgym_invmgmt_rollout_in_t* in, int target_is_int) {
    return (in->policy == ORGYM_POLICY_BASE_STOCK && target_is_int) || in->policy == ORGYM_POLICY_RANDOM;
}

extern "C" int orgym_invmgmt_specialise(orgym_handle_t h, const orgym_invmgmt_rollout_in_t* in) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return ORGYM_E_INVALID;
    InvHandle* H = (InvHandle*)h;
    ORGYM_REQUIRE(in, "null argument");
    DeviceGuard g(H->base.device);
    const InvDev& P = H->dev;
    double target[MAXN];
    long long target_int[MAXN];
    int all_int = 1;
    if (in->policy == ORGYM_POLICY_BASE_STOCK) inv_base_stock_targets(P, in->param, target, target_int, &all_int);
    if (!inv_jit_policy_ok(in, all_int)) {
        orgym_set_error("only the on-device base-stock policy with integer levels and the random policy are specialised");
        return ORGYM_E_UNSUPPORTED;
    }
    if (H->wide) {
        orgym_set_error("wide_state handles run the ahead-of-time int64 kernel");
        return ORGYM_E_UNSUPPORTED;
    }
    cudaKernel_t fn = nullptr;
    int rc = inv_jit_get(H, in->policy == ORGYM_POLICY_BASE_STOCK ? 0 : 1, target_int, &fn);
    H->last_rollout_jit = rc == ORGYM_OK;
    return rc;
}

// bytes of caller-owned device scratch orgym_invmgmt_rollout needs through in->scratch_dev: 0 unless the lead-time rings
// of the ahead-of-time kernel cannot live in shared memory (worst case: int64 arithmetic, both rings)
extern "C" int64_t orgym_invmgmt_rollout_scratch_bytes(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return -1;
    InvHandle* H = (InvHandle*)h;
    const InvDev& P = H->dev;
    int64_t rslots = 0;
    for (int i = 0; i < P.n; i++) rslots += P.L[i] > 0 ? P.L[i] : 1;
    if (inv_alias_smem(P) + (size_t)rslots * ROLL_THREADS * 8 * 2 <= INV_STAGING_SMEM_LIMIT) return 0;
    return rslots * round_up(H->base.num_envs, ROLL_THREADS) * 8 * 2;
}

extern "C" int orgym_invmgmt_rollout(orgym_handle_t h, uint64_t seed, int64_t env_offset, uint32_t episode,
                                     const orgym_invmgmt_rollout_in_t* in, const orgym_invmgmt_rollout_out_t* out,
                                     void* stream) {
    if (orgym_check_handle(h, FAM_INVMGMT)) return ORGYM_E_INVALID;
    InvHandle* H = (InvHandle*)h;
    ORGYM_REQUIRE(in && out, "null argument");
    ORGYM_REQUIRE(in->policy >= 0 && in->policy <= ORGYM_POLICY_MLP, "unknown policy %d", in->policy);
    ORGYM_REQUIRE(in->policy != ORGYM_POLICY_ACTIONS || in->actions_dev, "policy ACTIONS needs actions_dev");
    if (in->policy == ORGYM_POLICY_RANDOM)
        for (int i = 0; i < ((InvHandle*)h)->dev.n; i++)
            ORGYM_REQUIRE(((InvHandle*)h)->dev.c[i] < 0x7fffffffLL, "random policy needs capacities below 2^31");
    DeviceGuard g(H->base.device);
    const InvDev& P = H->dev;
    InvRolloutArgs A;
    memset(&A, 0, sizeof(A));
    A.N = H->base.num_envs;
    A.env_offset = env_offset;
    A.seed = seed;
    A.episode = episode;
    A.policy = in->policy;
    if (in->policy == ORGYM_POLICY_BASE_STOCK)  // (lead_times + 1) * mu * sf (:186)
        inv_base_stock_targets(P, in->param, A.target, A.target_int, &A.target_is_int);
    for (int i = 0; i < P.n; i++) {
        A.rroff[i] = A.rslots;
        A.rslots += P.L[i] > 0 ? P.L[i] : 1;
    }
    A.actions = in->actions_dev;
    A.a_se = in->act_stride_env;
    A.a_st = in->act_stride_t;
    A.demand = in->demand_dev;
    A.d_se = in->dem_stride_env;
    A.d_st = in->dem_stride_t;
    A.ep_return = out->ep_return_dev;
    A.stats = out->stats_dev;
    A.reward_traj = out->reward_traj_dev;
    A.final_I = out->final_I_dev;
    A.final_B = out->final_B_dev;
    A.stats32 = out->stats32_dev;
    A.action_traj = out->action_traj_dev;
    A.partials = out->summary_dev ? H->partials : nullptr;
    // int32 arithmetic only when inv_value_bounds proves every state value below 2^30 and every per-episode sum below
    // 2^31: on-device policy (requests within [0, c]) and bounded demand -- the sampler's support, or a trace whose
    // values were copied to the device at create and are bounded by their config-time maximum.  Pre-staged actions /
    // replayed demand may be arbitrary int64 -> exact wide arithmetic
    const long long dmax = P.dem.kind != ORGYM_DIST_USER ? (long long)P.dem.base + (1LL << P.dem.log2k)
                           : in->demand_dev          ? (1LL << 40)
                                                     : H->user_dmax;
    double xvar = 0.0, xsum = 0.0;
    inv_value_bounds(P, (double)dmax, &xvar, &xsum);
    const bool bounded = xvar < 1073741824.0 && xsum < 2147483648.0;
    const bool wide = H->wide || in->policy == ORGYM_POLICY_ACTIONS || in->demand_dev != nullptr || !bounded;
    // fast path: kernels specialised for this configuration (register-resident rings, straight-line periods); the MLP
    // policy and the outputs they do not produce run the ahead-of-time kernels
    H->last_rollout_jit = 0;
    const int jit_mode = inv_jit_mode();
    cudaKernel_t jit_fn = nullptr;
    if (jit_mode && !wide && inv_jit_policy_ok(in, A.target_is_int) && !A.reward_traj && !A.final_I && !A.final_B &&
        !A.action_traj) {
        const int jrc = inv_jit_get(H, in->policy == ORGYM_POLICY_BASE_STOCK ? 0 : 1, A.target_int, &jit_fn);
        if (jrc != ORGYM_OK && jit_mode == 2) return jrc;  // strict: the reason is in orgym_last_error()
    }
    // every kernel writes one partial-sum row per ROLL_THREADS envs, so one reduction serves all three
    static_assert(INV_JIT_THREADS == ROLL_THREADS, "the specialised kernel's CTAs must match the partial-sum rows");
    if (jit_fn) {
        InvJitArgs J;
        memset(&J, 0, sizeof(J));
        J.N = A.N;
        J.env_offset = A.env_offset;
        J.seed = A.seed;
        J.episode = A.episode;
        for (int i = 0; i < P.n; i++) J.target[i] = (int32_t)A.target_int[i];
        J.table = P.dem.table;
        J.ep_return = A.ep_return;
        J.stats = A.stats;
        J.stats32 = A.stats32;
        J.partials = A.partials;
        void* args[] = {(void*)&J};
        const unsigned grid = (unsigned)((A.N + INV_JIT_THREADS - 1) / INV_JIT_THREADS);
        cudaError_t le = cudaLaunchKernel((const void*)jit_fn, dim3(grid), dim3(INV_JIT_THREADS), args, 0, (cudaStream_t)stream);
        if (le != cudaSuccess) {
            orgym_set_error("specialised rollout kernel launch failed: %s", cudaGetErrorString(le));
            return ORGYM_E_CUDA;
        }
        H->last_rollout_jit = 1;
    } else if (in->policy == ORGYM_POLICY_MLP) {
        InvMlpPlan M;
        size_t smem = 0;
        if (int rc = inv_mlp_plan(P, in->mlp, A.rslots, wide ? 8 : 4, &M, &smem)) return rc;
        if (wide)
            launch_mlp_rollout<long long>(H, A, M, smem, (cudaStream_t)stream);
        else
            launch_mlp_rollout<int>(H, A, M, smem, (cudaStream_t)stream);
        ORGYM_CUDA(cudaGetLastError());
    } else {
        const size_t ring = (size_t)A.rslots * ROLL_THREADS * (wide ? 8 : 4);
        size_t smem = inv_alias_smem(P) + ring * (in->policy == ORGYM_POLICY_BASE_STOCK ? 2 : 1);
        if (smem > INV_STAGING_SMEM_LIMIT) {  // rings too long for shared memory: caller-owned global scratch, generic kernel
            if (!in->scratch_dev) {
                orgym_set_error("lead-time rings (sum of lead times = %d) do not fit in shared memory: pass a scratch_dev buffer "
                                "of orgym_invmgmt_rollout_scratch_bytes() = %lld bytes", P.sumL,
                                (long long)orgym_invmgmt_rollout_scratch_bytes(h));
                return ORGYM_E_INVALID;
            }
            A.ring_scratch = in->scratch_dev;
            A.ring_stride = round_up(A.N, ROLL_THREADS);
            smem = inv_alias_smem(P);
        }
        if (wide)
            launch_rollout<long long>(H, A, smem, (cudaStream_t)stream);
        else
            launch_rollout<int>(H, A, smem, (cudaStream_t)stream);
        ORGYM_CUDA(cudaGetLastError());
    }
    if (out->summary_dev) {
        int rr = orgym_launch_reduce(H->partials, (int)((A.N + ROLL_THREADS - 1) / ROLL_THREADS), out->summary_dev,
                                     (cudaStream_t)stream);
        if (rr != ORGYM_OK) return rr;
    }
    return ORGYM_OK;
}
