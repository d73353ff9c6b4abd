// netinv.cu -- graph-structured network inventory env (reference: network_management.py).
//
// One env instance per thread.  The topology (flattened from networkx on the host: sorted reorder links,
// per-node predecessor / successor lists in adjacency order) travels as a __grid_constant__ kernel parameter,
// i.e. it lives in the constant bank; every loop over links / nodes is uniform across the warp, so the
// sequential per-supplier allocation of the reference runs divergence-free with one instance per lane.
// Per-instance float64 work vectors (X, consumed, R_t, Y, U, S_retail) sit in shared memory as [slot][thread]
// (conflict-free); the lead-time rings (last L_e fulfilled orders per link) stay in HBM as ring[slot][env] and are
// touched twice per link per period.
//
//   net_reset_kernel   reset (network_management.py:301-332) + first observation (:334-413)
//   net_sim_kernel     STEP mode: one period (:436-635) + observation;  ROLLOUT mode: fused reset + T periods
//   net_mlp_rollout_kernel  the fused rollout with an MLP actor evaluated on the device every period
//
// float64 throughout, evaluated in the reference's operation order (Python sum order = adjacency order).
#include "launch_util.cuh"
#include "mlp.cuh"
#include "netinv.cuh"

// t % d for 0 <= t < 2^20, 1 <= d <= 64 (exact, see invmgmt.cu)
__device__ __forceinline__ int net_mod(int t, int d, uint32_t magic) {
    return magic ? t - (int)__umulhi((uint32_t)t, magic) * d : 0;
}

// observation (:334-413): [U (M), X (J), per link with L>0: R[t-L..t-1] zero-padded on the left] as float32.
// ring slot s of a link holds the order of the latest period p with p % L == s (0 before any), so the window
// element q (oldest first) of the observation at period t is ring[(t + q) % L].  Ring loads are issued in batches
// of 8 before they are converted and stored, so that their latencies overlap.
template <int NTHR>
__device__ __forceinline__ void net_write_obs(const NetDev& P, const double* sU, const double* sX, int tid,
                                              const double* ring, int el, int t, float* o) {
    int k = 0;
    for (int r = 0; r < P.M; r++) o[k++] = (float)sU[r * NTHR + tid];
    for (int j = 0; j < P.J; j++) o[k++] = (float)sX[j * NTHR + tid];
    for (int i = 0; i < P.E; i++) {
        const int L = P.L[i];
        if (L == 0) continue;  // :353
        int s = net_mod(t, L, P.Lmagic[i]);
        const double* base = ring + (size_t)P.roff[i] * NET_TILE + el;
        for (int q0 = 0; q0 < L; q0 += 8) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                int sl = s + q0 + u;
                sl = sl >= L ? sl - L : sl;
                v[u] = (q0 + u < L) ? base[(size_t)sl * NET_TILE] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (q0 + u < L) o[k + q0 + u] = (float)v[u];
        }
        k += L;
    }
}

__global__ void __launch_bounds__(128) net_reset_kernel(const __grid_constant__ NetDev P, int64_t N, void* state,
                                                        int reseed, uint64_t seed, int64_t env_offset,
                                                        const uint8_t* __restrict__ mask, float* __restrict__ obs) {
    const int64_t e0 = (int64_t)blockIdx.x * 128, e = e0 + threadIdx.x;
    if (e < N && (!mask || mask[e])) {
        NetState st((char*)state + (e / NET_TILE) * net_tile_bytes(P), P);
        const int el = (int)(e % NET_TILE);
        for (int j = 0; j < P.J; j++) st.X[j * NET_TILE + el] = P.I0[j];  // :326
        for (int i = 0; i < P.E; i++) st.Y[i * NET_TILE + el] = 0.0;
        for (int r = 0; r < P.M; r++) st.U[r * NET_TILE + el] = 0.0;
        for (int k = 0; k < P.sumL; k++) st.ring[k * NET_TILE + el] = 0.0;
        if (P.ring32)
            for (int k = 0; k < P.sumL; k++) st.ring32[k * NET_TILE + el] = 0.0f;
        st.period[el] = 0;
        if (reseed) {
            st.key[el] = seed + (uint64_t)(env_offset + e);
            st.episode[el] = 0;
        } else
            st.episode[el] += 1;
    }
    // first observation [0 (M), I0 (J), 0 ...] written cooperatively: coalesced stores over the CTA's 128 rows
    const int W = P.obs_dim;
    const int nrows = (int)((N - e0) < 128 ? (N - e0) : 128);
    int r = 0, c = threadIdx.x;
    while (c >= W) { c -= W; r++; }
    for (int i = threadIdx.x; i < nrows * W; i += 128) {
        if (!mask || mask[e0 + r]) obs[e0 * W + i] = (c >= P.M && c < P.M + P.J) ? (float)P.I0[c - P.M] : 0.0f;
        c += 128;
        while (c >= W) { c -= W; r++; }
    }
}

#include "netinv_args.cuh"

// One period (:436-635) of one instance, the body shared by net_sim_kernel and net_mlp_rollout_kernel.  The work vectors
// sX, sC, sR, sY, sU, sS are shared-memory rows of stride NTHR ([slot][NTHR], this instance's column is tid); the
// lead-time rings live in ring[slot][NET_TILE] at column el and are written only when `valid`.
//   arow()        the float32 actions of the period (before the env's rint / max(0, .) rule): link i at arow()[i * ASTRIDE]
//   demand(r)     demand of retail link r before max(0, .): a replayed value (already rounded) or a draw
//   on_demand(r, d), on_profit(j, pj)   per-market demand and per-node profit, for the STEP info tensors
// Accumulates the episode statistics and returns the undiscounted profit of the period, in Python sum order.
template <int NTHR, int ASTRIDE, class Arow, class Demand, class OnDemand, class OnProfit>
__device__ __forceinline__ double net_period(const NetDev& P, int tid, int el, double* ring, bool valid, int t,
                                             double* sX, double* sC, double* sR, double* sY, double* sU, double* sS,
                                             Arow arow_of, Demand demand, OnDemand on_demand, OnProfit on_profit,
                                             double& s_sales, double& s_dem, double& s_unf, double& s_inv) {
    const int J = P.J, E = P.E, M = P.M;
    constexpr int np_ = NET_TILE;
    // ---- 0) place orders: sequential greedy allocation in sorted (supplier, purchaser) order (:448-490)
    for (int j = 0; j < J; j++) sC[j * NTHR + tid] = 0.0;
    double cons_s = 0.0;
    const float* arow = arow_of();
    for (int i = 0; i < E; i++) {
        double req = rint((double)arow[i * ASTRIDE]);  // Python round(): half to even
        req = req > 0.0 ? req : 0.0;                   // max(0, .)
        const int s = P.sup[i];
        double f = 0.0;
        if (s == -1)
            f = req;  // raw material: unlimited (:453-455)
        else if (s >= 0) {
            if (i == 0 || P.sup[i - 1] != s) cons_s = 0.0;
            double avail = sX[s * NTHR + tid] - cons_s;  // :459
            avail = avail > 0.0 ? avail : 0.0;           // :460
            double oa = avail;
            const double vs = P.v[s];
            if (P.is_factory[s]) {  // :464-478
                double mp = vs * avail;
                double lim = mp < P.C[s] ? mp : P.C[s];
                oa = lim < oa ? lim : oa;
            }
            f = oa < req ? oa : req;                 // :481
            cons_s += vs == 1.0 ? f : f / vs;        // :484-485 (x / 1.0 == x)
            if (i == E - 1 || P.sup[i + 1] != s) sC[s * NTHR + tid] = cons_s;
        }
        sR[i * NTHR + tid] = f;  // R[t] = S[t] = f (:488-490)
    }
    // ---- on-hand inventory (:516-528): arrivals R[t-L] summed in predecessor (adjacency) order
    for (int j = 0; j < J; j++) {
        double arr = 0.0;
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
            const int i = P.pred_idx[z], L = P.L[i];
            arr += L == 0 ? sR[i * NTHR + tid]
                          : ring[(P.roff[i] + net_mod(t, L, P.Lmagic[i])) * np_ + el];
        }
        sX[j * NTHR + tid] = (sX[j * NTHR + tid] + arr) - sC[j * NTHR + tid];
    }
    // ---- 1) pipeline inventory (:494-511) and ring commit: slot t % L held R[t-L] and now receives R[t]
    for (int i = 0; i < E; i++) {
        const int L = P.L[i];
        const double rt = sR[i * NTHR + tid];
        double arriving = rt;
        if (L > 0) {
            double* slot = ring + (P.roff[i] + net_mod(t, L, P.Lmagic[i])) * np_ + el;
            arriving = *slot;
            if (valid) *slot = rt;
        }
        sY[i * NTHR + tid] = (sY[i * NTHR + tid] - arriving) + rt;
    }
    // ---- 2-4) market demand, sales, backlog (:536-566)
    for (int r = 0; r < M; r++) {
        double d = demand(r);
        d = d > 0.0 ? d : 0.0;  // max(0, int(round(.))) (:540)
        const int j = P.rt_node[r];
        double fill = d + sU[r * NTHR + tid];
        double x = sX[j * NTHR + tid];
        double invr = x > 0.0 ? x : 0.0;
        double sl = invr < fill ? invr : fill;  // min(demand_to_fill, inv) (:548)
        sS[r * NTHR + tid] = sl;
        sX[j * NTHR + tid] = x - sl;
        double un = fill - sl;
        sU[r * NTHR + tid] = P.backlog ? un : 0.0;  // :560-563
        s_sales += sl;
        s_dem += d;
        s_unf += P.backlog ? un : 0.0;
        on_demand(r, d);
    }
    // ---- 5) profit per node, Python sum order (:578-613)
    double total = 0.0;
    for (int j = 0; j < J; j++) {
        double SR = 0.0, PC = 0.0, HCp = 0.0, sold = 0.0, UP = 0.0;
        for (int z = P.succ_ptr[j]; z < P.succ_ptr[j + 1]; z++) {
            const int l = P.succ_idx[z];
            double q, pr;
            if (l < E) {
                q = sR[l * NTHR + tid];
                pr = P.p[l];
            } else {
                q = sS[(l - E) * NTHR + tid];
                pr = P.rt_p[l - E];
                UP += P.rt_b[l - E] * sU[(l - E) * NTHR + tid];  // :608
            }
            SR += pr * q;  // :582
            sold += q;     // :599
        }
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
            const int i = P.pred_idx[z];
            PC += P.p[i] * sR[i * NTHR + tid];  // :586
            double y = sY[i * NTHR + tid];
            HCp += P.g[i] * (y > 0.0 ? y : 0.0);  // :591
        }
        double x = sX[j * NTHR + tid];
        double xp = x > 0.0 ? x : 0.0;
        double HC = P.h[j] * xp + HCp;  // :590-593
        double OC = 0.0;
        if (P.is_factory[j]) {  // :597-601
            const double vj = P.v[j];
            OC = vj > 0.0 ? P.o[j] * (vj == 1.0 ? sold : sold / vj) : 0.0;
        }
        if (!P.is_retail[j]) UP = 0.0;             // :605
        double pj = (((SR - PC) - OC) - HC) - UP;  // :611
        total += pj;
        s_inv += xp;
        on_profit(j, pj);
    }
    return total;
}

// 128 threads: at most 102 registers, so that 5 CTAs (the shared-memory work vectors of small graphs allow 6) stay
// resident per SM; without the bound ptxas takes 125 and the ROLLOUT mode runs 12 % slower at 4 CTAs/SM.
template <int NTHR>
__global__ void __launch_bounds__(NTHR, NTHR == 128 ? 5 : 0) net_sim_kernel(const __grid_constant__ NetDev P,
                                                       const __grid_constant__ NetSimArgs A) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int tid = threadIdx.x;
    const int64_t e0 = (int64_t)blockIdx.x * NTHR, e = e0 + tid;
    const bool valid = e < A.N;
    const int64_t ec = valid ? e : 0;  // clamp so that idle lanes stay in bounds
    const int J = P.J, E = P.E, M = P.M;
    double* sX = (double*)smem;      // [J]
    double* sC = sX + J * NTHR;      // [J] inventory consumed this period
    double* sR = sC + J * NTHR;      // [E] orders fulfilled this period
    double* sY = sR + E * NTHR;      // [E]
    double* sU = sY + E * NTHR;      // [M]
    double* sS = sU + M * NTHR;      // [M] retail sales this period
    float* otile = (float*)(sS + M * NTHR);  // STEP mode, when it fits: [NTHR][obs_stride] staging tile
    const int ostride = P.obs_dim | 1;       // odd row stride: conflict-free row writes
    NetState st((char*)A.state + (ec / NET_TILE) * net_tile_bytes(P), P);
    const int el = (int)(ec % NET_TILE);  // position inside the state tile
    double* ring = st.ring;
    constexpr int np_ = NET_TILE;

    uint64_t key;
    uint32_t episode;
    int t0, t1;
    bool do_step = valid;
    float* orow = A.use_tile ? otile + tid * ostride : (A.obs ? A.obs + ec * P.obs_dim : nullptr);
    if (A.rollout) {
        key = A.seed + (uint64_t)(A.env_offset + e);
        episode = A.episode;
        t0 = 0;
        t1 = P.T;
        for (int j = 0; j < J; j++) sX[j * NTHR + tid] = P.I0[j];
        for (int i = 0; i < E; i++) sY[i * NTHR + tid] = 0.0;
        for (int r = 0; r < M; r++) sU[r * NTHR + tid] = 0.0;
        if (valid)
            for (int k = 0; k < P.sumL; k++) ring[k * np_ + el] = 0.0;
    } else {
        key = st.key[el];
        episode = st.episode[el];
        t0 = st.period[el];
        t1 = t0 + 1;
        if (valid && t0 >= P.T) {  // episode already over
            do_step = false;
            if (A.autoreset == ORGYM_AUTORESET_NEXT_STEP) {
                for (int j = 0; j < J; j++) {
                    st.X[j * np_ + el] = P.I0[j];
                    sX[j * NTHR + tid] = P.I0[j];
                }
                for (int i = 0; i < E; i++) st.Y[i * np_ + el] = 0.0;
                for (int r = 0; r < M; r++) {
                    st.U[r * np_ + el] = 0.0;
                    sU[r * NTHR + tid] = 0.0;
                }
                for (int k = 0; k < P.sumL; k++) ring[k * np_ + el] = 0.0;
                st.period[el] = 0;
                st.episode[el] = episode + 1;
                net_write_obs<NTHR>(P, sU, sX, tid, ring, el, 0, orow);
                A.reward[e] = 0.0;
                A.terminated[e] = 0;
                A.truncated[e] = 0;
            } else {
                atomicOr(A.err, ORGYM_ERR_STEP_PAST_END);
                if (A.use_tile)
                    for (int z = 0; z < P.obs_dim; z++) orow[z] = A.obs[e * P.obs_dim + z];
                A.reward[e] = 0.0;
                A.terminated[e] = 0;
                A.truncated[e] = 1;
            }
        }
        if (do_step) {
            for (int j = 0; j < J; j++) sX[j * NTHR + tid] = st.X[j * np_ + el];
            for (int i = 0; i < E; i++) sY[i * NTHR + tid] = st.Y[i * np_ + el];
            for (int r = 0; r < M; r++) sU[r * NTHR + tid] = st.U[r * np_ + el];
        }
    }
    double ret = 0.0, s_sales = 0.0, s_dem = 0.0, s_unf = 0.0, s_inv = 0.0, last_reward = 0.0;
    if (!A.rollout && !do_step) t1 = t0;  // nothing to simulate for this lane

    for (int t = t0; t < t1; t++) {
        const double total = net_period<NTHR, 1>(
            P, tid, el, ring, valid, t, sX, sC, sR, sY, sU, sS,
            [&] {
                return A.policy == ORGYM_NET_POLICY_CONSTANT
                           ? A.actions
                           : A.actions + ec * A.a_se + (int64_t)(A.rollout ? t : 0) * A.a_st;
            },
            [&](int r) {
                return A.demand ? rint(A.demand[ec * A.d_se + (int64_t)(A.rollout ? t : 0) * A.d_st + r])
                                : (double)sample_fixed(P.dem[r], P.dem[r].table, key, episode, t, (uint32_t)r);
            },
            [&](int r, double d) {
                if (!A.rollout && A.info_demand && do_step) A.info_demand[NET_IIDX(A, e, M, r)] = d;
            },
            [&](int j, double pj) {
                if (!A.rollout && A.info_profit && do_step) A.info_profit[NET_IIDX(A, e, J, j)] = pj;
            },
            s_sales, s_dem, s_unf, s_inv);
        last_reward = P.disc[t] * total;  // :619
        ret += last_reward;
        if (A.rollout && A.reward_traj && valid) A.reward_traj[e * P.T + t] = last_reward;
        if (!A.rollout && do_step) {
            if (A.info_profit_total) A.info_profit_total[e] = total;
            if (A.info_sales) {
                for (int i = 0; i < E; i++) A.info_sales[NET_IIDX(A, e, E + M, i)] = sR[i * NTHR + tid];
                for (int r = 0; r < M; r++) A.info_sales[NET_IIDX(A, e, E + M, E + r)] = sS[r * NTHR + tid];
            }
        }
    }

    if (A.rollout) {
        if (valid) {
            if (A.ep_return) A.ep_return[e] = ret;
            if (A.stats) {
                A.stats[e * 4 + 0] = s_sales; A.stats[e * 4 + 1] = s_dem; A.stats[e * 4 + 2] = s_unf; A.stats[e * 4 + 3] = s_inv;
            }
            if (A.final_X) for (int j = 0; j < J; j++) A.final_X[e * J + j] = sX[j * NTHR + tid];
            if (A.final_Y) for (int i = 0; i < E; i++) A.final_Y[e * E + i] = sY[i * NTHR + tid];
            if (A.final_U) for (int r = 0; r < M; r++) A.final_U[e * M + r] = sU[r * NTHR + tid];
        }
        if (A.partials) {
            double v[7] = {valid ? 1.0 : 0.0, valid ? ret : 0.0, valid ? ret * ret : 0.0, valid ? s_sales : 0.0,
                           valid ? s_dem : 0.0, valid ? s_unf : 0.0, valid ? s_inv : 0.0};
            __shared__ double red[8][7];
            __syncthreads();
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
                for (int wv = 0; wv < NTHR / 32; wv++) x += red[wv][tid];
                A.partials[(size_t)blockIdx.x * 8 + tid] = x;
            }
        }
        return;
    }
    if (do_step) {
        const int tn = t0 + 1;
        const bool trunc = tn >= P.T;  // :624
        const bool reset_now = trunc && A.autoreset == ORGYM_AUTORESET_SAME_STEP;
        if (!reset_now) {
            for (int j = 0; j < J; j++) st.X[j * np_ + el] = sX[j * NTHR + tid];
            for (int i = 0; i < E; i++) st.Y[i * np_ + el] = sY[i * NTHR + tid];
            for (int r = 0; r < M; r++) st.U[r * np_ + el] = sU[r * NTHR + tid];
            st.period[el] = tn;
            net_write_obs<NTHR>(P, sU, sX, tid, ring, el, tn, orow);
        } else {
            if (A.final_obs) net_write_obs<NTHR>(P, sU, sX, tid, ring, el, tn, A.final_obs + e * P.obs_dim);
            for (int j = 0; j < J; j++) {
                st.X[j * np_ + el] = P.I0[j];
                sX[j * NTHR + tid] = P.I0[j];
            }
            for (int i = 0; i < E; i++) st.Y[i * np_ + el] = 0.0;
            for (int r = 0; r < M; r++) {
                st.U[r * np_ + el] = 0.0;
                sU[r * NTHR + tid] = 0.0;
            }
            for (int k = 0; k < P.sumL; k++) ring[k * np_ + el] = 0.0;
            st.period[el] = 0;
            st.episode[el] = episode + 1;
            net_write_obs<NTHR>(P, sU, sX, tid, ring, el, 0, orow);
        }
        A.reward[e] = last_reward;
        A.terminated[e] = 0;
        A.truncated[e] = trunc ? 1 : 0;
    }
    if (A.use_tile) {  // coalesced copy-out of the [env][obs_dim] block
        __syncthreads();
        const int nvalid = (int)((A.N - e0) < NTHR ? (A.N - e0) : NTHR);
        const int W = P.obs_dim, total = nvalid * W;
        float* g = A.obs + (size_t)e0 * W;
        int r = 0, c = tid;  // element i = tid + k*NTHR  ->  (row, col) tracked incrementally (no division)
        while (c >= W) { c -= W; r++; }
        for (int i = tid; i < total; i += NTHR) {
            __stcs(g + i, otile[r * ostride + c]);
            c += NTHR;
            while (c >= W) { c -= W; r++; }
        }
    }
}

__global__ void net_export_kernel(const __grid_constant__ NetDev P, int64_t N, const void* state,
                                  double* __restrict__ X, double* __restrict__ Y, double* __restrict__ U,
                                  int32_t* __restrict__ period) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= N) return;
    NetState st((char*)state + (e / NET_TILE) * net_tile_bytes(P), P);
    const int el = (int)(e % NET_TILE);
    if (X) for (int j = 0; j < P.J; j++) X[e * P.J + j] = st.X[j * NET_TILE + el];
    if (Y) for (int i = 0; i < P.E; i++) Y[e * P.E + i] = st.Y[i * NET_TILE + el];
    if (U) for (int r = 0; r < P.M; r++) U[e * P.M + r] = st.U[r * NET_TILE + el];
    if (period) period[e] = st.period[el];
}

// ---- observation assembly for large graphs (network_management.py:334-413) --------------------------------------------------
// The streaming STEP path for large graphs leaves the new state in HBM; this kernel turns it into row-major float32
// observation rows.  One CTA owns NET_OBS_ROWS = 32 instances (a quarter of a 128-instance state tile).  A state tile is
// slot-major ([slot][128 instances]), so the CTA's share of an observation COLUMN is 32 consecutive doubles: one
// coalesced 256-byte warp load -- 128 bytes for the window columns, which come from the tile's float32 copy of the rings
// (P.ring32).  The warps take the columns round-robin, NET_OBS_BATCH (float64) / NET_OBS_BATCH32 (float32) loads in flight
// per thread -- the kernel is bound by the round trips of a CTA, not by bytes: halving the bytes read did not move it,
// 22 instead of 12 loads per batch and 12 instead of 8 warps took it from 0.18 to 0.115 ms on the 64-node graph --,
// convert and scatter into a shared-memory image of the 32 finished rows (lane = instance; the row pitch obs_dim is odd for
// the large graphs -> conflict-free).  Those 32 rows are contiguous in the caller's [N][obs_dim] tensor, so they leave
// with ONE bulk store through the TMA engine (cp.async.bulk.global.shared::cta): full 32-byte sectors whatever the
// alignment of an individual row -- per-lane 4-byte stores of an odd-length row write every sector in two partial
// pieces.  (Two earlier forms are in the history of this file: bulk loads per column with direct stores, 0.21 ms for
// the 64-node graph, and bulk loads of 256-byte column pieces, 0.39 ms -- a bulk copy is a warp-uniform instruction, so
// per-lane copies are issued one lane at a time.)
// Which slot feeds which column depends on the period only through t mod L_i of every link (ring rotation); a group of
// instances that are not all in the same period (possible only after masked resets) takes the per-instance fallback.
#define NET_OBS_ROWS 32    // instances per CTA
#define NET_OBS_THREADS 384
#define NET_OBS_BATCH 12   // independent column loads in flight per thread
#define NET_OBS_BATCH32 22  // ... for the float32 ring columns (one register each)
static size_t net_obs_smem(const NetDev& P) {
    return 128 + (((size_t)P.obs_dim * 2 + 127) & ~(size_t)127) + (((size_t)NET_OBS_ROWS * P.obs_dim * 4 + 127) & ~(size_t)127);
}

NetPlan net_plan(const NetDev& P) {
    NetPlan plan;
    // auto: specialise graphs of up to 128 reorder links (the 64-node / 88-link synthetic graph compiles in 10-15 s,
    // once: cubins are cached on disk); ORGYM_NET_JIT=0 never, =1 always, =2 always and fail loudly
    const char* jv = getenv("ORGYM_NET_JIT");
    plan.jit = !jv ? (P.E <= 128 ? 1 : 0) : jv[0] == '0' ? 0 : jv[0] == '2' ? 2 : 1;
    // graph size selects the streaming STEP form; ORGYM_NET_JIT_STREAM=1 / 0 forces it on / off, so that small graphs
    // can test it
    const char* sv = getenv("ORGYM_NET_JIT_STREAM");
    plan.stream = sv ? (atoi(sv) ? 1 : 0) : (net_large_graph(P) ? 1 : 0);
    // Single-pass streaming form: usable when every inventory-holding supplier comes after its purchasers in node order
    // (true of the reference's graphs, which number nodes market -> raw material), so that a purchaser still finds its
    // suppliers' start-of-period inventory in the state tile.  ORGYM_NET_JIT_ONEPASS=0 forces the two-pass form, so
    // that graphs in the reference's numbering can test it.
    const char* ov = getenv("ORGYM_NET_JIT_ONEPASS");
    plan.onepass = !(ov && atoi(ov) == 0);
    for (int j = 0; j < P.J; j++)
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
            const int s = P.sup[P.pred_idx[z]];
            if (s >= 0 && s <= j) plan.onepass = 0;
        }
    // The streaming kernel stops after the state update and the TMA-staged net_obs_kernel writes the observation from
    // the float32 ring copy, unless 32 observation rows do not fit that kernel's shared memory: then the kernel's own
    // pass C writes it (ORGYM_NET_OBS_TMA=0 forces pass C, so that small graphs can test it; the ring copy stays).
    plan.ring32 = plan.stream && net_obs_smem(P) <= 200 * 1024;
    const char* tv = getenv("ORGYM_NET_OBS_TMA");
    plan.obs_kernel = plan.ring32 && !(tv && atoi(tv) == 0);
    return plan;
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__global__ void __launch_bounds__(NET_OBS_THREADS) net_obs_kernel(const __grid_constant__ NetDev P, int64_t N,
                                                                  const void* __restrict__ state, float* __restrict__ obs) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int W = P.obs_dim;
    uint16_t* colrow = (uint16_t*)(smem + 128);  // [obs_dim] 1 KB row of the tile that feeds column c
    float* out = (float*)(smem + 128 + (((size_t)W * 2 + 127) & ~(size_t)127));  // [32][obs_dim]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = NET_OBS_THREADS / 32;
    constexpr int QPT = NET_TILE / NET_OBS_ROWS;  // CTAs per state tile
    const int64_t tile_id = blockIdx.x / QPT;
    const int quarter = (int)(blockIdx.x % QPT);
    const int64_t e0 = tile_id * NET_TILE + (int64_t)quarter * NET_OBS_ROWS;
    if (e0 >= N) return;
    const int nvalid = (int)((N - e0) < NET_OBS_ROWS ? (N - e0) : NET_OBS_ROWS);
    const char* tile = (const char*)state + tile_id * net_tile_bytes(P);
    NetState st((void*)tile, P);
    const int el0 = quarter * NET_OBS_ROWS;
    const int t_me = lane < nvalid ? st.period[el0 + lane] : -1;
    const int t0 = st.period[el0];
    const int uniform = __syncthreads_and(lane >= nvalid || t_me == t0);
    if (!uniform) {  // rare: per-instance rows straight to global memory
        if (tid < nvalid)
            net_write_obs<NET_TILE>(P, st.U, st.X, el0 + tid, st.ring, el0 + tid, st.period[el0 + tid], obs + (e0 + tid) * W);
        return;
    }
    // float64 columns: rows of the tile, in units of 1 KB: [0] keys, [1, J] X, then Y (E), U (M); window columns: slots
    // of the float32 ring copy (512-byte rows of st.ring32), 4 instead of 8 bytes read per column and instance
    const int rowX = 1, rowU = 1 + P.J + P.E;
    for (int c = tid; c < P.M; c += NET_OBS_THREADS) colrow[c] = (uint16_t)(rowU + c);
    for (int c = tid; c < P.J; c += NET_OBS_THREADS) colrow[P.M + c] = (uint16_t)(rowX + c);
    for (int i = tid; i < P.E; i += NET_OBS_THREADS) {
        const int L = P.L[i];
        if (L == 0) continue;
        int sl = net_mod(t0, L, P.Lmagic[i]);  // window element q (oldest first) lives in ring slot (t + q) % L
        uint16_t* dst = colrow + P.M + P.J + P.roff[i];
        for (int q = 0; q < L; q++) {
            dst[q] = (uint16_t)(P.roff[i] + sl);
            sl = sl + 1 == L ? 0 : sl + 1;
        }
    }
    __syncthreads();
    const double* src = (const double*)tile + el0 + lane;  // + row * 128
    float* orow = out + (size_t)lane * W;
    const int WD = P.M + P.J;  // columns [0, WD) are float64 rows, [WD, W) float32 rows
    const float* src32 = st.ring32 + el0 + lane;
    // all of this warp's columns are requested into L2 at once (one instruction each, no register, no scoreboard slot):
    // the batched loads below then wait for L2, not for HBM, and the CTA's share is in flight from the first cycle
    for (int c = warp; c < WD; c += NW) prefetch_l2(src + (size_t)colrow[c] * NET_TILE);
    for (int c = WD + warp; c < W; c += NW) prefetch_l2(src32 + (size_t)colrow[c] * NET_TILE);
    for (int c0 = warp; c0 < WD; c0 += NW * NET_OBS_BATCH) {
        double v[NET_OBS_BATCH];
#pragma unroll
        for (int j = 0; j < NET_OBS_BATCH; j++) {
            const int c = c0 + j * NW;
            v[j] = c < WD ? __ldcs(src + (size_t)colrow[c] * NET_TILE) : 0.0;
        }
#pragma unroll
        for (int j = 0; j < NET_OBS_BATCH; j++) {
            const int c = c0 + j * NW;
            if (c < WD) orow[c] = (float)v[j];
        }
    }
    for (int c0 = WD + warp; c0 < W; c0 += NW * NET_OBS_BATCH32) {  // one register per value: a deeper batch
        float v[NET_OBS_BATCH32];
#pragma unroll
        for (int j = 0; j < NET_OBS_BATCH32; j++) {
            const int c = c0 + j * NW;
            v[j] = c < W ? __ldcs(src32 + (size_t)colrow[c] * NET_TILE) : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < NET_OBS_BATCH32; j++) {
            const int c = c0 + j * NW;
            if (c < W) orow[c] = v[j];
        }
    }
    float* g = obs + e0 * W;
    if ((nvalid & 3) == 0 && ((uintptr_t)g & 15) == 0) {  // 4 rows of any length are a multiple of 16 bytes
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
            bulk_s2g(g, out, (uint32_t)((size_t)nvalid * W * 4));
            bulk_commit();
            bulk_wait_read0();
        }
    } else {
        __syncthreads();
        const int total = nvalid * W;
        for (int i = tid; i < total; i += NET_OBS_THREADS) g[i] = out[i];
    }
}

static int net_obs_launch(const NetHandle* H, const void* state, float* obs, cudaStream_t s) {
    const int64_t N = H->base.num_envs;
    const int64_t tiles = (N + NET_TILE - 1) / NET_TILE;
    // (launching the four CTAs of a tile as one thread-block cluster, so that their quarter rows reach DRAM together, was
    // measured slower: 0.19-0.20 ms against 0.18 ms)
    net_obs_kernel<<<(unsigned)(tiles * (NET_TILE / NET_OBS_ROWS)), NET_OBS_THREADS, net_obs_smem(H->dev), s>>>(H->dev, N, state,
                                                                                                               obs);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

static void net_launch(const NetHandle* H, const NetSimArgs& A, size_t smem, cudaStream_t s) {
    unsigned grid = (unsigned)((A.N + H->threads - 1) / H->threads);
    if (H->threads == 128)
        net_sim_kernel<128><<<grid, 128, smem, s>>>(H->dev, A);
    else if (H->threads == 64)
        net_sim_kernel<64><<<grid, 64, smem, s>>>(H->dev, A);
    else
        net_sim_kernel<32><<<grid, 32, smem, s>>>(H->dev, A);
}

// ---- fused rollout driven by an MLP actor (ORGYM_NET_POLICY_MLP) -----------------------------------------------------
// One CTA of MLP_THREADS threads = the NET_TILE = 128 consecutive envs of one rollout scratch tile (their lead-time rings
// stay there, [slot][128], as in net_sim_kernel's ROLLOUT mode) and one row of the partial sums.  The CTA runs them as
// 128 / ESUB sub-tiles of ESUB envs one after the other; weights and biases are staged in shared memory once per CTA
// (mlp.cuh).  Thread tid < ESUB owns env e0 + tid of the current sub-tile: its float64 work vectors are column tid of
// [slot][ESUB] rows, its accumulators live in its registers.  The float32 observation tile [obs_dim][ESUB] is the
// network's input: U and X rows are rewritten after each period, the pipeline rows shifted left in place and appended
// with the orders fulfilled (R[t], what the ring receives).  Per period the whole CTA runs the hidden layers and then
// the last layer into the action tile [E][ESUB] (one barrier each); the owner threads take the period through
// net_period, the same code as net_sim_kernel, with that tile as the requests.
struct NetMlpArgs {
    MlpNet net;
    int obs_off, buf_off[2], act_off;  // float offsets in dynamic shared memory (the weights start at 0)
    int work_off;                      // byte offset of the float64 work vectors
    float* action_traj;                // [N,T,E] or NULL
    float hi[NE];                      // upper bound of the action Box
};

template <int ESUB>
__global__ void __launch_bounds__(MLP_THREADS, 2) net_mlp_rollout_kernel(const __grid_constant__ NetDev P,
                                                                        const __grid_constant__ NetSimArgs A,
                                                                        const __grid_constant__ NetMlpArgs M) {
    static_assert(NET_TILE % ESUB == 0 && ESUB % 32 == 0 && ESUB <= MLP_THREADS, "sub-tiles of whole warps");
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ double red[NET_TILE / 32][7];
    constexpr int log2E = ESUB == 64 ? 6 : 5;
    const int tid = threadIdx.x, NL = M.net.L, J = P.J, E = P.E, Mk = P.M, T = P.T;
    float* fs = (float*)smem;
    float* obs = fs + M.obs_off;
    float* act = fs + M.act_off;
    double* sX = (double*)(smem + M.work_off);  // [J]
    double* sC = sX + J * ESUB;                 // [J]
    double* sR = sC + J * ESUB;                 // [E]
    double* sY = sR + E * ESUB;                 // [E]
    double* sU = sY + E * ESUB;                 // [M]
    double* sS = sU + Mk * ESUB;                // [M]
    mlp_stage_weights(M.net, fs);
    const int Klast = M.net.K[NL - 1];
    const float* Wlast = fs + M.net.w_off[NL - 1];
    const float* blast = fs + M.net.b_off[NL - 1];
    const float* hin = NL == 1 ? obs : fs + M.buf_off[(NL - 2) & 1];  // input of the last layer
    double* ring = NetState((char*)A.state + (int64_t)blockIdx.x * net_tile_bytes(P), P).ring;
    const bool owner = tid < ESUB;
    for (int sub = 0; sub < NET_TILE / ESUB; sub++) {
        const int64_t e0 = (int64_t)blockIdx.x * NET_TILE + (int64_t)sub * ESUB;
        const int64_t e = e0 + tid;
        const bool valid = owner && e < A.N;
        const int64_t ec = valid ? e : 0;  // clamp so that idle lanes stay in bounds
        const int el = sub * ESUB + tid;   // column of the scratch tile
        if (e0 >= A.N) {  // CTA-uniform: the sums of the missing warps are zero, like idle lanes of net_sim_kernel
            if (tid < 7 * (ESUB / 32)) red[sub * (ESUB / 32) + tid / 7][tid % 7] = 0.0;
            continue;
        }
        const uint64_t key = A.seed + (uint64_t)(A.env_offset + e);
        double ret = 0.0, s_sales = 0.0, s_dem = 0.0, s_unf = 0.0, s_inv = 0.0;
        if (owner) {  // reset (:326) and its observation [0 (M), I0 (J), 0 ...]
            for (int j = 0; j < J; j++) sX[j * ESUB + tid] = P.I0[j];
            for (int i = 0; i < E; i++) sY[i * ESUB + tid] = 0.0;
            for (int r = 0; r < Mk; r++) sU[r * ESUB + tid] = 0.0;
            if (valid)
                for (int k = 0; k < P.sumL; k++) ring[k * NET_TILE + el] = 0.0;
            for (int z = 0; z < P.obs_dim; z++)
                obs[z * ESUB + tid] = (z >= Mk && z < Mk + J) ? (float)P.I0[z - Mk] : 0.0f;
        }
        __syncthreads();
        for (int t = 0; t < T; t++) {
            const float* in = obs;
            for (int l = 0; l < NL - 1; l++) {
                float* out = fs + M.buf_off[l & 1];
                mlp_hidden_layer(in, out, fs + M.net.w_off[l], fs + M.net.b_off[l], M.net.K[l], M.net.Np[l], ESUB, log2E,
                                 M.net.act);
                __syncthreads();
                in = out;
            }
            // last layer: acc = b, then K ascending FMAs, no activation; then np.clip to the action Box in float32, NaN kept
            for (int idx = tid; idx < E * ESUB; idx += MLP_THREADS) {
                const int n = idx >> log2E, c = idx & (ESUB - 1);
                float y = blast[n];
                for (int k = 0; k < Klast; k++) y = __fmaf_rn(Wlast[n * Klast + k], hin[k * ESUB + c], y);
                float a = y > 0.0f ? y : 0.0f;
                a = a < M.hi[n] ? a : M.hi[n];
                a = y != y ? y : a;
                act[idx] = a;
                if (M.action_traj && e0 + c < A.N) M.action_traj[((e0 + c) * T + t) * E + n] = a;
            }
            __syncthreads();
            if (owner) {
                const double total = net_period<ESUB, ESUB>(
                    P, tid, el, ring, valid, t, sX, sC, sR, sY, sU, sS, [&] { return (const float*)act + tid; },
                    [&](int r) {
                        return A.demand ? rint(A.demand[ec * A.d_se + (int64_t)t * A.d_st + r])
                                        : (double)sample_fixed(P.dem[r], P.dem[r].table, key, A.episode, t, (uint32_t)r);
                    },
                    [](int, double) {}, [](int, double) {}, s_sales, s_dem, s_unf, s_inv);
                const double rw = P.disc[t] * total;  // :619
                ret += rw;
                if (valid && A.reward_traj) A.reward_traj[e * T + t] = rw;
                // observation of period t + 1 (:334-413)
                for (int r = 0; r < Mk; r++) obs[r * ESUB + tid] = (float)sU[r * ESUB + tid];
                for (int j = 0; j < J; j++) obs[(Mk + j) * ESUB + tid] = (float)sX[j * ESUB + tid];
                int k = Mk + J;
                for (int i = 0; i < E; i++) {
                    const int L = P.L[i];
                    if (L == 0) continue;  // :353
                    for (int q = 0; q + 1 < L; q++) obs[(k + q) * ESUB + tid] = obs[(k + q + 1) * ESUB + tid];
                    obs[(k + L - 1) * ESUB + tid] = (float)sR[i * ESUB + tid];
                    k += L;
                }
            }
            __syncthreads();
        }
        if (valid) {
            if (A.ep_return) A.ep_return[e] = ret;
            if (A.stats) {
                A.stats[e * 4 + 0] = s_sales; A.stats[e * 4 + 1] = s_dem; A.stats[e * 4 + 2] = s_unf; A.stats[e * 4 + 3] = s_inv;
            }
            if (A.final_X) for (int j = 0; j < J; j++) A.final_X[e * J + j] = sX[j * ESUB + tid];
            if (A.final_Y) for (int i = 0; i < E; i++) A.final_Y[e * E + i] = sY[i * ESUB + tid];
            if (A.final_U) for (int r = 0; r < Mk; r++) A.final_U[e * Mk + r] = sU[r * ESUB + tid];
        }
        if (A.partials && owner) {  // warp of 32 consecutive envs: the xor tree of net_sim_kernel<128>
            const double v[7] = {valid ? 1.0 : 0.0, valid ? ret : 0.0, valid ? ret * ret : 0.0, valid ? s_sales : 0.0,
                                 valid ? s_dem : 0.0, valid ? s_unf : 0.0, valid ? s_inv : 0.0};
#pragma unroll
            for (int z = 0; z < 7; z++) {
                double x = v[z];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
                if ((tid & 31) == 0) red[sub * (ESUB / 32) + (tid >> 5)][z] = x;
            }
        }
    }
    if (A.partials) {
        __syncthreads();
        if (tid < 7) {  // the four warps in order, as net_sim_kernel<128>
            double x = 0.0;
            for (int wv = 0; wv < NET_TILE / 32; wv++) x += red[wv][tid];
            A.partials[(size_t)blockIdx.x * 8 + tid] = x;
        }
    }
}

// Checks an orgym_mlp_t and the action bound against the graph (ORGYM_E_INVALID) and lays out one CTA's shared memory
// for it: the largest sub-tile of ESUB in {64, 32} envs whose working set fits (ORGYM_E_UNSUPPORTED, with the sizes,
// when none does).
static int net_mlp_plan(const NetDev& P, const orgym_mlp_t* mlp, const float* action_high, NetMlpArgs* M, int* esub,
                        size_t* smem_out) {
    ORGYM_REQUIRE(mlp, "policy ORGYM_NET_POLICY_MLP needs in->mlp");
    ORGYM_REQUIRE(action_high, "policy ORGYM_NET_POLICY_MLP needs in->action_high");
    if (P.obs_dim > ORGYM_MLP_MAX_WIDTH && mlp->width[0] == P.obs_dim) {  // large graphs: the input alone does not fit
        const size_t need = 4 * (size_t)P.obs_dim * (round_up(std::max(mlp->width[1], 1), MLP_TN) + 32);
        orgym_set_error("mlp: the observation has %d values (at most %d): one CTA of 32 envs needs at least %zu bytes of "
                        "shared memory for the first layer's weights and the observation tile; this build's limit is %d",
                        P.obs_dim, ORGYM_MLP_MAX_WIDTH, need, MLP_SMEM_BUDGET);
        return ORGYM_E_UNSUPPORTED;
    }
    memset(M, 0, sizeof(*M));
    if (int rc = mlp_net_plan(mlp, P.obs_dim, P.E, "the number of reorder links", &M->net)) return rc;
    for (int i = 0; i < P.E; i++) M->hi[i] = action_high[i];
    const int L = M->net.L, hmax = M->net.hmax;
    const int nbuf = L >= 3 ? 2 : (L == 2 ? 1 : 0);
    const size_t work = 8 * (size_t)(2 * P.J + 2 * P.E + 2 * P.M);  // bytes per env
    size_t smem = 0;
    for (int E = 64; E >= 32; E /= 2) {
        int g = M->net.wfloats;
        M->obs_off = g;
        g += (int)round_up((int64_t)P.obs_dim * E, 4);
        M->buf_off[0] = g;
        g += nbuf >= 1 ? hmax * E : 0;
        M->buf_off[1] = g;
        g += nbuf >= 2 ? hmax * E : 0;
        M->act_off = g;
        g += P.E * E;
        M->work_off = (int)round_up((int64_t)g * 4, 16);
        smem = (size_t)M->work_off + work * E;
        *esub = E;
        if (smem <= MLP_SMEM_BUDGET) break;
    }
    if (smem > MLP_SMEM_BUDGET) {
        orgym_set_error("mlp: one CTA of 32 envs needs %zu bytes of shared memory (weights and biases %d floats, observation "
                        "tile %d x 32, %d activation tile(s) %d x 32, action tile %d x 32, work vectors %zu bytes x 32); "
                        "this build's limit is %d",
                        smem, M->net.wfloats, P.obs_dim, nbuf, hmax, P.E, work, MLP_SMEM_BUDGET);
        return ORGYM_E_UNSUPPORTED;
    }
    *smem_out = smem;
    return ORGYM_OK;
}

// ------------------------------------------------------------------------------------------------
// host side of the C ABI
// ------------------------------------------------------------------------------------------------
// validate + flatten a config into NetDev (no CUDA calls)
static int net_fill(const orgym_netinv_config_t* c, NetDev& P) {
    ORGYM_REQUIRE(c, "null argument");
    // mirrors network_management.py:197-238
    ORGYM_REQUIRE(c->num_periods > 0, "num_periods must be positive");
    ORGYM_REQUIRE(c->alpha > 0 && c->alpha <= 1, "alpha must be in (0, 1]");
    ORGYM_REQUIRE(c->num_main >= 1 && c->num_reorder >= 0 && c->num_retail >= 0, "empty network");
    if (c->num_main > NJ || c->num_reorder > NE || c->num_retail > NM) {
        orgym_set_error("network too large for this build: %d main nodes (max %d), %d reorder links (max %d), %d retail links (max %d)",
                        c->num_main, NJ, c->num_reorder, NE, c->num_retail, NM);
        return ORGYM_E_UNSUPPORTED;
    }
    memset(&P, 0, sizeof(P));
    P.T = c->num_periods;
    P.backlog = c->backlog ? 1 : 0;
    P.J = c->num_main;
    P.E = c->num_reorder;
    P.M = c->num_retail;
#define FAIL(code, ...)            \
    do {                           \
        orgym_set_error(__VA_ARGS__); \
        return code;               \
    } while (0)
    {
        for (int j = 0; j < P.J; j++) {
            P.I0[j] = c->node_I0[j];
            P.h[j] = c->node_h[j];
            P.is_factory[j] = c->node_is_factory[j];
            P.is_retail[j] = c->node_is_retail[j];
            P.C[j] = c->node_C[j];
            P.v[j] = c->node_v[j];
            P.o[j] = c->node_o[j];
            if (!(P.I0[j] >= 0)) FAIL(ORGYM_E_INVALID, "Node %d: Invalid or missing I0>=0", j);
            if (!(P.h[j] >= 0)) FAIL(ORGYM_E_INVALID, "Node %d: Invalid or missing h>=0", j);
            if (P.is_factory[j]) {
                if (!(P.C[j] > 0)) FAIL(ORGYM_E_INVALID, "Node %d: Invalid or missing C>0", j);
                if (!(P.o[j] >= 0)) FAIL(ORGYM_E_INVALID, "Node %d: Invalid or missing o>=0", j);
                if (!(P.v[j] > 0 && P.v[j] <= 1)) FAIL(ORGYM_E_INVALID, "Node %d: Invalid or missing v in (0, 1]", j);
            } else if (!(P.v[j] > 0))
                FAIL(ORGYM_E_INVALID, "Node %d: yield must be positive", j);
        }
        for (int i = 0; i < P.E; i++) {
            int s = c->re_supplier[i], pu = c->re_purchaser[i], L = c->re_lead[i];
            if (s < -2 || s >= P.J || pu < -1 || pu >= P.J) FAIL(ORGYM_E_INVALID, "reorder link %d: bad node index", i);
            if (L < 0) FAIL(ORGYM_E_INVALID, "Edge %d: Invalid or missing L>=0", i);
            if (L > ORGYM_NET_MAX_LEAD) FAIL(ORGYM_E_UNSUPPORTED, "lead time %d exceeds this build's limit of %d", L, ORGYM_NET_MAX_LEAD);
            if (!(c->re_p[i] >= 0) || !(c->re_g[i] >= 0)) FAIL(ORGYM_E_INVALID, "Edge %d: Invalid or missing p>=0 / g>=0", i);
            if (i > 0 && s >= 0 && c->re_supplier[i - 1] > s)
                FAIL(ORGYM_E_INVALID, "reorder links must be sorted by supplier (network_management.py:179)");
            P.sup[i] = (int16_t)s;
            if (s >= 0) P.has_seg[s] = 1;
            P.pur[i] = (int16_t)pu;
            P.L[i] = (int16_t)L;
            P.roff[i] = P.sumL;
            P.Lmagic[i] = L > 1 ? (uint32_t)((0x100000000ULL + L - 1) / L) : 0u;
            P.sumL += L;
            P.p[i] = c->re_p[i];
            P.g[i] = c->re_g[i];
        }
        // a supplier's links must be contiguous (they are, in sorted order); raw (-1) / unclassified (-2) may interleave
        for (int i = 1; i < P.E; i++)
            for (int k = 0; k + 1 < i; k++)
                if (P.sup[i] >= 0 && P.sup[k] == P.sup[i] && P.sup[i - 1] != P.sup[i])
                    FAIL(ORGYM_E_INVALID, "links of supplier %d are not contiguous", (int)P.sup[i]);
        for (int r = 0; r < P.M; r++) {
            int j = c->rt_retailer[r];
            if (j < 0 || j >= P.J) FAIL(ORGYM_E_INVALID, "retail link %d: retailer is not an inventory-holding node", r);
            if (!(c->rt_p[r] >= 0) || !(c->rt_b[r] >= 0)) FAIL(ORGYM_E_INVALID, "Edge %d: Invalid or missing p>=0 / b>=0", r);
            P.rt_node[r] = (int16_t)j;
            P.rt_p[r] = c->rt_p[r];
            P.rt_b[r] = c->rt_b[r];
        }
        if (c->succ_ptr[P.J] > NSUCC || c->pred_ptr[P.J] > NE) FAIL(ORGYM_E_UNSUPPORTED, "adjacency lists too long");
        for (int j = 0; j <= P.J; j++) {
            P.succ_ptr[j] = (int16_t)c->succ_ptr[j];
            P.pred_ptr[j] = (int16_t)c->pred_ptr[j];
        }
        for (int z = 0; z < c->succ_ptr[P.J]; z++) {
            if (c->succ_idx[z] < 0 || c->succ_idx[z] >= P.E + P.M) FAIL(ORGYM_E_INVALID, "bad successor link id");
            P.succ_idx[z] = (int16_t)c->succ_idx[z];
        }
        for (int z = 0; z < c->pred_ptr[P.J]; z++) {
            if (c->pred_idx[z] < 0 || c->pred_idx[z] >= P.E) FAIL(ORGYM_E_INVALID, "bad predecessor link id");
            P.pred_idx[z] = (int16_t)c->pred_idx[z];
        }
        P.obs_dim = P.M + P.J + P.sumL;  // :190
    }
#undef FAIL
    return ORGYM_OK;
}

extern "C" int orgym_netinv_create(const orgym_netinv_config_t* c, int64_t num_envs, int device, orgym_handle_t* out) {
    ORGYM_REQUIRE(c && out, "null argument");
    NetHandle* H = new NetHandle();
    NetDev& P = H->dev;
    int rc = net_fill(c, P);
    if (rc != ORGYM_OK) {
        delete H;
        return rc;
    }
#define FAIL(code, ...)            \
    do {                           \
        orgym_set_error(__VA_ARGS__); \
        rc = code;                 \
        goto done;                 \
    } while (0)
    {
        rc = orgym_handle_base_init(&H->base, FAM_NETINV, device, num_envs);
        if (rc != ORGYM_OK) goto done;
        {
            DeviceGuard g(device);
            std::vector<double> disc((size_t)P.T);
            for (int t = 0; t < P.T; t++) disc[(size_t)t] = std::pow(c->alpha, (double)t);
            double* dd = nullptr;
            if (cudaMalloc(&dd, 8 * (size_t)P.T) != cudaSuccess) FAIL(ORGYM_E_CUDA, "device allocation failed");
            H->allocs.push_back(dd);
            cudaMemcpy(dd, disc.data(), 8 * (size_t)P.T, cudaMemcpyHostToDevice);
            P.disc = dd;
            for (int r = 0; r < P.M; r++) {
                rc = orgym_build_alias(&c->rt_dist[r], 1, &P.dem[r], &H->allocs);
                if (rc != ORGYM_OK) goto done;
                if (P.dem[r].kind == ORGYM_DIST_USER && P.dem[r].user_D_len != P.T)
                    FAIL(ORGYM_E_INVALID, "Edge %d: user_D length %d != num_periods %d", r, P.dem[r].user_D_len, P.T);
            }
            size_t per_thread = 8 * (size_t)(2 * P.J + 2 * P.E + 2 * P.M);
            H->threads = 128;
            while (H->threads > 32 && per_thread * H->threads > 200 * 1024) H->threads /= 2;
            if (per_thread * H->threads > 200 * 1024) FAIL(ORGYM_E_UNSUPPORTED, "network work vectors do not fit in shared memory");
            H->smem = per_thread * H->threads;
            int nblocks = (int)((num_envs + 31) / 32);  // enough for any block size
            H->partials = nullptr;
            size_t pbytes = sizeof(double) * (8 * (size_t)nblocks + ORGYM_REDUCE_EXTRA);
            if (cudaMalloc(&H->partials, pbytes) != cudaSuccess) FAIL(ORGYM_E_CUDA, "device allocation failed");
            H->allocs.push_back(H->partials);
            cudaMemset(H->partials, 0, pbytes);
            if (P.T > (1 << 20)) FAIL(ORGYM_E_UNSUPPORTED, "num_periods above 2^20 is not supported");
            cudaFuncSetAttribute(net_sim_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(220 * 1024));
            cudaFuncSetAttribute(net_sim_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(220 * 1024));
            cudaFuncSetAttribute(net_sim_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(220 * 1024));
            cudaFuncSetAttribute(net_obs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(220 * 1024));
            H->plan = net_plan(P);
            P.ring32 = H->plan.ring32;
            // kernel specialised for this topology (NVRTC); unless it is required, a failure falls back to the generic
            // kernel above
            H->dem_dev = nullptr;
            if (H->plan.jit) {
                std::string jerr;
                if (net_jit_build(H, &jerr) != 0) {
                    if (H->plan.jit == 2) FAIL(ORGYM_E_CUDA, "ORGYM_NET_JIT=2 but specialisation failed: %s", jerr.c_str());
                    fprintf(stderr, "[orgym_b200] network kernel specialisation unavailable (%s); using the generic kernel\n",
                            jerr.substr(0, 600).c_str());
                }
            }
        }
    }
done:
#undef FAIL
    if (rc != ORGYM_OK) {
        if (H->base.magic == ORGYM_MAGIC) {
            DeviceGuard g(device);
            for (void* p : H->allocs) cudaFree(p);
            orgym_handle_base_free(&H->base);
        }
        delete H;
        return rc;
    }
    *out = (orgym_handle_t)H;
    return ORGYM_OK;
}

extern "C" int orgym_netinv_destroy(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_NETINV)) return ORGYM_E_INVALID;
    NetHandle* H = (NetHandle*)h;
    {
        DeviceGuard g(H->base.device);
        orgym_jit_release(&H->jit);
        for (void* p : H->allocs) cudaFree(p);
    }
    orgym_handle_base_free(&H->base);
    delete H;
    return ORGYM_OK;
}

extern "C" int64_t orgym_netinv_state_bytes(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_NETINV)) return -1;
    NetHandle* H = (NetHandle*)h;
    return net_state_bytes(H->dev, H->base.num_envs);
}
extern "C" int32_t orgym_netinv_obs_dim(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_NETINV)) return -1;
    return ((NetHandle*)h)->dev.obs_dim;
}

extern "C" int orgym_netinv_reset(orgym_handle_t h, void* state_dev, int reseed, uint64_t seed, int64_t env_offset,
                                  const uint8_t* mask_dev, float* obs_dev, void* stream) {
    if (orgym_check_handle(h, FAM_NETINV)) return ORGYM_E_INVALID;
    NetHandle* H = (NetHandle*)h;
    ORGYM_REQUIRE(state_dev && obs_dev, "state_dev and obs_dev are required");
    DeviceGuard g(H->base.device);
    int64_t N = H->base.num_envs;
    net_reset_kernel<<<(unsigned)((N + 127) / 128), 128, 0, (cudaStream_t)stream>>>(H->dev, N, state_dev, reseed,
                                                                                  seed, env_offset, mask_dev, obs_dev);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

extern "C" int orgym_netinv_step(orgym_handle_t h, void* state_dev, const float* actions_dev,
                                 const double* demand_override_dev, int autoreset_mode, float* obs_dev,
                                 double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                                 const orgym_netinv_info_t* info, void* stream) {
    if (orgym_check_handle(h, FAM_NETINV)) return ORGYM_E_INVALID;
    NetHandle* H = (NetHandle*)h;
    ORGYM_REQUIRE(state_dev && actions_dev && obs_dev && reward_dev && terminated_dev && truncated_dev,
                  "state, actions, obs, reward, terminated and truncated pointers are required");
    ORGYM_REQUIRE(autoreset_mode >= 0 && autoreset_mode <= 2, "bad autoreset mode");
    DeviceGuard g(H->base.device);
    const NetDev& P = H->dev;
    NetSimArgs A;
    memset(&A, 0, sizeof(A));
    A.N = H->base.num_envs;
    A.rollout = 0;
    A.state = state_dev;
    A.policy = ORGYM_NET_POLICY_ACTIONS;
    A.actions = actions_dev;
    A.a_se = P.E;
    A.a_st = 0;
    A.demand = demand_override_dev;
    A.d_se = P.M;
    A.d_st = 0;
    A.autoreset = autoreset_mode;
    A.obs = obs_dev;
    A.reward = reward_dev;
    A.terminated = terminated_dev;
    A.truncated = truncated_dev;
    if (info) {
        A.info_demand = info->demand_dev;
        A.info_sales = info->sales_dev;
        A.info_profit = info->profit_dev;
        A.info_profit_total = info->profit_total_dev;
        ORGYM_REQUIRE(info->info_ld == 0 || info->info_ld >= H->base.num_envs, "info_ld must be 0 (row-major) or >= num_envs");
        A.info_ld = info->info_ld;
        A.final_obs = info->final_obs_dev;
    }
    A.err = H->base.err_dev;
    if (H->jit.fn) {
        int jrc = net_jit_launch(H, A, (cudaStream_t)stream);
        if (jrc != ORGYM_OK) return jrc;
        // large graphs: the streaming kernel leaves the state in HBM; the observation is assembled by the TMA-staged kernel
        if (H->plan.obs_kernel) return net_obs_launch(H, state_dev, obs_dev, (cudaStream_t)stream);
        return ORGYM_OK;
    }
    size_t tile = (size_t)H->threads * (P.obs_dim | 1) * 4;
    A.use_tile = (H->smem + tile <= 200 * 1024) ? 1 : 0;
    net_launch(H, A, H->smem + (A.use_tile ? tile : 0), (cudaStream_t)stream);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

extern "C" int orgym_netinv_export_state(orgym_handle_t h, const void* state_dev, double* X_dev, double* Y_dev,
                                         double* U_dev, int32_t* period_dev, void* stream) {
    if (orgym_check_handle(h, FAM_NETINV)) return ORGYM_E_INVALID;
    NetHandle* H = (NetHandle*)h;
    ORGYM_REQUIRE(state_dev, "state_dev is required");
    DeviceGuard g(H->base.device);
    int64_t N = H->base.num_envs;
    net_export_kernel<<<(unsigned)((N + 127) / 128), 128, 0, (cudaStream_t)stream>>>(H->dev, N, state_dev, X_dev,
                                                                                   Y_dev, U_dev, period_dev);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

extern "C" int orgym_netinv_rollout(orgym_handle_t h, void* scratch_dev, uint64_t seed, int64_t env_offset,
                                    uint32_t episode, const orgym_netinv_rollout_in_t* in,
                                    const orgym_netinv_rollout_out_t* out, void* stream) {
    if (orgym_check_handle(h, FAM_NETINV)) return ORGYM_E_INVALID;
    NetHandle* H = (NetHandle*)h;
    ORGYM_REQUIRE(in && out && scratch_dev, "null argument");
    ORGYM_REQUIRE(in->policy == ORGYM_NET_POLICY_ACTIONS || in->policy == ORGYM_NET_POLICY_CONSTANT ||
                      in->policy == ORGYM_NET_POLICY_MLP,
                  "unknown policy %d", in->policy);
    const bool mlp = in->policy == ORGYM_NET_POLICY_MLP;
    ORGYM_REQUIRE(mlp || in->actions_dev, "actions_dev is required");
    ORGYM_REQUIRE(mlp || !out->action_traj_dev, "action_traj_dev is written only by ORGYM_NET_POLICY_MLP rollouts");
    NetMlpArgs MA;
    int esub = 0;
    size_t mlp_smem = 0;
    if (mlp)
        if (int rc = net_mlp_plan(H->dev, in->mlp, in->action_high, &MA, &esub, &mlp_smem)) return rc;
    DeviceGuard g(H->base.device);
    NetSimArgs A;
    memset(&A, 0, sizeof(A));
    A.N = H->base.num_envs;
    A.env_offset = env_offset;
    A.rollout = 1;
    A.state = scratch_dev;
    A.seed = seed;
    A.episode = episode;
    A.policy = in->policy;
    A.actions = in->actions_dev;
    A.a_se = in->act_stride_env;
    A.a_st = in->act_stride_t;
    A.demand = in->demand_dev;
    A.d_se = in->dem_stride_env;
    A.d_st = in->dem_stride_t;
    A.ep_return = out->ep_return_dev;
    A.stats = out->stats_dev;
    A.reward_traj = out->reward_traj_dev;
    A.final_X = out->final_X_dev;
    A.final_Y = out->final_Y_dev;
    A.final_U = out->final_U_dev;
    A.partials = out->summary_dev ? H->partials : nullptr;
    const int thr = mlp ? NET_TILE : H->jit.fn ? NET_JIT_THREADS : H->threads;
    int nblocks = (int)((A.N + thr - 1) / thr);
    if (mlp) {  // always the ahead-of-time kernel, whatever ORGYM_NET_JIT says
        MA.action_traj = out->action_traj_dev;
        if (esub == 64) {
            orgym_ensure_dyn_smem<net_mlp_rollout_kernel<64>>(mlp_smem);
            net_mlp_rollout_kernel<64><<<nblocks, MLP_THREADS, mlp_smem, (cudaStream_t)stream>>>(H->dev, A, MA);
        } else {
            orgym_ensure_dyn_smem<net_mlp_rollout_kernel<32>>(mlp_smem);
            net_mlp_rollout_kernel<32><<<nblocks, MLP_THREADS, mlp_smem, (cudaStream_t)stream>>>(H->dev, A, MA);
        }
    } else if (H->jit.fn) {
        int rc = net_jit_launch(H, A, (cudaStream_t)stream);
        if (rc != ORGYM_OK) return rc;
    } else
        net_launch(H, A, H->smem, (cudaStream_t)stream);
    ORGYM_CUDA(cudaGetLastError());
    if (out->summary_dev) {
        int rr = orgym_launch_reduce(H->partials, nblocks, out->summary_dev, (cudaStream_t)stream);
        if (rr != ORGYM_OK) return rr;
    }
    return ORGYM_OK;
}

// debugging / test aid: the CUDA source the specialiser generates for a config (no GPU needed); compile_check != 0
// also runs it through NVRTC.  Returns the source length (excluding the terminator) in *needed.
extern "C" int orgym_netinv_codegen(const orgym_netinv_config_t* cfg, int compile_check, char* buf, int64_t buflen,
                                    int64_t* needed) {
    NetDev* P = new NetDev();
    int rc = net_fill(cfg, *P);
    if (rc != ORGYM_OK) {
        delete P;
        return rc;
    }
    const NetPlan plan = net_plan(*P);
    P->ring32 = plan.ring32;
    std::string src = net_jit_source(*P, plan);
    delete P;
    if (needed) *needed = (int64_t)src.size();
    if (buf && buflen > 0) {
        size_t n = src.size() < (size_t)buflen - 1 ? src.size() : (size_t)buflen - 1;
        memcpy(buf, src.data(), n);
        buf[n] = 0;
    }
    if (compile_check) {
        std::string err;
        int jr = orgym_jit_compile_only(src, &err);
        if (jr != 0) {
            orgym_set_error("%s", err.substr(0, 900).c_str());
            return ORGYM_E_UNSUPPORTED;
        }
    }
    return ORGYM_OK;
}

extern "C" int orgym_netinv_is_specialised(orgym_handle_t h) {
    if (orgym_check_handle(h, FAM_NETINV)) return ORGYM_E_INVALID;
    return ((NetHandle*)h)->jit.fn ? 1 : 0;
}
