/*
 * orgym_b200.h -- C ABI of the B200-native batched inventory simulator.
 *
 * The reference (jacklu2016/or-gym-inventory) is pure Python and has no FFI
 * layer; its plug-in contract is the Gymnasium `Env` protocol.  Each entry
 * point below replaces one method of that protocol for a whole batch of
 * independent env instances resident in HBM.  `file:line` citations are into
 * the reference tree.
 *
 * Conventions
 *  - plain C: opaque handle, plain pointers and sizes, no torch / C++ types;
 *  - every `*_dev` pointer is DEVICE memory owned by the CALLER (e.g. a torch
 *    CUDA tensor's data_ptr()); the library allocates only its handle and the
 *    small read-only tables uploaded by `*_create` (alias tables, alpha**t,
 *    block partial sums); no device memory is allocated or freed on the
 *    reset/step/rollout path (the rare configurations whose working set needs
 *    global scratch take it from the caller: *_rollout_scratch_bytes).  The
 *    one lazy step is the NVRTC build of a specialised rollout kernel on the
 *    first eligible orgym_invmgmt_rollout (about 1 s, cubin cached on disk);
 *    orgym_invmgmt_specialise does it ahead of time;
 *  - all calls are asynchronous and ordered on `stream` (a cudaStream_t passed
 *    as void*; NULL = legacy default stream);
 *  - return value 0 = ok, negative = error (ORGYM_E_*), message available from
 *    orgym_last_error() (thread-local); nothing throws across the ABI;
 *  - a handle is not thread-safe and runs ONE rollout at a time (its block
 *    partial-sum buffer is shared by rollouts on any stream); distinct handles
 *    may be used concurrently.
 *  - there is NO CPU fallback: without a CUDA device every compute entry point
 *    returns ORGYM_E_CUDA.
 *
 * State memory.  `*_state_bytes(h)` tells the caller how many bytes of device
 * memory one batch needs; the caller allocates it (256-byte aligned) and passes
 * it to reset/step.  The layout is struct-of-arrays (`field[slot][env]`) so that
 * one-env-per-thread kernels read and write it fully coalesced; it is private to
 * the library (use the *_export_* calls to look inside).
 *
 * Random numbers.  Demand is drawn from a counter-based Philox4x32-10 stream
 * keyed by (seed + global env id) with counter (period, episode, stream id):
 * results do not depend on the batch size, the launch geometry or how the env
 * id range is sharded over GPUs (`env_offset`).  Passing a `demand_override`
 * array replays a recorded demand trace instead (bit-exact parity path).
 */
#ifndef ORGYM_B200_H
#define ORGYM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORGYM_VERSION 100 /* 0.1.0 */

#define ORGYM_OK 0
#define ORGYM_E_INVALID (-1)     /* bad argument / config (mirrors the reference's asserts) */
#define ORGYM_E_CUDA (-2)        /* CUDA runtime error, or no device */
#define ORGYM_E_UNSUPPORTED (-3) /* valid for the reference but outside this build's limits */

/* compile-time limits of this build.  Every configuration inside them runs; the fast paths additionally need the
 * per-CTA working set to fit in shared memory -- serial env step: 128 x obs_dim x (4|8) B observation tile (else the
 * rows are written directly); serial env rollout: 128 x sum(max(L_i,1)) x (4|8) B x (1|2) rings (else the caller
 * provides a scratch buffer, orgym_invmgmt_rollout_scratch_bytes); network env: specialised kernels up to 128 reorder
 * links. */
#define ORGYM_INV_MAX_STAGES 16 /* inventory-holding stages n = m-1 */
#define ORGYM_INV_MAX_LEAD 64
#define ORGYM_NV_MAX_LEAD 64
#define ORGYM_NET_MAX_NODES 64    /* main (inventory-holding) nodes */
#define ORGYM_NET_MAX_REORDER 160 /* reorder links */
#define ORGYM_NET_MAX_RETAIL 32   /* retail (market) links */
#define ORGYM_NET_MAX_LEAD 64

typedef struct orgym_handle_s* orgym_handle_t;

const char* orgym_last_error(void);
int orgym_version(void);
/* number of visible CUDA devices (0 when there is none; never fails) */
int orgym_device_count(void);

/* autoreset behaviour of *_step (gymnasium >= 1.0 AutoresetMode) */
#define ORGYM_AUTORESET_DISABLED 0  /* stepping a finished env is an error (reference: IndexError) */
#define ORGYM_AUTORESET_NEXT_STEP 1 /* a finished env is reset by the NEXT step call (action ignored, reward 0) */
#define ORGYM_AUTORESET_SAME_STEP 2 /* reset in the step that finishes; last obs goes to final_obs */

/* sticky per-handle device error bits, read back with orgym_errors() */
#define ORGYM_ERR_STEP_PAST_END 1u /* step on a finished env with autoreset disabled */
#define ORGYM_ERR_INT32_RANGE 2u   /* a value left the int32 range while the compact state format was selected */

/* demand distributions, numbered as the reference's `dist` (inventory_management.py:169-184) */
#define ORGYM_DIST_POISSON 1   /* p0 = mu */
#define ORGYM_DIST_BINOMIAL 2  /* p0 = n, p1 = p */
#define ORGYM_DIST_RANDINT 3   /* p0 = low, p1 = high (inclusive) */
#define ORGYM_DIST_GEOMETRIC 4 /* p0 = p; support 1,2,... like numpy */
#define ORGYM_DIST_USER 5      /* deterministic trace user_D[period] */

typedef struct {
    int32_t kind; /* ORGYM_DIST_* */
    double p0, p1;
    const int64_t* user_D; /* HOST pointer, ORGYM_DIST_USER only */
    int32_t user_D_len;
} orgym_dist_t;

/* ------------------------------------------------------------------------- *
 * Serial multi-echelon env: InvManagementMasterEnv (inventory_management.py:19)
 * ------------------------------------------------------------------------- */
typedef struct {
    int32_t num_stages;         /* m = len(I0)+1  (inventory_management.py:98) */
    int32_t periods;            /* :67 */
    int32_t backlog;            /* :75  1 = backlog, 0 = lost sales */
    int32_t wide_state;         /* 1 = int64 state (exact for any action); 0 = compact int32 state with range check */
    const int64_t* init_inv;    /* [m-1] I0  (:87) */
    const int64_t* capacity;    /* [m-1] c   (:93) */
    const int64_t* lead_time;   /* [m-1] L   (:94) */
    const double* unit_price;   /* [m] float32-rounded [p]+r[:-1] (:89) */
    const double* unit_cost;    /* [m] float32-rounded r          (:90) */
    const double* demand_cost;  /* [m] float32-rounded k          (:91) */
    const double* holding_cost; /* [m] float32-rounded h+[0]      (:92) */
    double alpha;               /* :78, reward = alpha**t * profit (:322) */
    orgym_dist_t dist;          /* :169-184 */
} orgym_invmgmt_config_t;

/* optional per-step outputs (any pointer may be NULL); mirrors the info dict of step (:334-345) */
typedef struct {
    int64_t* demand_dev;      /* [N]    demand_realized */
    int64_t* sales_dev;       /* [N,m]  sales */
    int64_t* unfulfilled_dev; /* [N,m]  unfulfilled */
    double* profit_dev;       /* [N]    period_profit (undiscounted) */
    int64_t* final_obs_dev;   /* [N,obs_dim] last observation of an episode (SAME_STEP autoreset) */
    /* layout of sales / unfulfilled: 0 = row-major [N][m]; ld > 0 = column-major [m][ld], ld >= N, element (env, k)
     * at k*ld + env (coalesced stores).  final_obs_dev is always row-major. */
    int64_t info_ld;
} orgym_invmgmt_info_t;

int orgym_invmgmt_create(const orgym_invmgmt_config_t* cfg, int64_t num_envs, int device, orgym_handle_t* out);
int orgym_invmgmt_destroy(orgym_handle_t h);
int64_t orgym_invmgmt_state_bytes(orgym_handle_t h);
int32_t orgym_invmgmt_obs_dim(orgym_handle_t h); /* (m-1)*(lt_max+1)  (:119) */
int32_t orgym_invmgmt_act_dim(orgym_handle_t h); /* m-1 */

/* reset (inventory_management.py:186-222) + first _get_obs (:354-391).
 * reseed != 0: env i gets Philox key seed + env_offset + i and episode 0; reseed == 0: keys kept, episode += 1.
 * mask_dev: NULL = all envs, else uint8[N], only envs with mask != 0 are reset (their obs rows are rewritten). */
int orgym_invmgmt_reset(orgym_handle_t h, void* state_dev, int reseed, uint64_t seed, int64_t env_offset,
                        const uint8_t* mask_dev, int64_t* obs_dev, void* stream);

/* one period for every env: step (inventory_management.py:224-352) + _get_obs.
 * actions_dev: [N,m-1], int64 (action_is_f64 == 0) or float64 (truncated toward 0 after max(a,0), :250).
 * demand_override_dev: NULL = sample on device, else int64[N] demand for this period (replay). */
int orgym_invmgmt_step(orgym_handle_t h, void* state_dev, const void* actions_dev, int action_is_f64,
                       const int64_t* demand_override_dev, int autoreset_mode, int64_t* obs_dev,
                       double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                       const orgym_invmgmt_info_t* info, void* stream);

/* copy the live state out for inspection / parity tests (any pointer may be NULL):
 * I int64[N,m-1], B int64[N,m], period int32[N]. */
int orgym_invmgmt_export_state(orgym_handle_t h, const void* state_dev, int64_t* I_dev, int64_t* B_dev,
                               int32_t* period_dev, void* stream);

/* on-device policies for the fused rollout */
#define ORGYM_POLICY_ACTIONS 0    /* pre-staged actions */
#define ORGYM_POLICY_BASE_STOCK 1 /* benchmark_InvManagementBacklogEnv.py:142-198; param[0] = safety factor, param[1] = mu */
#define ORGYM_POLICY_RANDOM 2     /* a_i ~ U{0..c_i} from a separate Philox sub-stream */
#define ORGYM_POLICY_MLP 3        /* actor network evaluated on the device, in->mlp */

/* A trained multilayer-perceptron actor (e.g. stable-baselines3's MlpPolicy: policy_net + action_net), evaluated inside
 * the fused rollout.  Each period the network sees exactly the observation step() returns (inventory_management.py:
 * 354-391): I[t] first, then the last min(t, lt_max) requested orders, left-aligned and oldest first, zeros after them.
 * Numerics:
 *   x   = float32(obs)                  round to nearest (= torch .float())
 *   h_l = act(W_l h_{l-1} + b_l)        float32; each output: acc = b, then acc = fmaf(w_k, x_k, acc) for k = 0..K-1
 *                                       ascending (no split-K, no cross-env reduction); act = tanhf (the accurate one,
 *                                       not tanh.approx) or max(x, 0) with NaN kept
 *   y   = W_L h_{L-1} + b_L             no activation after the last Linear
 *   q_i = (int64) trunc(min(max((double)y_i, 0), (double)c_i)),   NaN -> 0
 * i.e. SB3's deterministic predict for a Box action space (the Gaussian mean clipped to [low, high]) followed by the
 * env's own float-action rule (max(a, 0), truncation, :250).  Requests lie in [0, c_i], so sampled-demand MLP rollouts
 * use the compact int32 arithmetic exactly like the base-stock policy, and results are a pure function of (weights,
 * seed, global env id, episode): independent of batch size, launch geometry and env_offset sharding. */
#define ORGYM_MLP_MAX_LAYERS 4
#define ORGYM_MLP_MAX_WIDTH 256
#define ORGYM_MLP_TANH 1
#define ORGYM_MLP_RELU 2
typedef struct {
    int32_t num_layers;                            /* Linear layers, 1..ORGYM_MLP_MAX_LAYERS */
    int32_t activation;                            /* ORGYM_MLP_TANH | ORGYM_MLP_RELU, after every Linear but the last */
    int32_t width[ORGYM_MLP_MAX_LAYERS + 1];       /* width[0] = obs_dim, width[num_layers] = m-1 */
    const float* weight_dev[ORGYM_MLP_MAX_LAYERS]; /* [width[l+1]][width[l]] row-major = torch.nn.Linear.weight */
    const float* bias_dev[ORGYM_MLP_MAX_LAYERS];   /* [width[l+1]] or NULL */
} orgym_mlp_t;

typedef struct {
    int32_t policy;
    double param[4];
    /* ORGYM_POLICY_ACTIONS: element (env e, period t, stage i) at actions_dev[e*stride_env + t*stride_t + i] */
    const int64_t* actions_dev;
    int64_t act_stride_env, act_stride_t;
    /* optional demand replay: element (e, t) at demand_dev[e*stride_env + t*stride_t]; NULL = sample */
    const int64_t* demand_dev;
    int64_t dem_stride_env, dem_stride_t;
    /* device scratch of orgym_invmgmt_rollout_scratch_bytes(h) bytes; may be NULL when that is 0 (almost always) */
    void* scratch_dev;
    /* HOST pointer, read only when policy == ORGYM_POLICY_MLP.  ORGYM_E_INVALID for a malformed network (layer count,
     * widths outside 1..ORGYM_MLP_MAX_WIDTH or not matching obs_dim / m-1, null weights); ORGYM_E_UNSUPPORTED when the
     * weights, activations, observation tile and lead-time rings of one CTA do not fit in shared memory. */
    const orgym_mlp_t* mlp;
} orgym_invmgmt_rollout_in_t;

/* per-episode results; every pointer may be NULL.  stats columns are the reference evaluator's metrics
 * (benchmark_InvManagementBacklogEnv.py:381-441): [sum sales[0], sum demand, sum unfulfilled[0], sum_t sum_i max(0,I_i)] */
typedef struct {
    double* ep_return_dev;   /* [N]  sum_t reward_t, accumulated in period order */
    int64_t* stats_dev;      /* [N,4] */
    double* reward_traj_dev; /* [N,T] per-period reward (parity tests) */
    int64_t* final_I_dev;    /* [N,m-1] */
    int64_t* final_B_dev;    /* [N,m] */
    double* summary_dev;     /* [8] batch sums: n, sum ret, sum ret^2, sum sales, sum demand, sum stockout, sum end inv, 0 */
    int32_t* stats32_dev;    /* [N,4] the same statistics as stats_dev, saturated to int32 (halves the result traffic) */
    int64_t* action_traj_dev; /* [N,T,m-1] requested orders per period (the reference's action_log, :268); any policy */
} orgym_invmgmt_rollout_out_t;

/* fused reset + `periods` steps of every env with state held on chip (no state_dev needed).
 * Demand / random-policy streams are the same Philox streams reset+step would use for (seed, env_offset+i, episode). */
int orgym_invmgmt_rollout(orgym_handle_t h, uint64_t seed, int64_t env_offset, uint32_t episode,
                          const orgym_invmgmt_rollout_in_t* in, const orgym_invmgmt_rollout_out_t* out,
                          void* stream);

/* bytes of caller-owned device scratch a rollout needs (in->scratch_dev): 0 unless the lead-time rings cannot live in
 * shared memory (sum of max(L_i,1) beyond ~100) */
int64_t orgym_invmgmt_rollout_scratch_bytes(orgym_handle_t h);

/* The fused rollout is additionally specialised per configuration AND policy at run time: for 1..6 stages, up to 64
 * periods and a sum of lead times up to 40, the on-device base-stock (integer levels) and random policies run kernels
 * generated as straight-line CUDA (lead-time rings in registers, every index, price and base-stock level a literal, so
 * the compiler folds whatever does not depend on the demand; the profit in integer arithmetic when the generator can
 * prove that no float64 operation of the reference's expression rounds) and compiled for sm_100a with NVRTC.  Results
 * are bit-identical to the ahead-of-time kernel.  Rollouts that request reward_traj, final_I/B or action_traj, and
 * ORGYM_POLICY_MLP rollouts, always run the ahead-of-time kernels (also under ORGYM_INV_JIT=2).
 *   orgym_invmgmt_specialise  builds the kernel for in->policy / in->param now (ORGYM_OK), or says why it cannot:
 *                             ORGYM_E_UNSUPPORTED = configuration / policy outside the specialiser's range
 *                             (ORGYM_POLICY_MLP is never specialised),
 *                             ORGYM_E_CUDA = NVRTC unavailable or the compile failed; orgym_last_error() has the log.
 *                             Without this call the first eligible rollout builds it (up to 16 variants per handle).
 *   environment ORGYM_INV_JIT 0 = ahead-of-time kernels only; 1 (default) = specialise, fall back silently to the
 *                             ahead-of-time kernel; 2 = an eligible rollout that cannot be specialised is an error.
 *   orgym_invmgmt_codegen     returns the generated source for `in` (NULL = the benchmark's base-stock, levels
 *                             (L_i+1) * dist.p0) and, with compile_check != 0, runs it through NVRTC (no GPU needed). */
int orgym_invmgmt_specialise(orgym_handle_t h, const orgym_invmgmt_rollout_in_t* in);
int orgym_invmgmt_codegen(const orgym_invmgmt_config_t* cfg, const orgym_invmgmt_rollout_in_t* in, int compile_check,
                          char* buf, int64_t buflen, int64_t* needed);
/* diagnostic (no GPU needed): rigorous bounds on the integers of an episode driven by an on-device policy (requests within
 * [0, c_i]): *xvar bounds |on-hand|, |backlog|, |order|, |sales| of any stage and period, *xsum the per-episode statistics,
 * *profit_mag (may be NULL) the sum of |terms| of one period's profit.  They decide between int32 and int64 rollout
 * arithmetic and feed the specialiser's proof that the profit never rounds. */
int orgym_invmgmt_value_bounds(const orgym_invmgmt_config_t* cfg, double* xvar, double* xsum, double* profit_mag);
/* 1 when the most recent rollout of this handle ran a specialised kernel (or orgym_invmgmt_specialise just built one) */
int orgym_invmgmt_is_specialised(orgym_handle_t h);

/* ------------------------------------------------------------------------- *
 * Newsvendor: NewsvendorEnv (newsvendor.py:13)
 * ------------------------------------------------------------------------- */
typedef struct {
    int32_t lead_time;          /* newsvendor.py:65 (already clamped >= 0) */
    int32_t step_limit;         /* :68 */
    double max_inventory;       /* :66 */
    double max_order_quantity;  /* :67 */
    double p_max, h_max, k_max, mu_max; /* :69-72 */
} orgym_newsvendor_config_t;

typedef struct {
    int64_t* demand_dev; /* [N] */
    double* parts_dev;   /* [N,4] revenue, purchase_cost, holding_cost, lost_sales_penalty (newsvendor.py:195-199) */
    float* final_obs_dev; /* [N,obs_dim] (SAME_STEP autoreset) */
    int64_t info_ld;      /* layout of parts: 0 = row-major [N][4]; ld > 0 = column-major [4][ld], ld >= N */
} orgym_newsvendor_info_t;

int orgym_newsvendor_create(const orgym_newsvendor_config_t* cfg, int64_t num_envs, int device, orgym_handle_t* out);
int orgym_newsvendor_destroy(orgym_handle_t h);
int64_t orgym_newsvendor_state_bytes(orgym_handle_t h);
int32_t orgym_newsvendor_obs_dim(orgym_handle_t h); /* lead_time + 5 (:76) */

/* reset (newsvendor.py:100-123).  fixed_params_dev: NULL = draw (price,cost,h,k,mu) with the five-uniform
 * recipe (:105-111) from the env's Philox stream; else float64[N,5] per-env parameters
 * (options={'fixed_params':...}, benchmark_newsvendor_sb3_rllib.py:276-291).  Parameters given here stay pinned:
 * the automatic resets of orgym_newsvendor_step keep them (the benchmark's env re-applies them on every reset)
 * until the env is reset again with fixed_params_dev == NULL. */
int orgym_newsvendor_reset(orgym_handle_t h, void* state_dev, int reseed, uint64_t seed, int64_t env_offset,
                           const uint8_t* mask_dev, const double* fixed_params_dev, float* obs_dev, void* stream);

/* step (newsvendor.py:125-204).  actions_dev float32[N,1].  demand_override_dev int64[N] or NULL. */
int orgym_newsvendor_step(orgym_handle_t h, void* state_dev, const float* actions_dev,
                          const int64_t* demand_override_dev, int autoreset_mode, float* obs_dev,
                          double* reward_dev, uint8_t* terminated_dev, uint8_t* truncated_dev,
                          const orgym_newsvendor_info_t* info, void* stream);

/* float64[N,5] price, cost, h, k, mu as Python floats (newsvendor.py:105-111) */
int orgym_newsvendor_export_params(orgym_handle_t h, const void* state_dev, double* params_dev, void* stream);

#define ORGYM_NV_POLICY_ACTIONS 0
#define ORGYM_NV_POLICY_ORDER_UP_TO 1 /* benchmark_newsvendor.py:97-111;   param[0] = safety factor */
#define ORGYM_NV_POLICY_CLASSIC 2     /* benchmark_newsvendor.py:113-161 (k_vs_h); param[0] = safety factor */
#define ORGYM_NV_POLICY_SS 3          /* benchmark_newsvendor_sb3_rllib.py:363-371; param[0] = S buffer factor */
#define ORGYM_NV_POLICY_MLP 4         /* actor network evaluated on the device, in->mlp */

/* ORGYM_NV_POLICY_MLP: a trained actor network (orgym_mlp_t, width[0] = lead_time + 5, width[num_layers] = 1), e.g. a
 * stable-baselines3 MlpPolicy as benchmark_newsvendor.py:164 wraps it, evaluated inside the fused rollout.  Per period,
 * for each env:
 *   x    = the float32 observation step() returns: price, cost, h, k, mu, then the pipeline oldest first (:206-208)
 *   h_l, y = exactly the serial env's contract (orgym_mlp_t above): acc = b, then fmaf ascending in k; accurate tanhf
 *          or NaN-keeping ReLU; no activation after the last Linear
 *   a    = NaN if y is NaN, else min(max(y, 0f), (float)max_order_quantity)   (SB3 predict's np.clip to the Box, float32)
 * a then takes the env's own action rule, exactly like an ORGYM_NV_POLICY_ACTIONS action (.item(), np.clip in float64,
 * :131-132); action_traj_dev records a.  A NaN action places no order when lead_time > 0; with lead_time = 0 it is also
 * the stock on hand (:136-139), so the reward is NaN, as in the reference.  Results are a pure function of (weights,
 * seed, global env id, episode): independent of batch size and env_offset sharding. */

typedef struct {
    int32_t policy;
    double param[4];
    const float* actions_dev; /* (e,t) at actions_dev[e*stride_env + t*stride_t] */
    int64_t act_stride_env, act_stride_t;
    const int64_t* demand_dev;
    int64_t dem_stride_env, dem_stride_t;
    const double* fixed_params_dev; /* float64[N,5] or NULL */
    /* HOST pointer, read only when policy == ORGYM_NV_POLICY_MLP.  ORGYM_E_INVALID for a missing or malformed network
     * (layer count, widths outside 1..ORGYM_MLP_MAX_WIDTH, width[0] != lead_time + 5, width[num_layers] != 1, null
     * weights); ORGYM_E_UNSUPPORTED when the weights, activations, observation tile and Poisson CDF tile of one CTA do
     * not fit in shared memory. */
    const orgym_mlp_t* mlp;
} orgym_newsvendor_rollout_in_t;

typedef struct {
    double* ep_return_dev;   /* [N] */
    double* stats_dev;       /* [N,4]: sum sales units, sum demand, sum lost units, sum excess units */
    double* reward_traj_dev; /* [N,T] */
    float* action_traj_dev;  /* [N,T] actions the policy produced */
    float* final_obs_dev;    /* [N,obs_dim] */
    double* summary_dev;     /* [8] n, sum ret, sum ret^2, sum sales, sum demand, sum lost, sum excess, 0 */
} orgym_newsvendor_rollout_out_t;

int orgym_newsvendor_rollout(orgym_handle_t h, uint64_t seed, int64_t env_offset, uint32_t episode,
                             const orgym_newsvendor_rollout_in_t* in, const orgym_newsvendor_rollout_out_t* out,
                             void* stream);

/* ------------------------------------------------------------------------- *
 * Network env: NetInvMgmtMasterEnv (network_management.py:26)
 * The caller flattens the networkx graph (network_management.py:146-195) into the arrays below.
 * Node indices are positions in `main_nodes` (sorted, :176); a supplier that is a raw-material node
 * (:169) is encoded as -1.
 * ------------------------------------------------------------------------- */
typedef struct {
    int32_t num_periods; /* :67 */
    int32_t backlog;     /* :68 (after the ctor quirk :83-85 has been resolved by the caller) */
    double alpha;        /* :69 */
    /* main nodes, in sorted order (:176) */
    int32_t num_main;
    const double* node_I0;         /* [J] (:326) */
    const double* node_h;          /* [J] holding cost (:590) */
    const uint8_t* node_is_factory;/* [J] 'C' in attrs (:170) */
    const uint8_t* node_is_retail; /* [J] in self.retail (:174), gates the backlog penalty (:605) */
    const double* node_C;          /* [J] capacity (factories) */
    const double* node_v;          /* [J] yield; 1.0 for distributors (:484) */
    const double* node_o;          /* [J] operating cost (factories, :601) */
    /* reorder links in sorted (supplier, purchaser) order (:179) = action order (:442) */
    int32_t num_reorder;
    const int32_t* re_supplier;  /* [E] main-node index, -1 = raw material, -2 = unclassified supplier (order 0) */
    const int32_t* re_purchaser; /* [E] main-node index (or -1 if the purchaser holds no inventory) */
    const int32_t* re_lead;      /* [E] L (:184) */
    const double* re_p;          /* [E] purchase price (:586) */
    const double* re_g;          /* [E] pipeline holding cost (:591) */
    /* retail links in graph.edges() order (:158) */
    int32_t num_retail;
    const int32_t* rt_retailer; /* [M] main-node index */
    const double* rt_p;         /* [M] price (:582) */
    const double* rt_b;         /* [M] backlog cost (:608) */
    const orgym_dist_t* rt_dist;/* [M] demand distribution (:240-267); ORGYM_DIST_USER = user_D trace */
    /* profit terms keep the reference's Python-sum order: per main node, the successor list (:582, :599, :608)
     * and the predecessor list (:586, :591) in networkx adjacency order.  Entries are link ids:
     * reorder link e -> e ; retail link r -> num_reorder + r. */
    const int32_t* succ_ptr; /* [J+1] CSR offsets */
    const int32_t* succ_idx; /* [succ_ptr[J]] */
    const int32_t* pred_ptr; /* [J+1] */
    const int32_t* pred_idx; /* [pred_ptr[J]] reorder link ids */
} orgym_netinv_config_t;

typedef struct {
    double* demand_dev;    /* [N,M] D[t]   */
    double* sales_dev;     /* [N,E+M] fulfilled reorder links then retail links, S[t] */
    double* profit_dev;    /* [N,J] P[t] per node */
    double* profit_total_dev; /* [N] undiscounted period profit (:630) */
    float* final_obs_dev;  /* [N,obs_dim] (SAME_STEP autoreset) */
    /* layout of the two-dimensional tensors above (demand, sales, profit): 0 = row-major [N][dim];
     * ld > 0 = column-major [dim][ld] with ld >= N, element (env, k) at k*ld + env -- every store of the kernels is then
     * a coalesced one (the row-major form costs the 64-node step kernel ~30 %).  final_obs_dev is always row-major. */
    int64_t info_ld;
} orgym_netinv_info_t;

int orgym_netinv_create(const orgym_netinv_config_t* cfg, int64_t num_envs, int device, orgym_handle_t* out);
int orgym_netinv_destroy(orgym_handle_t h);
int64_t orgym_netinv_state_bytes(orgym_handle_t h);
int32_t orgym_netinv_obs_dim(orgym_handle_t h); /* M + J + sum(L)  (:190) */

/* reset (network_management.py:301-332) + _get_obs (:334-413) */
int orgym_netinv_reset(orgym_handle_t h, void* state_dev, int reseed, uint64_t seed, int64_t env_offset,
                       const uint8_t* mask_dev, float* obs_dev, void* stream);

/* step (network_management.py:436-635).  actions_dev float32[N,E]; demand_override_dev float64[N,M] or NULL */
int orgym_netinv_step(orgym_handle_t h, void* state_dev, const float* actions_dev,
                      const double* demand_override_dev, int autoreset_mode, float* obs_dev, double* reward_dev,
                      uint8_t* terminated_dev, uint8_t* truncated_dev, const orgym_netinv_info_t* info,
                      void* stream);

/* X float64[N,J], Y float64[N,E], U float64[N,M], period int32[N]; any may be NULL */
int orgym_netinv_export_state(orgym_handle_t h, const void* state_dev, double* X_dev, double* Y_dev,
                              double* U_dev, int32_t* period_dev, void* stream);

#define ORGYM_NET_POLICY_ACTIONS 0
#define ORGYM_NET_POLICY_CONSTANT 1 /* benchmark_NetInvMgmtBacklogEnv.py:119-136: same float32 action vector every period */
#define ORGYM_NET_POLICY_MLP 2      /* actor network evaluated on the device, in->mlp */

/* ORGYM_NET_POLICY_MLP: a trained actor network (orgym_mlp_t, width[0] = obs_dim, width[num_layers] = E), e.g. the
 * stable-baselines3 MlpPolicy that benchmark_NetInvMgmtLostSalesEnv_sb3_rllib.py trains, evaluated inside the fused
 * rollout.  Per period, for each env:
 *   x    = the float32 observation step() returns: U (M), then X (J), then for each link with L > 0 its pipeline, oldest
 *          first (:334-413); at t = 0 the reset observation
 *   h_l, y = exactly the serial env's contract (orgym_mlp_t above): acc = b, then fmaf ascending in k; accurate tanhf
 *          or NaN-keeping ReLU; no activation after the last Linear
 *   a_i  = NaN if y_i is NaN, else min(max(y_i, 0f), action_high[i])   (SB3 predict's np.clip to the Box, float32)
 * a then takes the env's own action rule, exactly like an ORGYM_NET_POLICY_ACTIONS action: rint((double)a), then
 * max(., 0), so a NaN action orders 0; action_traj_dev records a.  Results are a pure function of (weights, seed, global
 * env id, episode): independent of batch size and env_offset sharding.  MLP rollouts always run the ahead-of-time kernel,
 * whatever ORGYM_NET_JIT says (also under ORGYM_NET_JIT=2). */

typedef struct {
    int32_t policy;
    const float* actions_dev; /* ACTIONS: (e,t,i) at [e*stride_env + t*stride_t + i]; CONSTANT: float32[E] */
    int64_t act_stride_env, act_stride_t;
    const double* demand_dev; /* (e,t,r) at [e*stride_env + t*stride_t + r] or NULL */
    int64_t dem_stride_env, dem_stride_t;
    /* HOST pointers, read at the call only when policy == ORGYM_NET_POLICY_MLP.  mlp: ORGYM_E_INVALID for a missing or
     * malformed network (layer count, widths outside 1..ORGYM_MLP_MAX_WIDTH, width[0] != obs_dim, width[num_layers] !=
     * E, null weights); ORGYM_E_UNSUPPORTED, with the sizes in the message, when the weights, activations, observation
     * and action tiles and work vectors of one CTA do not fit in shared memory even for 32 envs.  action_high:
     * float32[E], the upper bound of the action Box (single_action_space.high); ORGYM_E_INVALID when NULL. */
    const orgym_mlp_t* mlp;
    const float* action_high;
} orgym_netinv_rollout_in_t;

typedef struct {
    double* ep_return_dev;   /* [N] */
    double* stats_dev;       /* [N,4]: sum retail sales, sum demand, sum unfulfilled (end-of-period backlog), sum_t sum_j max(0,X_j) */
    double* reward_traj_dev; /* [N,T] */
    double* final_X_dev;     /* [N,J] */
    double* final_Y_dev;     /* [N,E] */
    double* final_U_dev;     /* [N,M] */
    double* summary_dev;     /* [8] */
    float* action_traj_dev;  /* [N,T,E] actions the policy took; ORGYM_NET_POLICY_MLP only (ORGYM_E_INVALID otherwise) */
} orgym_netinv_rollout_out_t;

/* fused reset + num_periods steps; scratch_dev holds the per-env lead-time rings while the rollout runs
 * (orgym_netinv_state_bytes() bytes are enough). */
int orgym_netinv_rollout(orgym_handle_t h, void* scratch_dev, uint64_t seed, int64_t env_offset, uint32_t episode,
                         const orgym_netinv_rollout_in_t* in, const orgym_netinv_rollout_out_t* out, void* stream);

/* The network kernels are specialised per topology at create time: the flattened graph is emitted as straight-line
 * CUDA source and compiled for sm_100a with NVRTC (fallback: a generic kernel that reads the topology from the
 * constant bank; automatic up to 128 reorder links, ORGYM_NET_JIT=0 forces the generic kernel, =1 specialises any
 * size, =2 additionally makes a failed specialisation an error; cubins are cached under $ORGYM_JIT_CACHE or
 * ~/.cache/orgym_b200).  This entry point returns
 * that source for inspection and, with compile_check != 0, runs it through NVRTC; it needs no GPU. */
int orgym_netinv_codegen(const orgym_netinv_config_t* cfg, int compile_check, char* buf, int64_t buflen,
                         int64_t* needed);
/* 1 if this handle runs the topology-specialised kernels, 0 if it runs the generic one */
int orgym_netinv_is_specialised(orgym_handle_t h);

/* ------------------------------------------------------------------------- *
 * shared helpers
 * ------------------------------------------------------------------------- */
/* sticky device error bits of a handle (ORGYM_ERR_*); synchronises `stream`; clears them when clear != 0 */
int orgym_errors(orgym_handle_t h, uint32_t* bits_out, int clear, void* stream);

/* K6: draw count samples per distribution instance for the statistical tests:
 * out_dev[i] = sample of `dist` for (seed, env = env_offset + i / per_env, period = i % per_env). */
int orgym_sample_demand(const orgym_dist_t* dist, uint64_t seed, int64_t env_offset, int64_t num_envs,
                        int32_t per_env, int device, int64_t* out_dev, void* stream);
/* general Poisson sampler with a per-element mean (the Newsvendor path): out_dev[i] ~ Poisson(mu_dev[i]) */
int orgym_sample_poisson_mu(const double* mu_dev, uint64_t seed, int64_t env_offset, int64_t count, int32_t period,
                            int device, int64_t* out_dev, void* stream);

/* ------------------------------------------------------------------------- *
 * Evaluation report: the summary row of process_and_report_results
 * (benchmark_InvManagementBacklogEnv.py:493-504, benchmark_NetInvMgmtBacklogEnv.py:320-330) for one batch of
 * episodes, computed on the device from the per-episode outputs of a rollout -- exact order statistics by radix
 * select, two-pass variance, sums reduced in a fixed order (bitwise reproducible).  Nothing synchronises the host.
 *   ep_return_dev  float64[n] episode returns (TotalReward)
 *   stats_dev      [n,4] (sales, demand, unfulfilled / lost, on-hand sum) as int64 (stats_kind 0), int32 (1) or
 *                  float64 (2); NULL = reward columns only
 *   scratch_dev    orgym_report_scratch_bytes(n) bytes, 256-byte aligned
 *   report_dev     float64[ORGYM_REPORT_LEN]: [0] episodes, [1] mean, [2] median (pandas: midpoint of the two central
 *                  order statistics), [3] std (ddof = 1), [4] min, [5] max of the returns, [6] mean service level
 *                  sales/demand (1.0 for an episode without demand, :425), [7] mean unfulfilled quantity, [8] mean of
 *                  on-hand sum / periods, [9] sum of returns, [10] sum of squared deviations, [11] candidates the
 *                  select kept after its second pass (diagnostic)
 * ------------------------------------------------------------------------- */
#define ORGYM_REPORT_LEN 16
int64_t orgym_report_scratch_bytes(int64_t num_episodes);
int orgym_evaluation_report(int device, const double* ep_return_dev, const void* stats_dev, int stats_kind,
                            int64_t num_episodes, int32_t periods, void* scratch_dev, double* report_dev, void* stream);

/* device timing of the most recent rollout/step launch of this handle is not part of the ABI:
 * time with CUDA events on `stream`. */

#ifdef __cplusplus
}
#endif
#endif /* ORGYM_B200_H */
