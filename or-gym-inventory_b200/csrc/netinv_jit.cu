// netinv_jit.cu -- network env: the topology compiled into the instruction stream.
//
// The generic kernel (netinv.cu) interprets the flattened graph from the constant bank: every link / node visit
// pays for index loads, address arithmetic and loop control (ncu: ~3200 warp-instructions per warp-step on the
// default 9-node graph, most of them bookkeeping).  Here the same period (network_management.py:436-635) is emitted as
// straight-line CUDA source for ONE topology -- literal link / node indices, literal prices and lead times, per-
// instance state in registers -- compiled for sm_100a with NVRTC when the env is created.  Evaluation order of every
// floating-point expression is exactly the generic kernel's (= the reference's); the parity tests run both.
#include <algorithm>
#include <cstdarg>
#include <vector>

#include "netinv.cuh"
#include "netinv_args.cuh"

namespace {
struct Src {
    std::string s;
    void operator()(const char* fmt, ...) {
        char buf[2048];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        s += buf;
        s += '\n';
    }
};
// exact double literal (hexadecimal floating constant, C++17)
std::string lit(double v) {
    char buf[64];
    if (v == 0.0) return "0.0";
    snprintf(buf, sizeof(buf), "%a", v);
    return buf;
}
// One allocation step of supplier s (network_management.py:459-485): what its on-hand inventory x leaves after the
// consumption `cons` of its earlier links, capped by a factory's capacity, fills the request `req` into f.  `head`
// starts the first line, `ind` indents the others.
void emit_alloc(Src& o, const NetDev& P, int s, const std::string& head, const std::string& ind, const std::string& x,
                const std::string& cons, const std::string& f) {
    o("%sdouble avail = %s - %s; avail = avail > 0.0 ? avail : 0.0; double oa = avail;", head.c_str(), x.c_str(), cons.c_str());
    if (P.is_factory[s])
        o("%s{ double mp = %s * avail; double lim = mp < %s ? mp : %s; oa = lim < oa ? lim : oa; }", ind.c_str(),
          lit(P.v[s]).c_str(), lit(P.C[s]).c_str(), lit(P.C[s]).c_str());
    o("%s%s = oa < req ? oa : req;", ind.c_str(), f.c_str());
}
// what the fill f of one of its links takes from supplier s: f / v (x / 1.0 == x, so yield 1 divides by nothing)
std::string consumed(const NetDev& P, int s, const std::string& f) { return P.v[s] == 1.0 ? f : f + " / " + lit(P.v[s]); }
// ring commit of the streaming kernel: `v` goes into the ring slot `slot` and into its float32 copy
std::string ring_commit(const NetDev& P, const std::string& slot, const std::string& v) {
    return "*" + slot + " = " + v + ";" + (P.ring32 ? " r32[" + slot + " - ring] = (float)" + v + ";" : "");
}
void emit_step_stream(Src& o, const NetDev& P, const NetPlan& plan, int min_blocks);
}  // namespace

std::string net_jit_source(const NetDev& P, const NetPlan& plan) {
    const int J = P.J, E = P.E, M = P.M;
    Src o;
    o.s += orgym_jit_device_rng_src();
    o.s += orgym_jit_net_args_src();
    o("#define NTHR %d", NET_JIT_THREADS);
    o("#define NJ %d\n#define NE %d\n#define NM %d\n#define NOBS %d\n#define NSUML %d\n#define NT %d", J, E, M, P.obs_dim,
      P.sumL, P.T);
    o("#define OSTRIDE %d", P.obs_dim | 1);
    // state tiles (netinv.cuh): NP instances per tile, slot stride NP, so every state access is base + constant
    o("#define NP %d\n#define TILE_BYTES %lldLL", NET_TILE, (long long)net_tile_bytes(P));
    // ---- observation writer (:334-413)
    o("// order request of one link: round half to even, negative -> 0 (network_management.py:449)");
    o("__device__ __forceinline__ double net_reqf(float a) { const double q = rint((double)a); return q > 0.0 ? q : 0.0; }");
    o("__device__ __forceinline__ double net_req(const float* a) { return net_reqf(__ldg(a)); }");
    o("__device__ __forceinline__ void write_obs(const double (&X)[NJ > 0 ? NJ : 1], const double (&U)[NM > 0 ? NM : 1],");
    o("    const double* __restrict__ ring, int el, int t, float* o) {");
    for (int r = 0; r < M; r++) o("  o[%d] = (float)U[%d];", r, r);
    for (int j = 0; j < J; j++) o("  o[%d] = (float)X[%d];", M + j, j);
    {
        int k = M + J;
        for (int i = 0; i < E; i++) {
            const int L = P.L[i];
            if (L == 0) continue;
            o("  { const int s0 = t %% %d; const double* b = ring + %d * NP + el;", L, P.roff[i]);
            o("    double v[%d];", L);
            o("    _Pragma(\"unroll\") for (int q = 0; q < %d; q++) { int sl = s0 + q; sl = sl >= %d ? sl - %d : sl; v[q] = b[sl * NP]; }",
              L, L, L);
            o("    _Pragma(\"unroll\") for (int q = 0; q < %d; q++) o[%d + q] = (float)v[q]; }", L, k);
            k += L;
        }
    }
    o("}");
    // ---- kernels: the same period body is emitted twice, with the mode fixed at compile time.  STEP is bound by HBM
    // latency and wants many resident warps (<= 102 registers -> 5 CTAs/SM); ROLLOUT is issue-bound and wants no spills.
    auto emit_kernel = [&](const char* kname, int rollout, int min_blocks) {
    o("#define ROLL %d", rollout);
    o("extern \"C\" __global__ void __launch_bounds__(NTHR, %d) %s(const NetSimArgs A, const double* __restrict__ disc,", min_blocks, kname);
    o("    const AliasDev* __restrict__ dem) {");
    o("  extern __shared__ __align__(16) unsigned char smem[];");
    o("  float* otile = (float*)smem;");
    o("  const int tid = threadIdx.x;");
    o("  const long long e0 = (long long)blockIdx.x * NTHR, e = e0 + tid;");
    o("  const bool valid = e < A.N;");
    o("  const long long ec = valid ? e : 0;");
    o("  const int el = (int)(ec %% NP);");
    o("  char* sb = (char*)A.state + (ec / NP) * TILE_BYTES;");
    o("  unsigned long long* s_key = (unsigned long long*)sb;");
    o("  double* s_X = (double*)(sb + 8 * NP); double* s_Y = s_X + NJ * NP; double* s_U = s_Y + NE * NP;");
    o("  double* ring = s_U + NM * NP;");
    o("  int* s_period = (int*)(ring + NSUML * NP); unsigned int* s_episode = (unsigned int*)(s_period + NP);");
    o("  double X[NJ > 0 ? NJ : 1], Y[NE > 0 ? NE : 1], U[NM > 0 ? NM : 1], R[NE > 0 ? NE : 1], S[NM > 0 ? NM : 1], Cn[NJ > 0 ? NJ : 1];");
    o("  unsigned long long key; unsigned int episode; int t0, t1; bool do_step = valid;");
    o("  float* orow = A.use_tile ? otile + tid * OSTRIDE : (A.obs ? A.obs + ec * NOBS : (float*)0);");
    // initial state literals
    auto emit_reset_regs = [&](const char* ind) {
        for (int j = 0; j < J; j++) o("%sX[%d] = %s;", ind, j, lit(P.I0[j]).c_str());
        for (int i = 0; i < E; i++) o("%sY[%d] = 0.0;", ind, i);
        for (int r = 0; r < M; r++) o("%sU[%d] = 0.0;", ind, r);
    };
    auto emit_reset_state = [&](const char* ind) {
        for (int j = 0; j < J; j++) o("%ss_X[%d * NP + el] = %s;", ind, j, lit(P.I0[j]).c_str());
        o("%sfor (int i = 0; i < NE; i++) s_Y[i * NP + el] = 0.0;", ind);
        o("%sfor (int r = 0; r < NM; r++) s_U[r * NP + el] = 0.0;", ind);
        o("%sfor (int k = 0; k < NSUML; k++) ring[k * NP + el] = 0.0;", ind);
        o("%ss_period[el] = 0;", ind);
    };
    o("  if (ROLL) {");
    o("    key = A.seed + (unsigned long long)(A.env_offset + e); episode = A.episode; t0 = 0; t1 = NT;");
    emit_reset_regs("    ");
    o("    if (valid) for (int k = 0; k < NSUML; k++) ring[k * NP + el] = 0.0;");
    o("  } else {");
    o("    key = s_key[el]; episode = s_episode[el]; t0 = s_period[el]; t1 = t0 + 1;");
    o("    if (valid && t0 >= NT) {");
    o("      do_step = false;");
    o("      if (A.autoreset == ORGYM_AUTORESET_NEXT_STEP) {");
    emit_reset_state("        ");
    emit_reset_regs("        ");
    o("        s_episode[el] = episode + 1;");
    o("        write_obs(X, U, ring, el, 0, orow);");
    o("        A.reward[e] = 0.0; A.terminated[e] = 0; A.truncated[e] = 0;");
    o("      } else {");
    o("        atomicOr(A.err, ORGYM_ERR_STEP_PAST_END);");
    o("        if (A.use_tile) for (int z = 0; z < NOBS; z++) orow[z] = A.obs[e * NOBS + z];");
    o("        A.reward[e] = 0.0; A.terminated[e] = 0; A.truncated[e] = 1;");
    o("      }");
    o("    }");
    o("    if (do_step) {");
    for (int j = 0; j < J; j++) o("      X[%d] = s_X[%d * NP + el];", j, j);
    for (int i = 0; i < E; i++) o("      Y[%d] = s_Y[%d * NP + el];", i, i);
    for (int r = 0; r < M; r++) o("      U[%d] = s_U[%d * NP + el];", r, r);
    o("    }");
    o("  }");
    o("  double ret = 0.0, s_sales = 0.0, s_dem = 0.0, s_unf = 0.0, s_inv = 0.0, last_reward = 0.0;");
    o("  if (!ROLL && !do_step) t1 = t0;");
    o("  for (int t = t0; t < t1; t++) {");
    // arrivals: all ring loads up front (independent -> overlapped)
    for (int i = 0; i < E; i++)
        if (P.L[i] > 0) {
            o("    const long long sl%d = (%d + t %% %d) * NP + el;", i, P.roff[i], P.L[i]);
            o("    const double Ar%d = ring[sl%d];", i, i);
        }
    o("    const float* arow = A.policy == ORGYM_NET_POLICY_CONSTANT ? A.actions : A.actions + ec * A.a_se + (long long)(ROLL ? t : 0) * A.a_st;");
    // 0) orders (:448-490)
    for (int j = 0; j < J; j++) o("    Cn[%d] = 0.0;", j);
    o("    double cons = 0.0;");
    for (int i = 0; i < E; i++) {
        const int s = P.sup[i];
        o("    { double req = rint((double)arow[%d]); req = req > 0.0 ? req : 0.0;", i);
        if (s == -1)
            o("      R[%d] = req; }", i);
        else if (s < 0)
            o("      R[%d] = 0.0; (void)req; }", i);
        else {
            if (i == 0 || P.sup[i - 1] != s) o("      cons = 0.0;");
            emit_alloc(o, P, s, "      ", "      ", "X[" + std::to_string(s) + "]", "cons", "double f");
            o("      cons += %s;", consumed(P, s, "f").c_str());
            o("      R[%d] = f;", i);
            if (i == E - 1 || P.sup[i + 1] != s) o("      Cn[%d] = cons;", s);
            o("    }");
        }
    }
    // on-hand (:516-528)
    for (int j = 0; j < J; j++) {
        o("    { double arr = 0.0;");
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
            const int i = P.pred_idx[z];
            if (P.L[i] == 0)
                o("      arr += R[%d];", i);
            else
                o("      arr += Ar%d;", i);
        }
        o("      X[%d] = (X[%d] + arr) - Cn[%d]; }", j, j, j);
    }
    // 1) pipeline (:494-511) + ring commit
    for (int i = 0; i < E; i++) {
        if (P.L[i] == 0)
            o("    Y[%d] = (Y[%d] - R[%d]) + R[%d];", i, i, i, i);
        else {
            o("    Y[%d] = (Y[%d] - Ar%d) + R[%d];", i, i, i, i);
            o("    if (valid) ring[sl%d] = R[%d];", i, i);
        }
    }
    // 2-4) market (:536-566)
    for (int r = 0; r < M; r++) {
        const int j = P.rt_node[r];
        o("    { double d;");
        o("      if (A.demand) d = rint(A.demand[ec * A.d_se + (long long)(ROLL ? t : 0) * A.d_st + %d]);", r);
        o("      else d = (double)sample_fixed(dem[%d], dem[%d].table, key, episode, t, %du);", r, r, r);
        o("      d = d > 0.0 ? d : 0.0;");
        o("      double fill = d + U[%d]; double x = X[%d]; double invr = x > 0.0 ? x : 0.0;", r, j);
        o("      double sl = invr < fill ? invr : fill; S[%d] = sl; X[%d] = x - sl; double un = fill - sl;", r, j);
        o("      U[%d] = %s; s_sales += sl; s_dem += d; s_unf += %s;", r, P.backlog ? "un" : "0.0", P.backlog ? "un" : "0.0");
        o("      if (!ROLL && A.info_demand && do_step) A.info_demand[NET_IIDX(A, e, NM, %d)] = d; }", r);
    }
    // 5) profit (:578-613)
    o("    double total = 0.0;");
    for (int j = 0; j < J; j++) {
        o("    { double SR = 0.0, PC = 0.0, HCp = 0.0, sold = 0.0, UP = 0.0;");
        for (int z = P.succ_ptr[j]; z < P.succ_ptr[j + 1]; z++) {
            const int l = P.succ_idx[z];
            if (l < E) {
                o("      SR += %s * R[%d]; sold += R[%d];", lit(P.p[l]).c_str(), l, l);
            } else {
                const int r = l - E;
                if (P.is_retail[j]) o("      UP += %s * U[%d];", lit(P.rt_b[r]).c_str(), r);
                o("      SR += %s * S[%d]; sold += S[%d];", lit(P.rt_p[r]).c_str(), r, r);
            }
        }
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
            const int i = P.pred_idx[z];
            o("      PC += %s * R[%d]; { double y = Y[%d]; HCp += %s * (y > 0.0 ? y : 0.0); }", lit(P.p[i]).c_str(), i, i,
              lit(P.g[i]).c_str());
        }
        o("      double x = X[%d]; double xp = x > 0.0 ? x : 0.0; double HC = %s * xp + HCp; double OC = 0.0;", j, lit(P.h[j]).c_str());
        if (P.is_factory[j]) {
            if (!(P.v[j] > 0.0))
                o("      OC = 0.0;");
            else if (P.v[j] == 1.0)
                o("      OC = %s * sold;", lit(P.o[j]).c_str());
            else
                o("      OC = %s * (sold / %s);", lit(P.o[j]).c_str(), lit(P.v[j]).c_str());
        }
        o("      (void)sold; double pj = (((SR - PC) - OC) - HC) - UP; total += pj; s_inv += xp;");
        o("      if (!ROLL && A.info_profit && do_step) A.info_profit[NET_IIDX(A, e, NJ, %d)] = pj; }", j);
    }
    o("    last_reward = disc[t] * total; ret += last_reward;");
    o("    if (ROLL && A.reward_traj && valid) A.reward_traj[e * NT + t] = last_reward;");
    o("    if (!ROLL && do_step) {");
    o("      if (A.info_profit_total) A.info_profit_total[e] = total;");
    o("      if (A.info_sales) {");
    for (int i = 0; i < E; i++) o("        A.info_sales[NET_IIDX(A, e, NE + NM, %d)] = R[%d];", i, i);
    for (int r = 0; r < M; r++) o("        A.info_sales[NET_IIDX(A, e, NE + NM, %d)] = S[%d];", E + r, r);
    o("      }");
    o("    }");
    o("  }");  // t loop
    // ---- epilogue: ROLLOUT
    o("  if (ROLL) {");
    o("    if (valid) {");
    o("      if (A.ep_return) A.ep_return[e] = ret;");
    o("      if (A.stats) { A.stats[e * 4 + 0] = s_sales; A.stats[e * 4 + 1] = s_dem; A.stats[e * 4 + 2] = s_unf; A.stats[e * 4 + 3] = s_inv; }");
    o("      if (A.final_X) {");
    for (int j = 0; j < J; j++) o("        A.final_X[e * NJ + %d] = X[%d];", j, j);
    o("      }\n      if (A.final_Y) {");
    for (int i = 0; i < E; i++) o("        A.final_Y[e * NE + %d] = Y[%d];", i, i);
    o("      }\n      if (A.final_U) {");
    for (int r = 0; r < M; r++) o("        A.final_U[e * NM + %d] = U[%d];", r, r);
    o("      }");
    o("    }");
    o("    if (A.partials) {");
    o("      double v[7] = {valid ? 1.0 : 0.0, valid ? ret : 0.0, valid ? ret * ret : 0.0, valid ? s_sales : 0.0, valid ? s_dem : 0.0, valid ? s_unf : 0.0, valid ? s_inv : 0.0};");
    o("      __shared__ double red[NTHR / 32][7];");
    o("      _Pragma(\"unroll\") for (int z = 0; z < 7; z++) { double x = v[z];");
    o("        _Pragma(\"unroll\") for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);");
    o("        if ((tid & 31) == 0) red[tid >> 5][z] = x; }");
    o("      __syncthreads();");
    o("      if (tid < 7) { double x = 0.0; for (int wv = 0; wv < NTHR / 32; wv++) x += red[wv][tid]; A.partials[(long long)blockIdx.x * 8 + tid] = x; }");
    o("    }");
    o("    return;");
    o("  }");
    // ---- epilogue: STEP
    o("  if (do_step) {");
    o("    const int tn = t0 + 1; const bool trunc = tn >= NT;");
    o("    const bool reset_now = trunc && A.autoreset == ORGYM_AUTORESET_SAME_STEP;");
    o("    if (!reset_now) {");
    for (int j = 0; j < J; j++) o("      s_X[%d * NP + el] = X[%d];", j, j);
    for (int i = 0; i < E; i++) o("      s_Y[%d * NP + el] = Y[%d];", i, i);
    for (int r = 0; r < M; r++) o("      s_U[%d * NP + el] = U[%d];", r, r);
    o("      s_period[el] = tn;");
    o("      write_obs(X, U, ring, el, tn, orow);");
    o("    } else {");
    o("      if (A.final_obs) write_obs(X, U, ring, el, tn, A.final_obs + e * NOBS);");
    emit_reset_state("      ");
    emit_reset_regs("      ");
    o("      s_episode[el] = episode + 1;");
    o("      write_obs(X, U, ring, el, 0, orow);");
    o("    }");
    o("    A.reward[e] = last_reward; A.terminated[e] = 0; A.truncated[e] = trunc ? 1 : 0;");
    o("  }");
    o("  if (A.use_tile) {");
    o("    __syncthreads();");
    o("    const int nvalid = (int)((A.N - e0) < NTHR ? (A.N - e0) : NTHR);");
    o("    const int total = nvalid * NOBS;");
    o("    float* g = A.obs + e0 * NOBS;");
    o("    for (int i = tid; i < total; i += NTHR) { const int r = i / NOBS, c = i - r * NOBS; __stcs(g + i, otile[r * OSTRIDE + c]); }");
    o("  }");
    o("}");
    o("#undef ROLL");
    };
    // small graphs: STEP 5 CTAs/SM (<= 102 registers), ROLLOUT 3; large graphs (hundreds of live float64 values per
    // instance) spill either way and run best with all 255 registers (measured on the 64-node synthetic graph)
    const bool big = net_large_graph(P);
    if (plan.stream)  // large graphs: state stays in HBM, coalesced 32-column tiles
        // 64 registers per thread: a launch of 2^17 instances is 28 warps per SM, so with 8 CTAs of 128 threads per SM the
        // whole batch is resident in one wave (measured on the 64-node graph: 0.470 vs 0.486 ms for the step pair at 128
        // registers)
        emit_step_stream(o, P, plan, 8);
    else
        emit_kernel("net_jit_step", 0, big ? 2 : 5);
    emit_kernel("net_jit_rollout", 1, big ? 1 : 3);
    o("// step_kernel_kind=%s", plan.stream ? "stream" : "register");
    return o.s;
}


// ---- streaming STEP kernel for large graphs --------------------------------------------------------------------------------
// With hundreds of float64 values per instance the register-resident kernel above spills and runs at 2 CTAs/SM.  In
// STEP mode the state lives in HBM anyway, so this variant never keeps it in registers: pass A walks the sorted links,
// allocates orders and parks R_t / consumed in a per-instance scratch area of the state buffer; pass B walks the main
// nodes, and for each one loads exactly what it needs (its X, consumed, the arrivals / pipeline entries of its
// predecessor links, the backlog of its market links, the R_t of its successor links), updates state in place and
// finishes the node's profit; pass C rebuilds the observation from the final state.  Same operations in the same
// order as the other kernels; few live registers -> many resident warps -> the loads overlap.  The row-major action
// and observation blocks move through 32-column shared-memory tiles, so every global access is coalesced whatever
// the observation length.
namespace {
void emit_step_stream(Src& o, const NetDev& P, const NetPlan& plan, int min_blocks) {
    const int J = P.J, E = P.E, M = P.M, W = P.obs_dim;
    auto emit_reset = [&](const char* ind) {  // the instance's initial state, stored to its tile
        for (int j = 0; j < J; j++) o("%ss_X[%d * NP + el] = %s;", ind, j, lit(P.I0[j]).c_str());
        o("%sfor (int i = 0; i < NE; i++) s_Y[i * NP + el] = 0.0;", ind);
        o("%sfor (int r = 0; r < NM; r++) s_U[r * NP + el] = 0.0;", ind);
        o("%sfor (int k = 0; k < NSUML; k++) ring[k * NP + el] = 0.0;", ind);
        if (P.ring32) o("%sfor (int k = 0; k < NSUML; k++) r32[k * NP + el] = 0.0f;", ind);
        o("%ss_period[el] = 0; s_episode[el] = episode + 1;", ind);
    };
    o("extern \"C\" __global__ void __launch_bounds__(NTHR, %d) net_jit_step(const NetSimArgs A, const double* __restrict__ disc,", min_blocks);
    o("    const AliasDev* __restrict__ dem) {");
    o("  extern __shared__ __align__(16) unsigned char smem_raw[];");
    o("  float* tile = (float*)smem_raw;   // [NTHR][33] 32-column staging tile (+1 padding column: conflict-free)");
    o("  const int tid = threadIdx.x;");
    o("  const long long e0 = (long long)blockIdx.x * NTHR, e = e0 + tid;");
    o("  const int nvalid = (int)((A.N - e0) < NTHR ? (A.N - e0) : NTHR);");
    o("  const bool valid = tid < nvalid;");
    o("  const long long ec = valid ? e : 0;");
    o("  const int el = (int)(ec %% NP);");
    o("  char* sb = (char*)A.state + (ec / NP) * TILE_BYTES;");
    o("  unsigned long long* s_key = (unsigned long long*)sb;");
    o("  double* s_X = (double*)(sb + 8 * NP); double* s_Y = s_X + NJ * NP; double* s_U = s_Y + NE * NP;");
    o("  double* ring = s_U + NM * NP;");
    o("  int* s_period = (int*)(ring + NSUML * NP); unsigned int* s_episode = (unsigned int*)(s_period + NP);");
    o("  double* sc_R = (double*)(s_episode + NP); double* sc_C = sc_R + NE * NP;");
    if (P.ring32) o("  float* const r32 = (float*)(sc_C + NJ * NP);   // float32 copy of the rings, read by net_obs_kernel");
    o("  float* trow = tile + tid * 33;");
    // every warp transposes the 32 rows of its own lanes: the staging tile needs warp-level synchronisation only,
    // so the warps of a CTA drift apart and cover each other's memory latency
    o("  const int ln = tid & 31, wrow0 = tid & ~31, wrow1 = nvalid < wrow0 + 32 ? (nvalid > wrow0 ? nvalid : wrow0) : wrow0 + 32;");
    o("  bool do_step = valid;");
    o("  int t = 0; unsigned int episode = 0; unsigned long long key = 0;");
    o("  if (valid) {");
    o("    t = s_period[el]; episode = s_episode[el]; key = s_key[el];");
    o("    if (t >= NT) {");
    o("      do_step = false;");
    o("      if (A.autoreset == ORGYM_AUTORESET_NEXT_STEP) {");
    emit_reset("        ");
    o("        A.reward[e] = 0.0; A.terminated[e] = 0; A.truncated[e] = 0;");
    o("      } else {");
    o("        atomicOr(A.err, ORGYM_ERR_STEP_PAST_END);");
    o("        A.reward[e] = 0.0; A.terminated[e] = 0; A.truncated[e] = 1;");
    o("      }");
    o("    }");
    o("  }");
    // Visit of main node j once the R_t of its links are known, the same in both forms: arrivals, pipeline update and
    // ring commit of its inbound links, its on-hand inventory less the consumption `cons`, its market links, its
    // profit.  In scope: the loaded rows x<j>, y<i>, ar<i>, u<r>, the ring slots slot<i> and R_t rt<i> of its inbound
    // links, and the R_t of each outbound link l as <succ><l>.
    auto emit_visit = [&](int j, const std::string& cons, const std::string& succ) {
        o("      { double arr = 0.0, PC = 0.0, HCp = 0.0;");
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
            const int i = P.pred_idx[z];
            if (P.L[i] == 0)
                o("        { const double ar = rt%d;", i);
            else
                o("        { const double ar = ar%d; %s", i,
                  ring_commit(P, "slot" + std::to_string(i), "rt" + std::to_string(i)).c_str());
            o("          arr += ar; const double yn = (y%d - ar) + rt%d; s_Y[%d * NP + el] = yn;", i, i, i);
            o("          PC += %s * rt%d; HCp += %s * (yn > 0.0 ? yn : 0.0); }", lit(P.p[i]).c_str(), i, lit(P.g[i]).c_str());
        }
        o("        double x = (x%d + arr) - %s;", j, cons.c_str());
        o("        double SR = 0.0, sold = 0.0, UP = 0.0;");
        for (int r = 0; r < M; r++) {
            if (P.rt_node[r] != j) continue;
            o("        double S%d, U%d;", r, r);
            o("        { double d;");
            o("          if (A.demand) d = rint(A.demand[e * A.d_se + %d]);", r);
            o("          else d = (double)sample_fixed(dem[%d], dem[%d].table, key, episode, t, %du);", r, r, r);
            o("          d = d > 0.0 ? d : 0.0;");
            o("          const double fill = d + u%d; const double invr = x > 0.0 ? x : 0.0;", r);
            o("          S%d = invr < fill ? invr : fill; x = x - S%d; const double un = fill - S%d; U%d = %s;", r, r, r, r,
              P.backlog ? "un" : "0.0");
            o("          s_U[%d * NP + el] = U%d;", r, r);
            o("          if (A.info_demand) A.info_demand[NET_IIDX(A, e, NM, %d)] = d;", r);
            o("          if (A.info_sales) A.info_sales[NET_IIDX(A, e, NE + NM, %d)] = S%d; }", E + r, r);
        }
        o("        s_X[%d * NP + el] = x;", j);
        for (int z = P.succ_ptr[j]; z < P.succ_ptr[j + 1]; z++) {
            const int l = P.succ_idx[z];
            if (l < E)
                o("        SR += %s * %s%d; sold += %s%d;", lit(P.p[l]).c_str(), succ.c_str(), l, succ.c_str(), l);
            else {
                const int r = l - E;
                if (P.is_retail[j]) o("        UP += %s * U%d;", lit(P.rt_b[r]).c_str(), r);
                o("        SR += %s * S%d; sold += S%d;", lit(P.rt_p[r]).c_str(), r, r);
            }
        }
        o("        const double xp = x > 0.0 ? x : 0.0; const double HC = %s * xp + HCp; double OC = 0.0;", lit(P.h[j]).c_str());
        if (P.is_factory[j]) {
            if (!(P.v[j] > 0.0))
                o("        OC = 0.0;");
            else if (P.v[j] == 1.0)
                o("        OC = %s * sold;", lit(P.o[j]).c_str());
            else
                o("        OC = %s * (sold / %s);", lit(P.o[j]).c_str(), lit(P.v[j]).c_str());
        }
        o("        (void)sold; const double pj = (((SR - PC) - OC) - HC) - UP; total += pj;");
        o("        if (A.info_profit) A.info_profit[NET_IIDX(A, e, NJ, %d)] = pj; }", j);
    };
    std::vector<int> has_pur(E, 0);  // the link's purchaser holds inventory (it is visited with that node)
    for (int j = 0; j < J; j++)
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) has_pur[P.pred_idx[z]] = 1;
    o("  // stream_form=%s", plan.onepass ? "onepass" : "twopass");
    if (plan.onepass) {
        // ---- single pass over the main nodes.  The two-pass form below parks every R_t and every supplier's consumption in
        // scratch rows of the state tile between its passes: with the whole batch resident that is 1 KB per instance
        // written and read back through DRAM (the scratch of 2^17 instances exceeds the L2).  Here a node recomputes what
        // it needs instead: the allocation of a supplier is a function of that supplier's start-of-period inventory and
        // the requests on its own links, so purchaser j re-runs the supplier's allocation chain up to its link (same
        // operations, same order -> the same float64 R_t), and a supplier runs its whole chain for its sales and
        // consumption.  Suppliers follow their purchasers in node order, so their X row still holds X[t].  Requests are
        // read per lane from the row-major action tensor (a lane's row is 4*E bytes, L1-resident between uses).
        std::vector<int> seg0(J, -1), seg1(J, -1);
        for (int i = 0; i < E; i++)
            if (P.sup[i] >= 0) {
                if (seg0[P.sup[i]] < 0) seg0[P.sup[i]] = i;
                seg1[P.sup[i]] = i;
            }
        o("  const float* const arow = A.actions + ec * NE;");
        o("#define REQ(i) net_req(arow + (i))");
        // allocation chain of supplier s from its first link to link i1; f of link i lands in variable <pfx><i>
        auto emit_chain = [&](int s, int i1, const std::string& xvar, const std::string& pfx, const std::string& ind,
                              bool keep_cons) {
            o("%sdouble cons_%s = 0.0;", ind.c_str(), pfx.c_str());
            for (int i = seg0[s]; i <= i1; i++) {
                const std::string f = pfx + std::to_string(i);
                o("%sdouble %s;", ind.c_str(), f.c_str());
                emit_alloc(o, P, s, ind + "{ const double req = rq" + std::to_string(i) + "; ", ind + "  ", xvar, "cons_" + pfx, f);
                if (i < i1 || keep_cons)
                    o("%s  cons_%s += %s; }", ind.c_str(), pfx.c_str(), consumed(P, s, f).c_str());
                else
                    o("%s  }", ind.c_str());
            }
        };
        auto emit_rt = [&](int i, const std::string& xvar, const char* ind) {  // declares rt<i>
            const int s = P.sup[i];
            if (s == -1)
                o("%sconst double rt%d = rq%d;", ind, i, i);
            else if (s < 0)
                o("%sconst double rt%d = 0.0;", ind, i);
            else {
                emit_chain(s, i, xvar, "g" + std::to_string(i) + "_", ind, false);
                o("%sconst double rt%d = g%d_%d;", ind, i, i, i);
            }
            o("%sif (A.info_sales) A.info_sales[NET_IIDX(A, e, NE + NM, %d)] = rt%d;", ind, i, i);
        };
        auto req_links = [&](int i) {  // links whose request the R_t of link i depends on
            std::vector<int> v;
            const int s = P.sup[i];
            if (s == -1)
                v.push_back(i);
            else if (s >= 0)
                for (int l = seg0[s]; l <= i; l++) v.push_back(l);
            return v;
        };
        // Loads of a node: float64 state rows (name, address) and the requests (links) it needs.  (Issuing the loads of
        // node j + 1 as asynchronous global->shared copies -- cp.async, 8- and 4-byte pieces into a two-stage per-lane
        // landing zone -- before node j is computed was measured at 0.54 ms against 0.42 ms for the step pair: small
        // cp.async copies are slow, and the 28 KB landing zone per CTA costs the L1 that holds the action rows.)
        struct NodeLd {
            std::vector<std::pair<std::string, std::string>> d8;
            std::vector<int> acts;
        };
        std::vector<NodeLd> nld((size_t)J);
        for (int j = 0; j < J; j++) {
            NodeLd& n = nld[(size_t)j];
            char nb[64], ab[96];
            snprintf(nb, sizeof(nb), "x%d", j);
            snprintf(ab, sizeof(ab), "s_X + %d * NP + el", j);
            n.d8.push_back({nb, ab});
            std::vector<char> need((size_t)E, 0);
            for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
                const int i = P.pred_idx[z], L = P.L[i], sp = P.sup[i];
                if (sp >= 0) {
                    snprintf(nb, sizeof(nb), "xq%d", i);
                    snprintf(ab, sizeof(ab), "s_X + %d * NP + el", sp);
                    n.d8.push_back({nb, ab});
                }
                snprintf(nb, sizeof(nb), "y%d", i);
                snprintf(ab, sizeof(ab), "s_Y + %d * NP + el", i);
                n.d8.push_back({nb, ab});
                if (L > 0) {
                    snprintf(nb, sizeof(nb), "ar%d", i);
                    snprintf(ab, sizeof(ab), "ring + (%d + t %% %d) * NP + el", P.roff[i], L);
                    n.d8.push_back({nb, ab});
                }
                for (int l : req_links(i)) need[(size_t)l] = 1;
            }
            for (int r = 0; r < M; r++)
                if (P.rt_node[r] == j) {
                    snprintf(nb, sizeof(nb), "u%d", r);
                    snprintf(ab, sizeof(ab), "s_U + %d * NP + el", r);
                    n.d8.push_back({nb, ab});
                }
            if (P.has_seg[j])
                for (int l = seg0[j]; l <= seg1[j]; l++) need[(size_t)l] = 1;
            for (int l = 0; l < E; l++)
                if (need[(size_t)l]) n.acts.push_back(l);
        }
        o("  double total = 0.0;");
        o("  if (do_step) {");
        // reorder links whose purchaser holds no inventory: pipeline bookkeeping only (before any X row changes)
        for (int i = 0; i < E; i++) {
            if (has_pur[i]) continue;
            const int s = P.sup[i], L = P.L[i];
            o("    {");
            if (s >= 0) o("      const double xq = s_X[%d * NP + el];", s);
            for (int l : req_links(i)) o("      const double rq%d = REQ(%d);", l, l);
            emit_rt(i, "xq", "      ");
            if (L == 0)
                o("      const double ar = rt%d;", i);
            else
                o("      double* slot = ring + (%d + t %% %d) * NP + el; const double ar = *slot; %s", P.roff[i], L,
                  ring_commit(P, "slot", "rt" + std::to_string(i)).c_str());
            o("      s_Y[%d * NP + el] = (s_Y[%d * NP + el] - ar) + rt%d; }", i, i, i);
        }
        // Each node ends in stores and (uniform) branches around the optional info outputs, basic-block boundaries the
        // compiler does not hoist loads across, so a warp pays one memory round trip per node.  Writing the loads of node
        // j + 1 or j + 2 before the arithmetic of node j does not shorten that: at the 64 registers that keep the whole
        // batch resident the looked-ahead values are spilled as they arrive (0.417 / 0.417 / 0.443 ms for a look-ahead of
        // 0 / 1 / 2 nodes).
        for (int j = 0; j < J; j++) {
            o("    {");
            const NodeLd& n = nld[(size_t)j];
            for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
                const int i = P.pred_idx[z], L = P.L[i];
                if (L > 0) o("      double* const slot%d = ring + (%d + t %% %d) * NP + el;", i, P.roff[i], L);
            }
            // loads first (all independent)
            for (const auto& d : n.d8) o("      const double %s = *(%s);", d.first.c_str(), d.second.c_str());
            for (int l : n.acts) o("      const double rq%d = REQ(%d);", l, l);
            // R_t of the inbound links, own allocation chain
            for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
                const int i = P.pred_idx[z];
                emit_rt(i, "xq" + std::to_string(i), "      ");
            }
            if (P.has_seg[j]) emit_chain(j, seg1[j], "x" + std::to_string(j), "qs", "      ", true);
            emit_visit(j, P.has_seg[j] ? "cons_qs" : "0.0", "qs");
            o("    }");
            // a CTA-wide barrier after every 4th node keeps the warps of a CTA within the same stretch of this long
            // straight-line kernel, so an instruction line is fetched once per CTA rather than once per warp (measured:
            // 0.417 ms without, 0.389-0.393 with, for any cadence from 1 to 8 nodes)
            if ((j + 1) % 4 == 0 && j + 1 < J) {
                o("  }");
                o("  __syncthreads();");
                o("  if (do_step) {");
            }
        }
    } else {
    // ---- pass A: orders, 32 links per action chunk
    o("  double cons = 0.0;");
    for (int j = 0; j < J; j++)
        if (P.has_seg[j]) o("  double xs%d = 0.0;", j);
    for (int c0 = 0; c0 < E; c0 += 32) {
        const int c1 = std::min(E, c0 + 32);
        o("  __syncwarp();");
        o("  for (int r = wrow0; r < wrow1; r++)");
        o("    if (%d + ln < NE) tile[r * 33 + ln] = A.actions[(e0 + r) * NE + %d + ln];", c0, c0);
        o("  __syncwarp();");
        o("  if (do_step) {");
        // independent loads first: the on-hand inventory of every supplier whose segment starts in this chunk
        for (int i = c0; i < c1; i++) {
            const int s = P.sup[i];
            if (s >= 0 && (i == 0 || P.sup[i - 1] != s)) o("    xs%d = s_X[%d * NP + el];", s, s);
        }
        for (int i = c0; i < c1; i++) {
            const int s = P.sup[i];
            o("    { double req = rint((double)trow[%d]); req = req > 0.0 ? req : 0.0; double f;", i - c0);
            if (s == -1)
                o("      f = req;");
            else if (s < 0)
                o("      f = 0.0; (void)req;");
            else {
                if (i == 0 || P.sup[i - 1] != s) o("      cons = 0.0;");
                emit_alloc(o, P, s, "      ", "      ", "xs" + std::to_string(s), "cons", "f");
                o("      cons += %s;", consumed(P, s, "f").c_str());
                if (i == E - 1 || P.sup[i + 1] != s) o("      sc_C[%d * NP + el] = cons;", s);
            }
            o("      sc_R[%d * NP + el] = f;", i);
            o("      if (A.info_sales) A.info_sales[NET_IIDX(A, e, NE + NM, %d)] = f; }", i);
        }
        o("  }");
    }
    // ---- pass B: nodes
    o("  double total = 0.0;");
    o("  if (do_step) {");
    // Nodes are independent of each other in this pass (every link has one purchaser, every market link one retailer;
    // R_t / consumed are read-only here): all loads of a node are issued first, then its arithmetic and stores.  One
    // node at a time measured fastest with the 64-register budget (0.419 ms for the step pair on the 64-node graph;
    // groups of 2 / 3 / 4 nodes: 0.433 / 0.449 / 0.470 ms) -- fewer live values, fewer spills.
    for (int j = 0; j < J; j++) {
        o("    {");
        struct Ld { std::string decl, addr; };
        std::vector<Ld> lds;
        char nb[160], ab[160];
        snprintf(nb, sizeof(nb), "double x%d", j);
        snprintf(ab, sizeof(ab), "s_X + %d * NP + el", j);
        lds.push_back({nb, ab});
        if (P.has_seg[j]) {
            snprintf(nb, sizeof(nb), "const double c%d", j);
            snprintf(ab, sizeof(ab), "sc_C + %d * NP + el", j);
            lds.push_back({nb, ab});
        }
        for (int z = P.pred_ptr[j]; z < P.pred_ptr[j + 1]; z++) {
            const int i = P.pred_idx[z], L = P.L[i];
            snprintf(nb, sizeof(nb), "const double rt%d", i);
            snprintf(ab, sizeof(ab), "sc_R + %d * NP + el", i);
            lds.push_back({nb, ab});
            snprintf(nb, sizeof(nb), "const double y%d", i);
            snprintf(ab, sizeof(ab), "s_Y + %d * NP + el", i);
            lds.push_back({nb, ab});
            if (L > 0) {
                o("      double* const slot%d = ring + (%d + t %% %d) * NP + el;", i, P.roff[i], L);
                snprintf(nb, sizeof(nb), "const double ar%d", i);
                snprintf(ab, sizeof(ab), "slot%d", i);
                lds.push_back({nb, ab});
            }
        }
        for (int r = 0; r < M; r++)
            if (P.rt_node[r] == j) {
                snprintf(nb, sizeof(nb), "const double u%d", r);
                snprintf(ab, sizeof(ab), "s_U + %d * NP + el", r);
                lds.push_back({nb, ab});
            }
        for (int z = P.succ_ptr[j]; z < P.succ_ptr[j + 1]; z++) {
            const int l = P.succ_idx[z];
            if (l < E) {
                snprintf(nb, sizeof(nb), "const double qs%d_%d", j, l);
                snprintf(ab, sizeof(ab), "sc_R + %d * NP + el", l);
                lds.push_back({nb, ab});
            }
        }
        for (const Ld& l : lds) o("      %s = *(%s);", l.decl.c_str(), l.addr.c_str());
        emit_visit(j, P.has_seg[j] ? "c" + std::to_string(j) : "0.0", "qs" + std::to_string(j) + "_");
        o("    }");
    }
    for (int i = 0; i < E; i++) {  // reorder links whose purchaser holds no inventory: pipeline bookkeeping only
        if (has_pur[i]) continue;
        const int L = P.L[i];
        o("    { const double rt = sc_R[%d * NP + el];", i);
        if (L == 0)
            o("      const double ar = rt;");
        else
            o("      double* slot = ring + (%d + t %% %d) * NP + el; const double ar = *slot; %s", P.roff[i], L,
              ring_commit(P, "slot", "rt").c_str());
        o("      s_Y[%d * NP + el] = (s_Y[%d * NP + el] - ar) + rt; }", i, i);
    }
    }
    o("    const int tn = t + 1; const bool trunc = tn >= NT;");
    o("    if (A.info_profit_total) A.info_profit_total[e] = total;");
    o("    A.reward[e] = disc[t] * total; A.terminated[e] = 0; A.truncated[e] = trunc ? 1 : 0;");
    o("    if (trunc && A.autoreset == ORGYM_AUTORESET_SAME_STEP) {");
    o("      if (A.final_obs) { double X[NJ], U[NM > 0 ? NM : 1];");
    o("        for (int j = 0; j < NJ; j++) X[j] = s_X[j * NP + el];");
    o("        for (int r = 0; r < NM; r++) U[r] = s_U[r * NP + el];");
    o("        write_obs(X, U, ring, el, tn, A.final_obs + e * NOBS); }");
    emit_reset("      ");
    o("    } else s_period[el] = tn;");
    o("  }");
    // ---- pass C: observation of the final state, 32 columns at a time (only when net_obs_kernel does not follow)
    if (plan.obs_kernel) {
        o("}");
        return;
    }
    o("  const int tobs = valid ? s_period[el] : 0;");
    {
        // column -> source expression
        std::vector<std::string> col((size_t)W);
        char buf[256];
        for (int r = 0; r < M; r++) {
            snprintf(buf, sizeof(buf), "s_U[%d * NP + el]", r);
            col[(size_t)r] = buf;
        }
        for (int j = 0; j < J; j++) {
            snprintf(buf, sizeof(buf), "s_X[%d * NP + el]", j);
            col[(size_t)(M + j)] = buf;
        }
        int k = M + J;
        for (int i = 0; i < E; i++) {
            const int L = P.L[i];
            if (L == 0) continue;
            o("  const int w%d = tobs %% %d;", i, L);
            for (int q = 0; q < L; q++) {
                snprintf(buf, sizeof(buf), "ring[(%d + (w%d + %d >= %d ? w%d + %d - %d : w%d + %d)) * NP + el]", P.roff[i], i, q, L,
                         i, q, L, i, q);
                col[(size_t)(k + q)] = buf;
            }
            k += L;
        }
        // double-buffered: the loads of chunk c+1 are issued before chunk c is flushed, so their latency overlaps the flush
        o("  float v[32];");
        o("  float vn[32];");
        auto emit_loads = [&](const char* dst, int c0) {
            const int c1 = std::min(W, c0 + 32);
            o("  if (valid) {");
            for (int c = c0; c < c1; c++) o("    %s[%d] = (float)%s;", dst, c - c0, col[(size_t)c].c_str());
            o("  }");
        };
        emit_loads("v", 0);
        for (int c0 = 0; c0 < W; c0 += 32) {
            const int c1 = std::min(W, c0 + 32);
            if (c0 + 32 < W) emit_loads("vn", c0 + 32);
            o("  _Pragma(\"unroll\") for (int c = 0; c < %d; c++) trow[c] = v[c];", c1 - c0);
            o("  __syncwarp();");
            o("  for (int r = wrow0; r < wrow1; r++)");
            o("    if (%d + ln < NOBS) __stcs(A.obs + (e0 + r) * NOBS + %d + ln, tile[r * 33 + ln]);", c0, c0);
            o("  __syncwarp();");
            if (c0 + 32 < W) o("  _Pragma(\"unroll\") for (int c = 0; c < 32; c++) v[c] = vn[c];");
        }
    }
    o("}");
}
}  // namespace

int net_jit_build(NetHandle* H, std::string* err) {
    const NetDev& P = H->dev;
    std::string src = net_jit_source(P, H->plan);
    int rc = orgym_jit_compile(src, "net_jit_step", &H->jit, err);
    if (rc != 0) return rc;
    if (cudaLibraryGetKernel(&H->jit_rollout, H->jit.lib, "net_jit_rollout") != cudaSuccess) {
        *err = "net_jit_rollout missing from the specialised module";
        cudaGetLastError();
        orgym_jit_release(&H->jit);
        return 11;
    }
    // device copy of the per-link demand descriptors
    H->dem_dev = nullptr;
    if (cudaMalloc(&H->dem_dev, sizeof(AliasDev) * (size_t)(P.M > 0 ? P.M : 1)) != cudaSuccess) {
        *err = "device allocation failed";
        orgym_jit_release(&H->jit);
        return 10;
    }
    H->allocs.push_back(H->dem_dev);
    if (P.M > 0) cudaMemcpy(H->dem_dev, P.dem, sizeof(AliasDev) * (size_t)P.M, cudaMemcpyHostToDevice);
    cudaFuncSetAttribute((const void*)H->jit.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaFuncSetAttribute((const void*)H->jit_rollout, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    cudaGetLastError();
    return 0;
}

int net_jit_launch(const NetHandle* H, const NetSimArgs& A_in, cudaStream_t s) {
    const NetDev& P = H->dev;
    NetSimArgs A = A_in;
    const int nthr = NET_JIT_THREADS;
    size_t tile = (size_t)nthr * (P.obs_dim | 1) * 4;
    size_t smem = 16;
    if (!A.rollout && H->plan.stream) {
        A.use_tile = 0;  // the streaming kernel stages through its own tiles
        // [NTHR][33] float staging tile of pass A (two-pass form) and pass C; the single-pass form stages nothing
        smem = H->plan.onepass && H->plan.obs_kernel ? 16 : (size_t)nthr * 33 * 4;
    } else if (!A.rollout) {
        A.use_tile = tile <= 160 * 1024 ? 1 : 0;
        if (A.use_tile) smem = tile;
    } else
        A.use_tile = 0;
    const double* disc = P.disc;
    const AliasDev* dem = H->dem_dev;
    void* args[] = {(void*)&A, (void*)&disc, (void*)&dem};
    unsigned grid = (unsigned)((A.N + nthr - 1) / nthr);
    cudaError_t e = cudaLaunchKernel((const void*)(A.rollout ? H->jit_rollout : H->jit.fn), dim3(grid), dim3(nthr), args, smem, s);
    if (e != cudaSuccess) {
        orgym_set_error("specialised network kernel launch failed: %s", cudaGetErrorString(e));
        return ORGYM_E_CUDA;
    }
    return ORGYM_OK;
}
