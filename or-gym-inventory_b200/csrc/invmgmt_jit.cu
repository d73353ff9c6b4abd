// invmgmt_jit.cu -- run-time specialisation of the serial multi-echelon env's fused rollout.
//
// The ahead-of-time kernel (invmgmt.cu: inv_rollout_kernel) keeps the lead-time rings in shared memory and indexes
// them with run-time positions; ncu attributes ~30 % of its 216 warp-instructions per env-step to that bookkeeping
// (ring address arithmetic, LDS/STS, position wrap-around, the policy switch, the period loop, Philox word selection).
// For a given configuration all of it is static: lead times, capacities, prices and the horizon are known at create
// time, and the ring position of period t is t mod L_i.  This generator therefore emits the T periods as straight-line
// CUDA -- every ring slot a named register, every index a literal, prices as hexadecimal float literals, discount
// factors from a constant-memory table -- and compiles it for sm_100a with NVRTC (jit.cu).  The arithmetic (integer
// dynamics, float64 reward terms in the reference's order, numpy's summation order, Philox streams) is the ahead-of-time
// kernel's statement by statement; tests/test_invmgmt_gpu.py checks the two kernels bit for bit against each other.
//
// Reference: inventory_management.py:224-352 (step), benchmark_InvManagementBacklogEnv.py:142-198 (BaseStockAgent).
#include "invmgmt_jit.cuh"

#include <cmath>
#include <cstdarg>

#include "jit.cuh"

namespace {
struct Src {
    std::string s;
    void operator()(const char* fmt, ...) {
        char buf[1024];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof(buf), fmt, ap);
        va_end(ap);
        s += buf;
        s += '\n';
    }
};
std::string lit(double v) {
    char buf[64];
    if (v == 0.0) return "0.0";
    snprintf(buf, sizeof(buf), "%a", v);
    return buf;
}

// integer form of a coefficient: c / 2^qexp (exact by construction of qexp)
long long coef_int(double c, int qexp) { return (long long)std::ldexp(c, -qexp); }

// policy: 0 = base-stock with integer levels (literals: everything that does not depend on the demand -- under
// base-stock that is the whole trajectory of the stages above the retailer, reference quirk :300 -- is folded by the
// compiler), 1 = uniform random orders on {0..c_i}
void emit_kernel(Src& o, const InvJitSpec& S, const char* name, int policy, int min_blocks) {
    const int n = S.n, T = S.T, K = 1 << S.log2k;
    const bool bs = policy == 0, bl = S.backlog != 0;
    int qexp = 0;
    const bool exact = inv_jit_profit_is_exact(S) && inv_jit_quantum(S, &qexp);
    // integer profit (exact only): sum_j (c_j / Q) * x_j in int64, one conversion per period -- or, when the rewards
    // are undiscounted and even the running sum over all periods provably never rounds, one conversion per episode
    bool disc_ok = true, undiscounted = true;
    for (int t = 0; t < T; t++) {
        const double dq = std::ldexp(S.disc[(size_t)t], qexp);
        if (S.disc[(size_t)t] != 1.0) undiscounted = false;
        if (!(dq == 0.0 || std::fabs(dq) > 1e-290)) disc_ok = false;  // scaling by Q must stay exact (no subnormals)
    }
    const bool iprofit = exact && disc_ok;
    const bool episode_sum = iprofit && undiscounted && inv_jit_profit_is_exact(S, T);
    const char* W4[4] = {"w.x", "w.y", "w.z", "w.w"};
    const char* A4[4] = {"a4.x", "a4.y", "a4.z", "a4.w"};
    // (random policy) periods re-rolled into a loop over blocks of UNR periods -- see below.
    // Block length 8 (4 for short horizons, straight-line below 8 periods).  A ring whose lead time divides the block
    // length keeps compile-time slot indices ((tb + u) mod L = u mod L), the others are shifted by L - 1 register moves
    // per period.  Measured on the default configuration (lead times 3, 5, 10; 2^24 x 30): straight-line 2.78-3.0 ms,
    // blocks of 4 2.57, 8 2.55, 12 2.56, 10 (two rings static, run-time Philox word) 2.78, 15 3.01 -- the block has to
    // stay small.
    const int UNR = bs ? 0 : (T >= 16 ? 8 : (T >= 8 ? 4 : 0));
    // The per-period discount factors (times 1/Q under the integer profit) come from a constant-memory table, in the
    // loop and in the straight-line periods alike: DMUL takes a constant-bank operand, whereas a float64 literal costs
    // two uniform-register moves every period.
    if (!episode_sum) {
        o("__constant__ double c_disc[%d] = {", T);
        for (int t = 0; t < T; t++)
            o("    %s,", lit(iprofit ? std::ldexp(S.disc[(size_t)t], qexp) : S.disc[(size_t)t]).c_str());
        o("};");
    }
    o("extern \"C\" __global__ void __launch_bounds__(NTHR, %d) %s(const InvJitArgs A) {", min_blocks, name);
    // alias table, one 32-bit word per bucket: (ceil(threshold / K) << log2k) | alias.  The acceptance test of
    // alias_draw, frac < threshold with frac = w << log2k (low log2k bits zero), is equivalent to
    // (frac | (K-1)) < packed word; buckets that always accept store their own index as alias.
    if (S.log2k > 0) {
        o("  __shared__ unsigned int tab[%d];", K);
        o("  for (int i = threadIdx.x; i < %d; i += NTHR) {", K);
        o("    const uint2 te = A.table[i];");
        o("    const unsigned long long tq = ((unsigned long long)te.x + %uull) >> %d;", (unsigned)(K - 1), S.log2k);
        o("    tab[i] = tq >= %lluull ? (unsigned int)i : (((unsigned int)tq << %d) | te.y);", 1ull << (32 - S.log2k), S.log2k);
        o("  }");
        o("  __syncthreads();");
    }
    o("  const int tid = threadIdx.x;");
    o("  const long long e = (long long)blockIdx.x * NTHR + tid;");
    o("  const bool valid = e < A.N;");
    o("  const unsigned long long key = A.seed + (unsigned long long)(A.env_offset + e);");
    o("  const unsigned int ep = A.episode;");
    for (int i = 0; i < n; i++) o("  int I_%d = %lld;", i, S.I0[i]);
    if (bl)
        for (int j = 0; j <= n; j++) o("  int B_%d = 0;", j);
    for (int i = 0; i < n; i++) {
        if (bs) o("  int ps_%d = 0;", i);
        for (int s = 0; s < S.L[i]; s++) {
            o("  int rr%d_%d = 0;", i, s);
            if (bs) o("  int ar%d_%d = 0;", i, s);
        }
    }
    o("  double ret = 0.0; int s_sales = 0, s_dem = 0, s_stock = 0, s_inv = 0;");
    if (episode_sum) o("  long long acc = 0;");
    o("  uint4 w = make_uint4(0u, 0u, 0u, 0u);");
    // Random policy: nothing folds (every stage sees random orders), and 30 straight-line periods are ~3000 instructions
    // that every warp fetches exactly once -- ncu showed `no_instruction` as that kernel's largest stall.  Its periods are
    // therefore emitted as a LOOP over blocks of UNR periods (UNR a multiple of 4, so the Philox word of a period stays a
    // compile-time choice) with the lead-time rings shifted by register moves instead of being indexed by t mod L, plus a
    // straight-line tail: a few hundred instructions that stay in the instruction cache.  Same arithmetic, same order.
    // per ring: shifted (slot 0 = arriving now, moved at the end of the period) or indexed by (period mod L)
    bool shift[ORGYM_INV_MAX_STAGES];
    for (int i = 0; i < n; i++) shift[i] = UNR > 0 && S.L[i] > 0 && UNR % S.L[i] != 0;
    const int Tloop = UNR > 0 ? T - T % UNR : 0;
    // max(on-hand of stage j after the period, 0); the clamp is left out where inv_value_bounds proves on-hand >= 0
    auto onhand = [&](int j) {
        char b[48];
        if (S.inv_nonneg[j])
            snprintf(b, sizeof(b), "Ic_%d", j);
        else
            snprintf(b, sizeof(b), "(Ic_%d > 0 ? Ic_%d : 0)", j, j);
        return std::string(b);
    };
    // emits period t; inside the loop t = tb + u is symbolic and only u is known here
    auto emit_period = [&](int t, int u, bool in_loop) {
        char tx[32], bx[32], dx[48];
        if (in_loop) {
            snprintf(tx, sizeof(tx), "(unsigned)(tb + %d)", u);
            snprintf(bx, sizeof(bx), "(unsigned)((tb >> 2) + %d)", u >> 2);
            snprintf(dx, sizeof(dx), "c_disc[tb + %d]", u);
        } else {
            snprintf(tx, sizeof(tx), "%uu", (unsigned)t);
            snprintf(bx, sizeof(bx), "%uu", (unsigned)(t >> 2));
            snprintf(dx, sizeof(dx), "c_disc[%d]", t);
        }
        const int w4 = (in_loop ? u : t) & 3;
        const int tq = in_loop ? u : t;               // ring slots of the non-shifted rings: (tb + u) mod L = u mod L
        if (in_loop)
            o("  {  // ---- period tb + %d", u);
        else
            o("  {  // ---- period %d", t);
        // policy
        if (bs) {
            for (int i = 0; i < n; i++) {
                o("    int q_%d = %lld - (I_%d + ps_%d); q_%d = q_%d > 0 ? q_%d : 0; q_%d = q_%d < %lld ? q_%d : %lld;", i,
                  S.target[i], i, i, i, i, i, i, i, S.c[i], i, S.c[i]);
            }
        } else {
            o("    uint4 a4;");
            for (int i = 0; i < n; i++) {
                if ((i & 3) == 0) o("    a4 = philox_block(key, %s, ep, STREAM_ACTION, %uu);", tx, (unsigned)(i >> 2));
                o("    const int q_%d = (int)mulhi32(%s, %lluu);", i, A4[i & 3], (unsigned long long)(S.c[i] + 1));
            }
        }
        // demand
        if (S.log2k > 0) {
            if (w4 == 0) o("    w = philox_block(key, %s, ep, STREAM_DEMAND, 0u);", bx);
            o("    int dl; { const unsigned int wv = %s, pe = tab[wv >> %d];", W4[w4], 32 - S.log2k);
            o("      dl = %d + (int)((((wv << %d) | %uu) < pe) ? (wv >> %d) : (pe & %uu)); }", S.base, S.log2k, (unsigned)(K - 1),
              32 - S.log2k, (unsigned)(K - 1));
        } else {
            o("    const int dl = %d;", S.base);
        }
        // dynamics (:253-312)
        for (int i = 0; i < n; i++) {
            if (bl)
                o("    const int cur_%d = q_%d + B_%d;", i, i, i + 1);
            else
                o("    const int cur_%d = q_%d;", i, i);
            o("    int r_%d = cur_%d < %lld ? cur_%d : %lld;", i, i, S.c[i], i, S.c[i]);
            if (i + 1 < n) o("    r_%d = I_%d < r_%d ? I_%d : r_%d;", i, i + 1, i, i + 1, i);
        }
        for (int i = 0; i < n; i++) {
            if (S.L[i] == 0)
                o("    int Ic_%d = I_%d + r_%d;", i, i, i);
            else
                o("    int Ic_%d = I_%d + rr%d_%d;", i, i, i, shift[i] ? 0 : tq % S.L[i]);
        }
        if (S.base >= 0)
            o("    const int d = dl;");  // the alias table's support starts at base >= 0: max(0, .) is the identity
        else
            o("    const int d = dl > 0 ? dl : 0;");
        if (bl)
            o("    const int fill = d + B_0;");
        else
            o("    const int fill = d;");
        o("    const int s0 = Ic_0 < fill ? Ic_0 : fill;");
        o("    Ic_0 -= s0;");
        for (int i = 1; i < n; i++) o("    Ic_%d -= r_%d;", i, i);
        o("    const int U_0 = fill - s0;");
        for (int i = 0; i < n; i++) o("    const int U_%d = cur_%d - r_%d;", i + 1, i, i);
        // profit (:315-321): elementwise float64, np.sum over m < 8 stages = sequential sum starting from 0.0
        if (iprofit) {
            // every float64 operation of the reference's expression is exact (inv_jit_profit_is_exact), so the profit
            // equals Q * sum_j (c_j / Q) * x_j with integer coefficients c_j / Q: IMADs instead of I2F + DFMA
            o("    long long pa = %s;", episode_sum ? "acc" : "0");
            // terms with the same integer coefficient are summed first (int32, bounded by the sum of their bounds) -- but
            // only within one class.  Under base-stock every quantity of the stages above the retailer is a compile-time
            // constant (reference quirk :300: a stage's on-hand never sees the order it ships downstream), so the
            // retailer's orders, sales, on-hand and unfulfilled quantities (class 0) are kept apart from those of the
            // upstream stages (class 1), which the compiler then folds into one constant per period.
            struct Term { long long c; std::string x; double bound; int cls; };
            std::vector<Term> terms;
            auto add = [&](long long c, const std::string& x, double bound, int cls) {
                if (c == 0) return;
                for (auto& tm : terms)
                    if (tm.c == c && tm.cls == cls && tm.bound + bound < 2147483647.0) {
                        tm.x += " + " + x;
                        tm.bound += bound;
                        return;
                    }
                terms.push_back({c, x, bound, cls});
            };
            // class of the quantities of stage i: its on-hand Ic_i, its fulfilled order r_i (the units stage i + 1 sells)
            // and its unfulfilled request U_{i+1}; i = -1 stands for the retail sale s0 and the unmet demand U_0
            auto cls_of = [&](int i) { return bs && i >= 1 ? 1 : 0; };
            char nm[64];
            for (int j = 0; j <= n; j++) {
                snprintf(nm, sizeof(nm), "U_%d", j);
                add(-coef_int(S.kc[j], qexp), nm, S.unf_bound[j], cls_of(j - 1));
                if (j < n) {
                    add(-coef_int(S.hc[j], qexp), onhand(j), S.inv_bound[j], cls_of(j));
                }
                if (j == 0)
                    snprintf(nm, sizeof(nm), "s0");
                else
                    snprintf(nm, sizeof(nm), "r_%d", j - 1);
                add(coef_int(S.up[j], qexp) - coef_int(S.uc[j], qexp), nm, S.sale_bound[j], cls_of(j - 1));
            }
            for (const auto& tm : terms) {
                const long long ac = tm.c < 0 ? -tm.c : tm.c;
                const char* op = tm.c < 0 ? "-=" : "+=";
                if (ac < 2147483648LL) {
                    o("    pa %s %lldLL * (long long)(%s);", op, ac, tm.x.c_str());  // one IMAD.WIDE
                    continue;
                }
                // coefficient beyond 32 bits: odd part times the integer (int32, by the bound), then a power of two
                int tz = 0;
                while (tz < 30 && ((ac >> tz) & 1) == 0) tz++;
                const long long odd = ac >> tz;
                if ((double)odd * tm.bound < 2147483647.0)
                    o("    pa %s %lldLL * (long long)(%lld * (%s));", op, 1LL << tz, odd, tm.x.c_str());
                else
                    o("    pa %s %lldLL * (long long)(%s);", op, ac, tm.x.c_str());
            }
            if (episode_sum)
                o("    acc = pa;");
            else  // |pa| < 2^51 (the proof leaves one bit of head-room): exact int64 -> float64 through the 2^52 + 2^51
                  // offset (two integer adds and one DADD instead of an I2F.F64.S64 on the quarter-rate pipe)
                o("    ret += %s * (__longlong_as_double(pa + 0x4338000000000000LL) - 0x1.8p52);", dx);
        } else if (exact) {
            // every operation is exact (inv_jit_profit_is_exact): one fused chain, (up - uc) folded into one coefficient
            o("    double pr = 0.0;");
            for (int j = n; j >= 0; j--) {
                o("    pr = fma(%s, (double)U_%d, pr);", lit(-S.kc[j]).c_str(), j);
                if (j < n) o("    { const int inv = %s; pr = fma(%s, (double)inv, pr); }", onhand(j).c_str(), lit(-S.hc[j]).c_str());
                if (j == 0)
                    o("    pr = fma(%s, (double)s0, pr);", lit(S.up[j] - S.uc[j]).c_str());
                else
                    o("    pr = fma(%s, (double)r_%d, pr);", lit(S.up[j] - S.uc[j]).c_str(), j - 1);
            }
            o("    ret += %s * pr;", dx);
        } else {
            for (int j = 0; j <= n; j++) {
                if (j == 0)
                    o("    double tm_%d; { const double s = (double)s0;", j);
                else
                    o("    double tm_%d; { const double s = (double)r_%d;", j, j - 1);
                o("      const double rev = %s * s, pc = %s * s, pen = %s * (double)U_%d;", lit(S.up[j]).c_str(),
                  lit(S.uc[j]).c_str(), lit(S.kc[j]).c_str(), j);
                if (j == n)
                    o("      tm_%d = (rev - pc) - pen; }", j);
                else
                    o("      const int inv = %s; const double hold = %s * (double)inv; tm_%d = ((rev - pc) - hold) - pen; }",
                      onhand(j).c_str(), lit(S.hc[j]).c_str(), j);
            }
            o("    double pr = 0.0;");
            for (int j = 0; j <= n; j++) o("    pr = pr + tm_%d;", j);
            o("    ret += %s * pr;", dx);
        }
        // statistics and state
        o("    s_sales += s0; s_dem += d; s_stock += U_0;");
        for (int i = 0; i < n; i++) o("    I_%d = Ic_%d; s_inv += %s;", i, i, onhand(i).c_str());
        if (bl)
            for (int j = 0; j <= n; j++) o("    B_%d = U_%d;", j, j);
        // rings: slot t mod L_i held R[t - L_i] / the request of period t - L_i
        for (int i = 0; i < n; i++) {
            if (S.L[i] == 0) continue;
            if (shift[i]) {  // slot 0 has arrived: everything moves one period closer, the new order enters at the back
                for (int q = 0; q + 1 < S.L[i]; q++) o("    rr%d_%d = rr%d_%d;", i, q, i, q + 1);
                o("    rr%d_%d = r_%d;", i, S.L[i] - 1, i);
                continue;
            }
            const int s = tq % S.L[i];
            if (bs) o("    ps_%d = ps_%d + q_%d - ar%d_%d; ar%d_%d = q_%d;", i, i, i, i, s, i, s, i);
            o("    rr%d_%d = r_%d;", i, s, i);
        }
        o("  }");
    };
    if (UNR > 0) {
        o("  for (int tb = 0; tb < %d; tb += %d) {", Tloop, UNR);
        for (int u = 0; u < UNR; u++) emit_period(0, u, true);
        o("  }");
        for (int t = Tloop; t < T; t++) emit_period(t, 0, false);
    } else {
        for (int t = 0; t < T; t++) emit_period(t, 0, false);
    }
    if (episode_sum) o("  ret = (double)acc * %s;", lit(std::ldexp(1.0, qexp)).c_str());
    // outputs: identical to the ahead-of-time kernel
    o("  if (valid) {");
    o("    if (A.ep_return) A.ep_return[e] = ret;");
    o("    if (A.stats) *reinterpret_cast<longlong4*>(A.stats + e * 4) = make_longlong4((long long)s_sales, (long long)s_dem, (long long)s_stock, (long long)s_inv);");
    o("    if (A.stats32) *reinterpret_cast<int4*>(A.stats32 + e * 4) = make_int4(s_sales, s_dem, s_stock, s_inv);");
    o("  }");
    // Block partial sums.  The two float64 sums (return, return^2) keep their fixed-order xor-shuffle tree; the count and
    // the four statistics are integers whose float64 sums are exact in any order, so their warp sums are
    // integer reductions in hardware (REDUX, 16 bits at a time: no 32-bit sum can overflow) -- 8 instructions instead
    // of 50 shuffles and 25 float64 additions, the same values.
    o("  if (A.partials) {");
    o("    double v[7];");
    o("    v[0] = (double)__popc(__ballot_sync(0xffffffffu, valid));");
    o("    v[1] = valid ? ret : 0.0; v[2] = valid ? ret * ret : 0.0;");
    o("    _Pragma(\"unroll\") for (int q = 1; q < 3; q++)");
    o("      _Pragma(\"unroll\") for (int s = 16; s > 0; s >>= 1) v[q] += __shfl_xor_sync(0xffffffffu, v[q], s);");
    o("    { const int w4[4] = {valid ? s_sales : 0, valid ? s_dem : 0, valid ? s_stock : 0, valid ? s_inv : 0};");
    o("      _Pragma(\"unroll\") for (int q = 0; q < 4; q++) {   // x = (x >> 16) * 65536 + (x & 0xFFFF) for any int x (sales can be negative)");
    o("        const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)w4[q] & 0xFFFFu);");
    o("        const int hi = __reduce_add_sync(0xffffffffu, w4[q] >> 16);");
    o("        v[3 + q] = (double)((long long)hi * 65536 + (long long)lo); } }");
    o("    __shared__ double red[NTHR / 32][7];");
    o("    if ((tid & 31) == 0) { _Pragma(\"unroll\") for (int q = 0; q < 7; q++) red[tid >> 5][q] = v[q]; }");
    o("    __syncthreads();");
    o("    if (tid < 7) { double x = 0.0; for (int wv = 0; wv < NTHR / 32; wv++) x += red[wv][tid]; A.partials[(long long)blockIdx.x * 8 + tid] = x; }");
    o("  }");
    o("}");
}
}  // namespace

// The profit of a period is a sum of products coefficient x integer.  Every coefficient is a float32 value, i.e. an
// integer multiple of some power of two; let Q be the smallest such quantum over all coefficients.  Then every product,
// partial sum and difference that can occur is an integer multiple of Q, and float64 represents all multiples of Q below
// 2^53 * Q exactly.  If the largest possible magnitude (with two bits of head-room: below 2^51 * Q)  sum_j (|up_j| + |uc_j|) * |sold_j| + |hc_j| * inv_j + |kc_j| * unf_j
// (per-term bounds from inv_value_bounds) stays below that, no operation ever rounds: the reference's evaluation order,
// any re-association, fused multiply-adds and plain integer arithmetic on the coefficients / Q all give the same value,
// and the generator may use the cheapest form.
bool inv_jit_quantum(const InvJitSpec& S, int* qexp_out) {
    int qexp = 1 << 20;  // exponent of the finest quantum
    for (int j = 0; j <= S.n; j++) {
        const double cs[4] = {S.up[j], S.uc[j], S.hc[j], S.kc[j]};
        for (double c : cs) {
            if (!(c >= 0.0) || !std::isfinite(c)) return false;
            if (c == 0.0) continue;
            if ((double)(float)c != c) return false;  // not a float32 value: no 24-bit significand guarantee
            int e;
            double m = std::frexp(c, &e);             // c = m * 2^e, 0.5 <= m < 1
            long long mi = (long long)std::ldexp(m, 53);  // 53-bit integer significand
            int tz = 0;
            while ((mi & 1) == 0) { mi >>= 1; tz++; }
            qexp = std::min(qexp, e - 53 + tz);       // c = odd * 2^(e - 53 + tz)
        }
    }
    if (qexp == (1 << 20)) qexp = 0;                  // all coefficients zero
    *qexp_out = qexp;
    return true;
}

double inv_jit_profit_mag(const InvJitSpec& S) {
    double mag = 0.0;
    for (int j = 0; j <= S.n; j++)
        mag += (S.up[j] + S.uc[j]) * S.sale_bound[j] + S.hc[j] * S.inv_bound[j] + S.kc[j] * S.unf_bound[j];
    return mag;
}

bool inv_jit_profit_is_exact(const InvJitSpec& S, int periods) {
    if (S.xbound <= 0) return false;
    int qexp = 0;
    if (!inv_jit_quantum(S, &qexp)) return false;
    for (int j = 0; j <= S.n; j++)
        if (!(S.sale_bound[j] >= 0.0 && S.inv_bound[j] >= 0.0 && S.unf_bound[j] >= 0.0)) return false;
    const double limit = std::ldexp(1.0, 51 + qexp);  // a quarter of 2^53 * Q: |profit / Q| < 2^51, two bits of head-room
    return inv_jit_profit_mag(S) * (double)(periods > 1 ? periods : 1) < limit;
}

bool inv_jit_eligible(const InvJitSpec& S) {
    if (S.n < 1 || S.n > 6) return false;  // m = n + 1 < 8: the reward sum is numpy's sequential branch
    if (S.T < 1 || S.T > 64 || (int)S.disc.size() != S.T) return false;
    if (S.log2k < 0 || S.log2k > 10) return false;
    int sumL = 0;
    for (int i = 0; i < S.n; i++) {
        if (S.c[i] < 0 || S.c[i] > 0x3fffffffLL || S.I0[i] < 0 || S.I0[i] > 0x3fffffffLL) return false;
        sumL += S.L[i];
    }
    return sumL <= 40;  // two register-resident rings of sum(L) entries each
}

const char* inv_jit_kernel_name(int policy) { return policy == 0 ? "inv_jit_rollout_bs" : "inv_jit_rollout_rnd"; }

std::string inv_jit_source(const InvJitSpec& S) {
    Src o;
    o.s += orgym_jit_device_rng_src();
    o.s += orgym_jit_inv_args_src();
    o("#define NTHR %d", INV_JIT_THREADS);
    // base-stock keeps only the retailer's state per thread (the rest is folded): room for more resident CTAs
    // (minimum-CTA sweep in profiles/r02_sweeps.txt)
    emit_kernel(o, S, inv_jit_kernel_name(S.policy), S.policy, S.policy == 0 ? 8 : 4);
    return o.s;
}
