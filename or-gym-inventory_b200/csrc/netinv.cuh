// netinv.cuh -- declarations shared by the generic network kernel (netinv.cu) and the code generator (netinv_jit.cu)
#pragma once
#include "common.cuh"
#include "jit.cuh"

#define NJ ORGYM_NET_MAX_NODES
#define NE ORGYM_NET_MAX_REORDER
#define NM ORGYM_NET_MAX_RETAIL
#define NSUCC (NE + NM)

struct NetDev {
    int T, backlog, J, E, M, obs_dim, sumL;
    int ring32;  // the state tile carries a float32 copy of the lead-time rings for net_obs_kernel (NetPlan::ring32)
    const double* disc;  // [T] alpha**t
    double I0[NJ], h[NJ], C[NJ], v[NJ], o[NJ];
    uint8_t is_factory[NJ], is_retail[NJ];
    uint8_t has_seg[NJ];  // the node supplies at least one reorder link (its `consumed` scratch row is written every period)
    int16_t sup[NE], pur[NE], L[NE];
    int32_t roff[NE];
    uint32_t Lmagic[NE];  // ceil(2^32 / L): t % L by multiply-high (0 encodes L <= 1)
    double p[NE], g[NE];
    int16_t rt_node[NM];
    double rt_p[NM], rt_b[NM];
    int16_t succ_ptr[NJ + 1], pred_ptr[NJ + 1];
    int16_t succ_idx[NSUCC], pred_idx[NE];
    AliasDev dem[NM];
};

// Which kernels a handle runs, decided once per graph by net_plan (netinv.cu).  The state layout (NetDev::ring32), the
// generated source and the launches all read this one decision.
struct NetPlan {
    int jit;         // NVRTC specialisation: 0 never (generic kernel), 1 when it compiles, 2 required (failure is an error)
    int stream;      // the specialised STEP kernel is the streaming form: state stays in HBM (large graphs)
    int onepass;     // streaming form in its single-pass variant: suppliers follow their purchasers in node order
    int ring32;      // state tiles carry the float32 ring copy: stream, and net_obs_kernel's shared memory fits the rows
    int obs_kernel;  // net_obs_kernel writes the STEP observation instead of the streaming kernel's pass C (ring32)
};

// threads per CTA of the specialised kernels
#define NET_JIT_THREADS 128

struct NetHandle {
    HandleBase base;
    NetDev dev;
    NetPlan plan;
    int threads;  // threads per CTA of the generic kernel that fit the shared-memory work vectors
    size_t smem;
    std::vector<void*> allocs;
    double* partials;
    // run-time specialised kernel (netinv_jit.cu); jit.fn == nullptr -> generic kernel
    JitKernel jit;             // module + STEP kernel
    cudaKernel_t jit_rollout;  // ROLLOUT kernel of the same module
    AliasDev* dem_dev;  // device copy of dev.dem[] for the specialised kernel
};

// Hundreds of live float64 values per instance: the register-resident specialised kernels spill.  Such graphs get the
// streaming STEP form and launch bounds for 255 registers.
static inline bool net_large_graph(const NetDev& P) { return 2 * P.J + 3 * P.E + 2 * P.M > 128; }

// State layout: tiles of NET_TILE = 128 instances; inside a tile every field is slot-major,
//   [key u64][X J][Y E][U M][ring sumL] f64, [period i32][episode u32], [scratch: R_t E, consumed J] f64
// each slot a contiguous row of 128 values (1 KB).  A warp still reads a slot with fully coalesced 256-byte
// transactions, but -- unlike one global field[slot][env] array with a stride of round_up(N) elements -- the stride
// between slots is a compile-time constant (every access of the specialised kernels becomes base + immediate, no
// 64-bit index arithmetic) and the ~1700 slots of a 64-node graph that one CTA touches per period lie in one
// contiguous 1.7 MB region instead of being spread over as many distinct 1 MB-apart rows (TLB reach, DRAM pages).
#define NET_TILE 128
struct NetState {
    uint64_t* key;
    double *X, *Y, *U, *ring;
    float* ring32;  // [sumL][NET_TILE] float32 copy of `ring` (P.ring32), after the scratch area
    int32_t* period;
    uint32_t* episode;
    // tile_base = state + (env / NET_TILE) * net_tile_bytes(P); index the fields with [slot * NET_TILE + env % NET_TILE]
    __host__ __device__ NetState(void* tile_base, const NetDev& P) {
        char* p = (char*)tile_base;
        key = (uint64_t*)p;
        p += 8 * NET_TILE;
        X = (double*)p;
        Y = X + (size_t)P.J * NET_TILE;
        U = Y + (size_t)P.E * NET_TILE;
        ring = U + (size_t)P.M * NET_TILE;
        p = (char*)(ring + (size_t)P.sumL * NET_TILE);
        period = (int32_t*)p;
        p += 4 * NET_TILE;
        episode = (uint32_t*)p;
        p += 4 * NET_TILE + 8 * (size_t)(P.E + P.J) * NET_TILE;
        ring32 = P.ring32 ? (float*)p : nullptr;
    }
};
// ... followed by the per-instance scratch area [R_t E][consumed J] float64 used by the two-pass streaming STEP kernel
// and, for the large graphs whose observation is assembled by net_obs_kernel, by a float32 copy of the rings: the
// observation is float32 anyway, the values pass through unchanged, and the kernel that rebuilds 504 window columns
// per instance every period reads 4 instead of 8 bytes for each.  `ring` stays authoritative (arrivals are float64).
__host__ __device__ static inline int64_t net_tile_bytes(const NetDev& P) {
    return (int64_t)NET_TILE * (8 + 8 * (int64_t)(P.J + P.E + P.M + P.sumL) + 8 + 8 * (int64_t)(P.E + P.J) +
                                (P.ring32 ? 4 * (int64_t)P.sumL : 0));
}
static inline int64_t net_state_bytes(const NetDev& P, int64_t num_envs) {
    return ((num_envs + NET_TILE - 1) / NET_TILE) * net_tile_bytes(P);
}


// netinv.cu: the kernel plan of a graph, from its size and node order; the only reader of ORGYM_NET_JIT and of the test
// hooks ORGYM_NET_JIT_STREAM, ORGYM_NET_JIT_ONEPASS and ORGYM_NET_OBS_TMA
NetPlan net_plan(const NetDev& P);
// netinv_jit.cu: generate + compile the kernel specialised for this topology (returns 0 on success)
int net_jit_build(NetHandle* H, std::string* err);
int net_jit_launch(const NetHandle* H, const struct NetSimArgs& A, cudaStream_t s);
std::string net_jit_source(const NetDev& P, const NetPlan& plan);  // P.ring32 == plan.ring32
