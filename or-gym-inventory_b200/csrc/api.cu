// api.cu -- family-independent part of the C ABI: error string, version, handle header, error bits,
// alias-table construction for the fixed demand distributions, stand-alone samplers (K6).
#include "common.cuh"
#include "poisson_mu.cuh"
#include <mutex>

static thread_local std::string g_last_error;

void orgym_set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

extern "C" const char* orgym_last_error(void) { return g_last_error.c_str(); }
extern "C" int orgym_version(void) { return ORGYM_VERSION; }
extern "C" int orgym_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int orgym_handle_base_init(HandleBase* b, int family, int device, int64_t num_envs) {
    b->magic = ORGYM_MAGIC;
    b->family = family;
    b->device = device;
    b->num_envs = num_envs;
    b->err_dev = nullptr;
    int n = orgym_device_count();
    if (n <= 0) {
        orgym_set_error("no CUDA device is visible; or-gym-inventory_b200 has no CPU fallback");
        return ORGYM_E_CUDA;
    }
    ORGYM_REQUIRE(device >= 0 && device < n, "device %d out of range (0..%d)", device, n - 1);
    ORGYM_REQUIRE(num_envs >= 1, "num_envs must be >= 1");
    DeviceGuard g(device);
    ORGYM_CUDA(cudaMalloc(&b->err_dev, sizeof(uint32_t)));
    ORGYM_CUDA(cudaMemset(b->err_dev, 0, sizeof(uint32_t)));
    return ORGYM_OK;
}

void orgym_handle_base_free(HandleBase* b) {
    if (b->err_dev) {
        DeviceGuard g(b->device);
        cudaFree(b->err_dev);
        b->err_dev = nullptr;
    }
    b->magic = 0;
}

int orgym_check_handle(const void* h, int family) {
    const HandleBase* b = (const HandleBase*)h;
    if (!b || b->magic != ORGYM_MAGIC || (family && b->family != family)) {
        orgym_set_error("invalid handle");
        return ORGYM_E_INVALID;
    }
    return ORGYM_OK;
}

extern "C" int orgym_errors(orgym_handle_t h, uint32_t* bits_out, int clear, void* stream) {
    if (orgym_check_handle(h, 0)) return ORGYM_E_INVALID;
    HandleBase* b = (HandleBase*)h;
    DeviceGuard g(b->device);
    cudaStream_t s = (cudaStream_t)stream;
    uint32_t bits = 0;
    ORGYM_CUDA(cudaMemcpyAsync(&bits, b->err_dev, sizeof(bits), cudaMemcpyDeviceToHost, s));
    ORGYM_CUDA(cudaStreamSynchronize(s));
    if (clear && bits) ORGYM_CUDA(cudaMemsetAsync(b->err_dev, 0, sizeof(uint32_t), s));
    if (bits_out) *bits_out = bits;
    return ORGYM_OK;
}

// ------------------------------------------------------------------------------------------------
// probability mass functions of the reference's demand distributions (inventory_management.py:169-184)
// ------------------------------------------------------------------------------------------------
int orgym_dist_pmf(const orgym_dist_t* d, std::vector<double>* pmf, int64_t* base) {
    pmf->clear();
    *base = 0;
    const double TAIL = 1e-19;
    switch (d->kind) {
        case ORGYM_DIST_POISSON: {
            double mu = d->p0;
            ORGYM_REQUIRE(mu >= 0 && std::isfinite(mu), "Poisson mean must be finite and >= 0 (got %g)", mu);
            if (mu == 0) {
                pmf->push_back(1.0);
                return ORGYM_OK;
            }
            int64_t lo = (int64_t)std::floor(mu - 12.0 * std::sqrt(mu) - 12.0);
            if (lo < 0) lo = 0;
            int64_t hi = (int64_t)std::ceil(mu + 14.0 * std::sqrt(mu) + 40.0);
            *base = lo;
            for (int64_t k = lo; k <= hi; k++) pmf->push_back(std::exp(-mu + k * std::log(mu) - std::lgamma((double)k + 1.0)));
            break;
        }
        case ORGYM_DIST_BINOMIAL: {
            double nn = d->p0, p = d->p1;
            ORGYM_REQUIRE(nn >= 0 && nn == std::floor(nn) && p >= 0 && p <= 1, "binomial needs integer n >= 0 and 0 <= p <= 1");
            int64_t n = (int64_t)nn;
            for (int64_t k = 0; k <= n; k++) {
                double lp = std::lgamma(nn + 1) - std::lgamma((double)k + 1) - std::lgamma((double)(n - k) + 1);
                double v;
                if (p == 0)
                    v = k == 0 ? 1.0 : 0.0;
                else if (p == 1)
                    v = k == n ? 1.0 : 0.0;
                else
                    v = std::exp(lp + k * std::log(p) + (n - k) * std::log1p(-p));
                pmf->push_back(v);
            }
            break;
        }
        case ORGYM_DIST_RANDINT: {
            double lo = d->p0, hi = d->p1;
            ORGYM_REQUIRE(lo == std::floor(lo) && hi == std::floor(hi) && hi >= lo, "randint needs integer low <= high");
            ORGYM_REQUIRE(lo > -2e9 && hi < 2e9, "randint bounds out of int32 range");
            *base = (int64_t)lo;
            int64_t len = (int64_t)(hi - lo) + 1;
            ORGYM_REQUIRE(len <= 4096, "randint support wider than 4096 values is not supported");
            pmf->assign((size_t)len, 1.0 / (double)len);
            break;
        }
        case ORGYM_DIST_GEOMETRIC: {
            double p = d->p0;
            ORGYM_REQUIRE(p > 0 && p <= 1, "geometric needs 0 < p <= 1");
            *base = 1;  // numpy's geometric counts trials: support 1, 2, ...
            double q = 1.0, tail = 1.0;
            while (tail > TAIL && pmf->size() < 4096) {
                pmf->push_back(q * p);
                q *= (1.0 - p);
                tail = q;
            }
            if (tail > TAIL) {  // numpy's geometric has unbounded support: never truncate-and-renormalise silently
                orgym_set_error("geometric(p=%g): %.3g of the probability mass lies beyond the 4096-entry alias table "
                                "(p must be at least about 0.0107)", p, tail);
                return ORGYM_E_UNSUPPORTED;
            }
            break;
        }
        default:
            orgym_set_error("distribution kind %d has no pmf", d->kind);
            return ORGYM_E_INVALID;
    }
    // trim negligible tails, normalise
    size_t a = 0, b = pmf->size();
    while (b - a > 1 && (*pmf)[a] < TAIL) a++;
    while (b - a > 1 && (*pmf)[b - 1] < TAIL) b--;
    std::vector<double> t(pmf->begin() + a, pmf->begin() + b);
    *base += (int64_t)a;
    double s = 0;
    for (double v : t) s += v;
    ORGYM_REQUIRE(s > 0, "degenerate distribution");
    for (double& v : t) v /= s;
    pmf->swap(t);
    if (pmf->size() > 4096) {
        orgym_set_error("demand distribution support (%zu values) exceeds the 4096-entry alias table", pmf->size());
        return ORGYM_E_UNSUPPORTED;
    }
    return ORGYM_OK;
}

// Walker/Vose alias construction over K >= pmf.size() buckets (the extra buckets have probability 0): bucket i gets
// {threshold (32-bit fixed point, accept i if u < threshold), alias index}
static void vose_alias(const std::vector<double>& pmf, size_t K, uint2* tab) {
    std::vector<double> q(K, 0.0);
    for (size_t i = 0; i < pmf.size(); i++) q[i] = pmf[i] * (double)K;
    std::vector<uint32_t> small, large;
    for (size_t i = 0; i < K; i++) (q[i] < 1.0 ? small : large).push_back((uint32_t)i);
    auto thr = [](double x) {
        double v = std::floor(x * 4294967296.0 + 0.5);
        if (v < 0) v = 0;
        if (v > 4294967295.0) v = 4294967295.0;
        return (uint32_t)v;
    };
    for (size_t i = 0; i < K; i++) tab[i] = make_uint2(0xFFFFFFFFu, (uint32_t)i);
    while (!small.empty() && !large.empty()) {
        uint32_t s = small.back(), l = large.back();
        small.pop_back();
        large.pop_back();
        tab[s] = make_uint2(thr(q[s]), l);
        q[l] = (q[l] + q[s]) - 1.0;
        (q[l] < 1.0 ? small : large).push_back(l);
    }
    // leftovers are 1.0 up to rounding: keep {0xFFFFFFFF, self}
}

// alias table with 2^log2k buckets for one of the fixed demand distributions
int orgym_build_alias(const orgym_dist_t* d, int user_clamp, AliasDev* out, std::vector<void*>* allocs) {
    memset(out, 0, sizeof(*out));
    out->kind = d->kind;
    out->user_clamp = user_clamp;
    if (d->kind == ORGYM_DIST_USER) {
        ORGYM_REQUIRE(d->user_D_len > 0 && d->user_D, "user_D trace is empty");
        int64_t* dev = nullptr;
        ORGYM_CUDA(cudaMalloc(&dev, sizeof(int64_t) * (size_t)d->user_D_len));
        allocs->push_back(dev);
        ORGYM_CUDA(cudaMemcpy(dev, d->user_D, sizeof(int64_t) * (size_t)d->user_D_len, cudaMemcpyHostToDevice));
        out->user_D = dev;
        out->user_D_len = d->user_D_len;
        return ORGYM_OK;
    }
    std::vector<double> pmf;
    int64_t base = 0;
    int rc = orgym_dist_pmf(d, &pmf, &base);
    if (rc) return rc;
    int log2k = 0;
    while ((size_t(1) << log2k) < pmf.size()) log2k++;
    size_t K = size_t(1) << log2k;
    std::vector<uint2> tab(K);
    vose_alias(pmf, K, tab.data());
    uint2* dev = nullptr;
    ORGYM_CUDA(cudaMalloc(&dev, sizeof(uint2) * K));
    allocs->push_back(dev);
    ORGYM_CUDA(cudaMemcpy(dev, tab.data(), sizeof(uint2) * K, cudaMemcpyHostToDevice));
    out->table = dev;
    out->log2k = log2k;
    out->base = (int32_t)base;
    return ORGYM_OK;
}

// ------------------------------------------------------------------------------------------------
// reciprocal table used by the Poisson recurrences (common.cuh)
// ------------------------------------------------------------------------------------------------
int orgym_rcp_table(int device, const double** out) {
    static double* tabs[64] = {nullptr};
    ORGYM_REQUIRE(device >= 0 && device < 64, "device index out of range");
    if (!tabs[device]) {
        DeviceGuard g(device);
        std::vector<double> h(ORGYM_RCP_N + 1, 0.0);
        for (int k = 1; k <= ORGYM_RCP_N; k++) h[(size_t)k] = 1.0 / (double)k;
        double* d = nullptr;
        ORGYM_CUDA(cudaMalloc(&d, sizeof(double) * h.size()));
        ORGYM_CUDA(cudaMemcpy(d, h.data(), sizeof(double) * h.size(), cudaMemcpyHostToDevice));
        tabs[device] = d;
    }
    *out = tabs[device];
    return ORGYM_OK;
}

// ------------------------------------------------------------------------------------------------
// alias tables of Poisson(4 i), i = 0 .. ntab-1, for the per-env-mean sampler (common.cuh: poisson_tab_draw)
// ------------------------------------------------------------------------------------------------
int orgym_poisson_tables(int device, double mu_hi, PoisTabDev* out) {
    struct Built {
        int device;
        PoisTabDev t;
    };
    static std::mutex mtx;
    static std::vector<Built> cache;
    ORGYM_REQUIRE(device >= 0, "device index out of range");
    if (!(mu_hi > 256.0)) mu_hi = 256.0;  // default coverage: the reference's mu_max = 200 with margin
    if (mu_hi > ORGYM_PT_MAX_MEAN) mu_hi = ORGYM_PT_MAX_MEAN;
    const int ntab = (int)std::floor(mu_hi / ORGYM_PT_G) + 1;
    std::lock_guard<std::mutex> lock(mtx);
    for (const Built& b : cache)
        if (b.device == device && b.t.ntab >= ntab) {
            *out = b.t;
            return ORGYM_OK;
        }
    std::vector<std::vector<double>> pmfs((size_t)ntab);
    std::vector<int64_t> bases((size_t)ntab, 0);
    size_t widest = 1;
    for (int i = 0; i < ntab; i++) {
        orgym_dist_t d;
        memset(&d, 0, sizeof(d));
        d.kind = ORGYM_DIST_POISSON;
        d.p0 = (double)(ORGYM_PT_G * i);
        if (int rc = orgym_dist_pmf(&d, &pmfs[(size_t)i], &bases[(size_t)i])) return rc;
        widest = std::max(widest, pmfs[(size_t)i].size());
    }
    int log2k = 0;
    while ((size_t(1) << log2k) < widest) log2k++;
    const size_t K = size_t(1) << log2k;
    std::vector<uint2> all((size_t)ntab * K), one(K);
    for (int i = 0; i < ntab; i++) {
        vose_alias(pmfs[(size_t)i], K, one.data());
        const uint32_t base = (uint32_t)bases[(size_t)i];
        ORGYM_REQUIRE(base + K <= 65536, "Poisson table values exceed 16 bits");
        for (size_t j = 0; j < K; j++)
            all[(size_t)i * K + j] = make_uint2(one[j].x, (base + (uint32_t)j) | ((base + one[j].y) << 16));
    }
    DeviceGuard g(device);
    uint2* dev = nullptr;
    ORGYM_CUDA(cudaMalloc(&dev, sizeof(uint2) * all.size()));
    ORGYM_CUDA(cudaMemcpy(dev, all.data(), sizeof(uint2) * all.size(), cudaMemcpyHostToDevice));
    Built b;
    b.device = device;
    b.t.tab = dev;
    b.t.log2k = log2k;
    b.t.ntab = ntab;
    cache.push_back(b);
    *out = b.t;
    return ORGYM_OK;
}

// ------------------------------------------------------------------------------------------------
// K6: stand-alone samplers for the statistical tests
// ------------------------------------------------------------------------------------------------
__global__ void sample_fixed_kernel(AliasDev A, uint64_t seed, int64_t env_offset, int64_t count, int per_env,
                                    int64_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    int64_t env = env_offset + i / per_env;
    int t = (int)(i % per_env);
    out[i] = sample_fixed(A, A.table, seed + (uint64_t)env, 0u, t, 0u);
}

extern "C" int orgym_sample_demand(const orgym_dist_t* dist, uint64_t seed, int64_t env_offset, int64_t num_envs,
                                   int32_t per_env, int device, int64_t* out_dev, void* stream) {
    ORGYM_REQUIRE(dist && out_dev && num_envs > 0 && per_env > 0, "bad arguments");
    ORGYM_REQUIRE(orgym_device_count() > 0, "no CUDA device");
    DeviceGuard g(device);
    std::vector<void*> allocs;
    AliasDev A;
    int rc = orgym_build_alias(dist, 0, &A, &allocs);
    if (rc == ORGYM_OK) {
        int64_t count = num_envs * per_env;
        sample_fixed_kernel<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(A, seed, env_offset, count,
                                                                                            per_env, out_dev);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
        if (e != cudaSuccess) {
            orgym_set_error("sample kernel failed: %s", cudaGetErrorString(e));
            rc = ORGYM_E_CUDA;
        }
    }
    for (void* p : allocs) cudaFree(p);
    return rc;
}

__global__ void sample_poisson_mu_kernel(const double* __restrict__ mu, PoisTabDev T, const double* __restrict__ rcp,
                                         uint64_t seed, int64_t env_offset, int64_t count, int period,
                                         int64_t* __restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    out[i] = poisson_mu(T, rcp, mu[i], seed + (uint64_t)(env_offset + i), 0u, period);
}

extern "C" int orgym_sample_poisson_mu(const double* mu_dev, uint64_t seed, int64_t env_offset, int64_t count,
                                       int32_t period, int device, int64_t* out_dev, void* stream) {
    ORGYM_REQUIRE(mu_dev && out_dev && count > 0, "bad arguments");
    ORGYM_REQUIRE(orgym_device_count() > 0, "no CUDA device");
    const double* rcp = nullptr;
    if (int rc = orgym_rcp_table(device, &rcp)) return rc;
    PoisTabDev T;  // default coverage (means below 260); larger means take the PTRS path
    if (int rc = orgym_poisson_tables(device, 0.0, &T)) return rc;
    DeviceGuard g(device);
    sample_poisson_mu_kernel<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(mu_dev, T, rcp, seed,
                                                                                              env_offset, count, period,
                                                                                              out_dev);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}

// ------------------------------------------------------------------------------------------------
// deterministic summary reduction (see common.cuh)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) orgym_reduce_partials_kernel(const double* __restrict__ partials, int nrows,
                                                                    double* __restrict__ scratch,
                                                                    unsigned int* __restrict__ ticket,
                                                                    double* __restrict__ out) {
    const int tid = threadIdx.x, nb = gridDim.x;
    const int rpb = (nrows + nb - 1) / nb;
    const int r0 = blockIdx.x * rpb, r1 = min(nrows, r0 + rpb);
    double v[7] = {0, 0, 0, 0, 0, 0, 0};
    // a thread's rows r, r + 256, ... are summed in that order; the loads of 4 of them are issued before the first add
    for (int r = r0 + tid; r < r1; r += 4 * 256) {
        double4 a[4], b[4];
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (r + k * 256 < r1) {
                a[k] = *reinterpret_cast<const double4*>(partials + (size_t)(r + k * 256) * 8);
                b[k] = *reinterpret_cast<const double4*>(partials + (size_t)(r + k * 256) * 8 + 4);
            }
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (r + k * 256 < r1) {
                v[0] += a[k].x; v[1] += a[k].y; v[2] += a[k].z; v[3] += a[k].w;
                v[4] += b[k].x; v[5] += b[k].y; v[6] += b[k].z;
            }
    }
    __shared__ double red[8][7];
    __shared__ int is_last;
#pragma unroll
    for (int q = 0; q < 7; q++) {
        double x = v[q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if ((tid & 31) == 0) red[tid >> 5][q] = x;
    }
    __syncthreads();
    if (tid < 7) {
        double x = 0.0;
        for (int w = 0; w < 8; w++) x += red[w][tid];
        scratch[(size_t)blockIdx.x * 8 + tid] = x;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = (atomicInc(ticket, (unsigned)nb - 1u) == (unsigned)nb - 1u);
    __syncthreads();
    if (is_last) {  // block-uniform: the barrier below is reached by every thread of the last CTA
        __threadfence();
        // the CTA sums are staged in shared memory by all threads at once, then added in block order as before
        __shared__ double fin[ORGYM_REDUCE_CTAS][7];
        for (int i = tid; i < nb * 7; i += 256) fin[i / 7][i % 7] = __ldcg(scratch + (size_t)(i / 7) * 8 + i % 7);
        __syncthreads();
        if (tid < 8) {
            double x = 0.0;
            if (tid < 7)
                for (int b = 0; b < nb; b++) x += fin[b][tid];
            out[tid] = x;
        }
    }
}

int orgym_launch_reduce(double* partials, int nrows, double* out_dev, cudaStream_t s) {
    double* scratch = partials + (size_t)nrows * 8;
    unsigned int* ticket = (unsigned int*)(scratch + ORGYM_REDUCE_CTAS * 8);
    int nb = nrows < 4096 ? 1 : ORGYM_REDUCE_CTAS;
    orgym_reduce_partials_kernel<<<nb, 256, 0, s>>>(partials, nrows, scratch, ticket, out_dev);
    ORGYM_CUDA(cudaGetLastError());
    return ORGYM_OK;
}
