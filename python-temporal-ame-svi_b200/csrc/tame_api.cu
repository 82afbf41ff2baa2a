// tame_api.cu -- the C ABI of include/tame_b200.h: handle management, sweep orchestration, ELBO reduction,
// the fit loop of src/inference/base.py:127-208, the device-side data generator and the NCCL plumbing.
#include <cuda_runtime.h>
#include <curand_kernel.h>
#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <thread>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/tame_b200.h"
#include "tame_kernels.cuh"

// ------------------------------------------------------------------------------------------------------
// bookkeeping
// ------------------------------------------------------------------------------------------------------
static constexpr size_t FIT_PART_DOUBLES = 10 * 1024;   // (grid <= 1024 blocks) x (6 + 4) partial sums of k_fit
static_assert(sizeof(tame_config) == 120, "tame_config layout is part of the ABI (ctypes mirror in _lib.py)");
static thread_local std::string g_err;
static std::atomic<int64_t> g_launches{0};
void tame_count_launch(int n) { g_launches += n; }

static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
// error reporting for the other translation units of the library (tame_align.cu)
int tame_set_error(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) return fail(TAME_ECUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
    } while (0)

extern const TameOps tame_ops_r1, tame_ops_r2, tame_ops_r3, tame_ops_r4, tame_ops_r5, tame_ops_r6, tame_ops_r7, tame_ops_r8;
const TameOps* tame_get_ops(int r) {
    static const TameOps* tab[] = {nullptr,      &tame_ops_r1, &tame_ops_r2, &tame_ops_r3, &tame_ops_r4,
                                   &tame_ops_r5, &tame_ops_r6, &tame_ops_r7, &tame_ops_r8};
    return (r >= 1 && r <= TAME_MAX_R) ? tab[r] : nullptr;
}

// ------------------------------------------------------------------------------------------------------
// NCCL, loaded lazily so that the single-GPU path has no dependency on it
// ------------------------------------------------------------------------------------------------------
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;
static int nccl_load() {
    if (g_nccl.lib) return TAME_OK;
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return fail(TAME_ENCCL, "cannot load libnccl.so.2: %s", dlerror());
#define SYM(field, name)                                                     \
    *(void**)(&g_nccl.field) = dlsym(lib, name);                             \
    if (!g_nccl.field) return fail(TAME_ENCCL, "libnccl lacks %s", name);
    SYM(GetUniqueId, "ncclGetUniqueId")
    SYM(CommInitRank, "ncclCommInitRank")
    SYM(CommDestroy, "ncclCommDestroy")
    SYM(Broadcast, "ncclBroadcast")
    SYM(AllReduce, "ncclAllReduce")
    SYM(GroupStart, "ncclGroupStart")
    SYM(GroupEnd, "ncclGroupEnd")
    SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
    g_nccl.lib = lib;
    return TAME_OK;
}
#define NK(call)                                                                                            \
    do {                                                                                                    \
        ncclResult_t r_ = (call);                                                                           \
        if (r_ != ncclSuccess) return fail(TAME_ENCCL, "%s:%d %s: %s", __FILE__, __LINE__, #call, g_nccl.GetErrorString(r_)); \
    } while (0)

// ------------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------------
struct tame_handle {
    tame_config cfg;
    const TameOps* ops = nullptr;
    int d = 0, nloc = 0, panel = 0;
    TameParams P{};
    cudaStream_t stream = nullptr;
    bool y_bound = false, state_bound = false, y_symmetric = false;
    bool y_f32 = false;                  // the bound Y is float (tame_bind_Y_f32): its kernels come from ops->f32
    const TameYOps& yops() const { return y_f32 ? ops->f32 : ops->f64; }
    bool skip_symcheck = false;          // tame_fit_batch's device-loop path: bind without the mirror check (and its sync)
    double* fit_scratch = nullptr;       // k_fit: per-block partial sums, control block, barrier counter
    int* sym_flag = nullptr;
    int* cursor = nullptr;
    // device scratch
    double *Craw = nullptr, *H = nullptr, *hab = nullptr, *tot = nullptr, *tot_partial = nullptr, *cst = nullptr;
    double *part_ll = nullptr, *part_cell = nullptr, *red6 = nullptr, *out6 = nullptr;
    int *progress = nullptr, *abort_flag = nullptr, *unit_counter = nullptr, *unit_done = nullptr;
    int epoch = 0, nparts = 1;
    int cap_n = 0, cap_T = 0;            // shape the buffers were sized for (tame_reconfigure accepts any n, T within it)
    bool fused = true, fused_multi = true;
    double2* hand = nullptr;
    void* peer_base[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // IPC mappings of the peers' hand buffers
    int npeers = 0;
    unsigned long long* dbg = nullptr;
    unsigned long long* trace = nullptr;
    int NS = 1, nb_ll = 0, nb_cell = 0;
    double* out6_pinned = nullptr;
    int* abort_pinned = nullptr;
    ncclComm_t comm = nullptr;
    // timing
    bool timing = false;
    std::vector<cudaEvent_t> ev;
    std::vector<int> ev_kind;   // kind of the interval that STARTS at event k (0 none,1 contract,2 chain,3 llmse)
    size_t ev_used = 0;
    double sweep_ms = 0, elbo_ms = 0, contract_ms = 0, chain_ms = 0, llmse_ms = 0;
};

static void ev_mark(tame_handle* h, int kind) {
    if (!h->timing) return;
    if (h->ev_used == h->ev.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->ev.push_back(e);
        h->ev_kind.push_back(0);
    }
    cudaEventRecord(h->ev[h->ev_used], h->stream);
    h->ev_kind[h->ev_used] = kind;
    ++h->ev_used;
}
// after a stream sync: fold the recorded intervals into the per-kind totals of the last iteration.
// kinds: 0 other (sweep side), 1 contract, 2 chain, 3 llmse, 4 sweep/ELBO boundary, 5 other (ELBO side)
static void ev_fold(tame_handle* h) {
    double sweep = 0, elbo = 0, contract = 0, chain = 0, llmse = 0;
    bool in_elbo = true;
    for (size_t k = 0; k < h->ev_used; ++k)
        if (h->ev_kind[k] == 4) in_elbo = false;   // a sweep was recorded: intervals before the boundary are its
    for (size_t k = 0; k + 1 < h->ev_used; ++k) {
        float ms = 0;
        cudaEventElapsedTime(&ms, h->ev[k], h->ev[k + 1]);
        const int kind = h->ev_kind[k];
        if (kind == 4) { in_elbo = true; continue; }
        (in_elbo ? elbo : sweep) += ms;
        if (kind == 1) contract += ms;
        if (kind == 2) chain += ms;
        if (kind == 3) llmse += ms;
    }
    h->ev_used = 0;
    h->sweep_ms = sweep; h->elbo_ms = elbo; h->contract_ms = contract; h->chain_ms = chain; h->llmse_ms = llmse;
}

// ------------------------------------------------------------------------------------------------------
// small non-templated kernels
// ------------------------------------------------------------------------------------------------------
// k_hab: sweep-invariant sums over partners, one pass over Y at bind time.
//   hab[i,t,0] = sum_{j!=i} p0*y0 + q*y1 ; hab[i,t,1] = sum_{j!=i} q*y0 + p1*y1   (structured_mf.py:324, rows a,b)
// grid (ceil(T/32), nloc), block (32, 8)
template <class YT>
__global__ void __launch_bounds__(256) k_hab(TameParams P) {
    const int lrow = blockIdx.y;
    const int i = tame_grow(lrow, P.panel, P.world, P.rank);
    const int t = blockIdx.x * 32 + threadIdx.x;
    const bool tv = t < P.T;
    double a0 = 0.0, a1 = 0.0;
    const YT* base = TameY<YT>::ptr(P) + ((size_t)lrow * P.n * P.T + (tv ? t : 0)) * 2;
    const size_t jstride = (size_t)P.T * 2;
    int j = threadIdx.y;
    for (; j + 24 < P.n; j += 32) {
        double2 y[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) y[u] = tv ? TameY<YT>::wide(TameY<YT>::ld_stream(base + (size_t)(j + 8 * u) * jstride)) : make_double2(0, 0);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (j + 8 * u != i) {
                a0 += P.p0 * y[u].x + P.q * y[u].y;
                a1 += P.q * y[u].x + P.p1 * y[u].y;
            }
        }
    }
    for (; j < P.n; j += 8) {
        if (tv && j != i) {
            double2 y = TameY<YT>::wide(TameY<YT>::ld_stream(base + (size_t)j * jstride));
            a0 += P.p0 * y.x + P.q * y.y;
            a1 += P.q * y.x + P.p1 * y.y;
        }
    }
    __shared__ double s0[8][33], s1[8][33];
    s0[threadIdx.y][threadIdx.x] = a0;
    s1[threadIdx.y][threadIdx.x] = a1;
    __syncthreads();
    if (threadIdx.y == 0 && tv) {
        double r0 = 0.0, r1 = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            r0 += s0[k][threadIdx.x];
            r1 += s1[k][threadIdx.x];
        }
        P.hab[((size_t)lrow * P.T + t) * 2 + 0] = r0;
        P.hab[((size_t)lrow * P.T + t) * 2 + 1] = r1;
    }
}

// Mirror check at bind time: Y[j,i,t,:] == swap(Y[i,j,t,:]) bit for bit for every i<j (the reference's generate_data
// writes both entries from one sample, temporal_ame.py:209-216; experiments may overwrite model.Y by hand).  Single GPU
// only (a rank holds only its own rows).  grid (ceil(T/32), n), block (32, 8); *flag is set to 1 on the first mismatch.
// Float Y is compared bit for bit as float.
template <class YT>
__global__ void __launch_bounds__(256) k_symcheck(TameParams P, int* flag) {
    const int i = blockIdx.y;
    const int t = blockIdx.x * 32 + threadIdx.x;
    if (t >= P.T) return;
    bool bad = false;
    for (int j = i + 1 + threadIdx.y; j < P.n; j += 8) {
        const auto a = TameY<YT>::ld_stream(TameY<YT>::ptr(P) + (((size_t)i * P.n + j) * P.T + t) * 2);
        const auto b = TameY<YT>::ld_stream(TameY<YT>::ptr(P) + (((size_t)j * P.n + i) * P.T + t) * 2);
        bad |= (TameY<YT>::bits(a.x) != TameY<YT>::bits(b.y)) || (TameY<YT>::bits(a.y) != TameY<YT>::bits(b.x));
    }
    if (bad) *flag = 1;
}

// Mirror check across ranks: a rank only holds its own rows, so the pair (Y[i,j], Y[j,i]) is split between two ranks.
// Every entry contributes a signed 64-bit hash of (unordered dyad, t, value as seen from the lower index): +h for i<j,
// -h of the swapped value for i>j; the wrap-around sum over ALL ranks (NCCL all-reduce) is 0 when every dyad is
// mirror-consistent and non-zero otherwise, up to a 2^-64 collision probability.  grid (ceil(T/32), nloc), block (32,8).
__device__ __forceinline__ unsigned long long tame_mix64(unsigned long long x) {
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull; x ^= x >> 27; x *= 0x94d049bb133111ebull; x ^= x >> 31;
    return x;
}
template <class YT>
__global__ void __launch_bounds__(256) k_symhash(TameParams P, unsigned long long* acc) {
    const int lrow = blockIdx.y;
    const int i = tame_grow(lrow, P.panel, P.world, P.rank);
    const int t = blockIdx.x * 32 + threadIdx.x;
    unsigned long long sum = 0;
    if (t < P.T) {
        for (int j = threadIdx.y; j < P.n; j += 8) {
            if (j == i) continue;
            const auto y = TameY<YT>::ld_stream(TameY<YT>::ptr(P) + (((size_t)lrow * P.n + j) * P.T + t) * 2);
            const int lo = min(i, j), hi = max(i, j);
            const unsigned long long key = ((unsigned long long)lo * P.n + hi) * (unsigned long long)P.T + t;
            const unsigned long long a = TameY<YT>::bits(i < j ? y.x : y.y);   // y_{lo,hi}
            const unsigned long long b = TameY<YT>::bits(i < j ? y.y : y.x);   // y_{hi,lo}
            const unsigned long long h = tame_mix64(tame_mix64(key ^ 0x9e3779b97f4a7c15ull) ^ tame_mix64(a) ^ (tame_mix64(b) * 3ull));
            sum += (i < j) ? h : (0ull - h);
        }
    }
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (threadIdx.x == 0) atomicAdd(acc, sum);
}

// red6 = {sq, quad, lp0, lpt, ent, tr}: deterministic two-level sum of the per-block partials
__global__ void __launch_bounds__(256) k_reduce6(const double* part_ll, int nb_ll, const double* part_cell, int nb_cell,
                                                 double* red6) {
    __shared__ double sh[6][256];
    double a[6] = {0, 0, 0, 0, 0, 0};
    for (int b = threadIdx.x; b < nb_ll; b += 256) {
        a[0] += part_ll[(size_t)b * 2 + 0];
        a[1] += part_ll[(size_t)b * 2 + 1];
    }
    for (int b = threadIdx.x; b < nb_cell; b += 256) {
#pragma unroll
        for (int k = 0; k < 4; ++k) a[2 + k] += part_cell[(size_t)b * 4 + k];
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) sh[k][threadIdx.x] = a[k];
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) {
#pragma unroll
            for (int k = 0; k < 6; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + s];
        }
        __syncthreads();
    }
    if (threadIdx.x < 6) red6[threadIdx.x] = sh[threadIdx.x][0];
}

// out6 = {ELBO, LL, LP0, LPT, H, MSE} from the (all-reduced) sums.
//   LL = -1/2 [ quad + npairs*T*(logdet R + 2 log 2pi) + (SMF) 0.1 * tr(R^-1)/d * (n-1) * sum_{i,t} tr X_cov[i,t] ]
//        structured_mf.py:124-150 (naive_mf.py:114-132 has no trace term); closed form per SURVEY.md appendix A.
//   MSE = sq / (n (n-1) T)                                                  temporal_ame.py:287-290
__global__ void k_finalize(const double* red6, int n, int T, int d, int mode, double p0, double p1, double logdetR,
                           double* out6) {
    const double LOG2PI = 1.8378770664093454835606594728112;
    const double npairs = 0.5 * (double)n * (double)(n - 1);
    double ll = red6[1] + npairs * (double)T * (logdetR + 2.0 * LOG2PI);
    if (mode != 0) ll += 0.1 * (p0 + p1) / (double)d * (double)(n - 1) * red6[5];
    ll *= -0.5;
    out6[1] = ll;
    out6[2] = red6[2];
    out6[3] = red6[3];
    out6[4] = red6[4];
    out6[0] = ((ll + red6[2]) + red6[3]) + red6[4];   // elbo += LL; += LP0; += LPT; += H   (structured_mf.py:117-121)
    out6[5] = red6[0] / ((double)n * (double)(n - 1) * (double)T);
}

// Y generator, one thread per (local row, partner, time).  temporal_ame.py:200-216 in distribution.  FP64 throughout; a
// float Y gets each value rounded once when it is stored (both halves of a dyad round the same double: mirror-consistent).
template <class YT>
__global__ void __launch_bounds__(256) k_generate(int n, int T, int r, double l00, double l10, double l11,
                                                  const double* __restrict__ X, unsigned long long seed, int row_begin,
                                                  int row_end, YT* __restrict__ Y) {
    const int D = 2 + 2 * r;
    const size_t total = (size_t)(row_end - row_begin) * n * T;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        const int t = (int)(idx % T);
        const int j = (int)((idx / T) % n);
        const int i = row_begin + (int)(idx / ((size_t)T * n));
        double y0 = 0.0, y1 = 0.0;
        if (i != j) {
            const int lo = min(i, j), hi = max(i, j);
            curandStatePhilox4_32_10_t st;
            curand_init(seed, ((unsigned long long)lo * n + hi) * (unsigned long long)T + t, 0, &st);
            const double2 z = curand_normal2_double(&st);
            const double e0 = l00 * z.x, e1 = l10 * z.x + l11 * z.y;     // (y_lo,hi ; y_hi,lo) noise
            const double* xi = X + ((size_t)i * T + t) * D;
            const double* xj = X + ((size_t)j * T + t) * D;
            double uv = 0.0, vu = 0.0;
            for (int a = 0; a < r; ++a) {
                uv = fma(xi[2 + a], xj[2 + r + a], uv);   // U_i . V_j
                vu = fma(xj[2 + a], xi[2 + r + a], vu);   // U_j . V_i
            }
            const double mu_ij = xi[0] + xj[1] + uv, mu_ji = xj[0] + xi[1] + vu;
            y0 = mu_ij + (i < j ? e0 : e1);
            y1 = mu_ji + (i < j ? e1 : e0);
        }
        Y[idx * 2 + 0] = (YT)y0;
        Y[idx * 2 + 1] = (YT)y1;
    }
}

// ------------------------------------------------------------------------------------------------------
// host helpers
// ------------------------------------------------------------------------------------------------------
static void matmul(const double* A, const double* B, double* C, int d, bool transA) {
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) {
            double s = 0.0;
            for (int k = 0; k < d; ++k) s += (transA ? A[k * d + i] : A[i * d + k]) * B[k * d + j];
            C[i * d + j] = s;
        }
}

static std::vector<double> constant_block(const tame_config* cfg, int d) {
    std::vector<double> c(6 * d * d);
    memcpy(&c[0], cfg->S0inv, sizeof(double) * d * d);
    memcpy(&c[d * d], cfg->Qinv, sizeof(double) * d * d);
    matmul(cfg->Qinv, cfg->Phi, &c[3 * d * d], d, false);          // Qinv Phi
    matmul(cfg->Phi, &c[3 * d * d], &c[2 * d * d], d, true);       // Phi' (Qinv Phi)      structured_mf.py:262
    matmul(cfg->Phi, cfg->Qinv, &c[4 * d * d], d, true);           // Phi' Qinv            structured_mf.py:264
    memcpy(&c[5 * d * d], cfg->Phi, sizeof(double) * d * d);
    return c;
}

// shape-dependent launch parameters of a handle (shared by tame_create and tame_reconfigure)
static int shape_nparts(int n) {
    int np = (n >= 512) ? 4 : (n >= 192 ? 2 : 1);
    if (const char* v = getenv("TAME_NPARTS")) np = std::max(1, std::min(TAME_MAX_PARTS, atoi(v)));
    return np;
}
static int shape_ns(int n) { return std::max(1, std::min(64, (n + 127) / 128)); }

// Point an existing single-GPU handle at another fit with the same r and device and a shape (n, T) within the one its
// buffers were sized for: new hyper-parameters, mode and learning rate; Y and the state are bound afresh by the caller.
// tame_fit_batch pools its handles with this (a handle is ~25 device / pinned allocations -- milliseconds on the host, and
// cudaFree synchronises the whole device).  Stale hand-over tags and unit stamps of earlier fits cannot be mistaken for
// current ones: they carry the handle's epoch, which only grows.
static int tame_reconfigure(tame_handle* h, const tame_config* cfg) {
    if (cfg->r != h->cfg.r || cfg->device != h->cfg.device || cfg->world != 1 || h->P.world != 1)
        return fail(TAME_EINVAL, "tame_reconfigure: latent dimension / device mismatch");
    if (cfg->n < 2 || cfg->T < 1 || cfg->n > h->cap_n || cfg->T > h->cap_T)
        return fail(TAME_EINVAL, "tame_reconfigure: shape (%d, %d) outside the handle's capacity (%d, %d)", cfg->n, cfg->T, h->cap_n, h->cap_T);
    if (cfg->mode < 0 || cfg->mode > 2) return fail(TAME_EINVAL, "unknown mode %d", cfg->mode);
    if (!cfg->Phi || !cfg->Qinv || !cfg->S0inv) return fail(TAME_EINVAL, "Phi/Qinv/S0inv must be given");
    CK(cudaSetDevice(h->cfg.device));
    const std::vector<double> c = constant_block(cfg, h->d);
    if (cfg->n != h->P.n || cfg->T != h->P.T) {
        const int n = cfg->n, T = cfg->T;
        h->nloc = n;
        h->NS = shape_ns(n);
        h->nparts = shape_nparts(n);
        h->P.n = n; h->P.T = T; h->P.nloc = n; h->P.nparts = h->nparts;
        h->P.probe_t = T - 1;
        if (const char* v = getenv("TAME_PROBE_T")) h->P.probe_t = std::max(0, std::min(T - 1, atoi(v)));
        const char* v = getenv("TAME_SWEEP");
        h->fused = !(v && strcmp(v, "panel") == 0) && (T + TAME_CHAIN_WPC - 1) / TAME_CHAIN_WPC + 1 <= h->ops->f64.sweep_capacity(1);
        h->nb_ll = h->ops->llmse_blocks(h->P);
        h->nb_cell = h->ops->cellterms_blocks(h->P);
    }
    h->cfg = *cfg;
    h->cfg.Phi = h->cfg.Qinv = h->cfg.S0inv = nullptr;
    // `c` is pageable host memory: the runtime stages it before cudaMemcpyAsync returns, the copy itself is stream-ordered
    CK(cudaMemcpyAsync(h->cst, c.data(), sizeof(double) * c.size(), cudaMemcpyHostToDevice, h->stream));
    TameParams& P = h->P;
    P.mode = cfg->mode;
    P.lr = cfg->lr;
    P.p0 = cfg->Rinv[0]; P.p1 = cfg->Rinv[3]; P.q = 0.5 * (cfg->Rinv[1] + cfg->Rinv[2]);
    P.Y = nullptr; P.Xm = nullptr; P.Xc = nullptr;
    h->y_bound = h->state_bound = h->y_symmetric = false;
    return TAME_OK;
}

// tame_bind_Y / tame_bind_Y_f32: the handle remembers the element type, every later launch takes that type's kernels
template <class YT>
static int bind_Y(tame_handle* h, const YT* Y) {
    if (!h || !Y) return fail(TAME_EINVAL, "null argument");
    CK(cudaSetDevice(h->cfg.device));
    h->P.Y = Y;
    h->y_f32 = std::is_same<YT, float>::value;
    dim3 grid((h->P.T + 31) / 32, h->nloc), block(32, 8);
    k_hab<YT><<<grid, block, 0, h->stream>>>(h->P);
    tame_count_launch(1);
    CK(cudaGetLastError());
    // mirror property of Y (single GPU): lets the ELBO/MSE pass stream only the i<j half.  TAME_SYMMETRIC=0 disables.
    h->y_symmetric = false;
    const char* sv = getenv("TAME_SYMMETRIC");
    if (h->skip_symcheck) { h->y_bound = true; return TAME_OK; }
    if (h->P.world == 1 && !(sv && atoi(sv) == 0)) {
        CK(cudaMemsetAsync(h->sym_flag, 0, sizeof(int), h->stream));
        k_symcheck<YT><<<grid, block, 0, h->stream>>>(h->P, h->sym_flag);
        tame_count_launch(1);
        int bad = 1;
        CK(cudaMemcpyAsync(&bad, h->sym_flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        h->y_symmetric = (bad == 0);
    }
    if (h->P.world > 1 && h->comm && !(sv && atoi(sv) == 0)) {
        // multi-GPU: signed hash sum over every rank's rows (needs tame_comm_init before tame_bind_Y)
        unsigned long long* acc = nullptr;
        CK(cudaMalloc((void**)&acc, sizeof(unsigned long long)));
        CK(cudaMemsetAsync(acc, 0, sizeof(unsigned long long), h->stream));
        k_symhash<YT><<<grid, block, 0, h->stream>>>(h->P, acc);
        tame_count_launch(1);
        NK(g_nccl.AllReduce(acc, acc, 1, ncclUint64, ncclSum, h->comm, h->stream));
        unsigned long long total = 1;
        CK(cudaMemcpyAsync(&total, acc, sizeof(total), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        cudaFree(acc);
        h->y_symmetric = (total == 0ull);
    }
    h->y_bound = true;
    return TAME_OK;
}

template <class YT>
static int generate_Y(int32_t n, int32_t T, int32_t r, const double R[4], const double* X_dev, uint64_t seed,
                      int32_t row_begin, int32_t row_end, YT* Y_dev, void* stream) {
    if (!R || !X_dev || !Y_dev || row_begin < 0 || row_end > n || row_end < row_begin) return fail(TAME_EINVAL, "bad argument");
    if (R[0] <= 0) return fail(TAME_EINVAL, "R must be positive definite");
    const double l00 = std::sqrt(R[0]), l10 = R[2] / l00, l11sq = R[3] - l10 * l10;
    if (l11sq <= 0) return fail(TAME_EINVAL, "R must be positive definite");
    const size_t total = (size_t)(row_end - row_begin) * n * T;
    if (total == 0) return TAME_OK;
    const int blocks = (int)std::min<size_t>((total + 255) / 256, 148 * 64);
    k_generate<YT><<<blocks, 256, 0, (cudaStream_t)stream>>>(n, T, r, l00, l10, std::sqrt(l11sq), X_dev, seed, row_begin, row_end, Y_dev);
    tame_count_launch(1);
    CK(cudaGetLastError());
    return TAME_OK;
}

extern "C" {

const char* tame_version(void) { return "tame_b200 0.1.0 (sm_100a, fp64)"; }
const char* tame_last_error(void) { return g_err.c_str(); }
int64_t tame_launch_count(void) { return g_launches.load(); }

int tame_create(const tame_config* cfg, tame_handle** out) {
    if (!cfg || !out) return fail(TAME_EINVAL, "null argument");
    if (cfg->n < 2 || cfg->T < 1) return fail(TAME_EINVAL, "need n >= 2 and T >= 1 (got n=%d T=%d)", cfg->n, cfg->T);
    if (cfg->r < 1 || cfg->r > TAME_MAX_R) return fail(TAME_EINVAL, "latent_dim r=%d unsupported (1..%d)", cfg->r, TAME_MAX_R);
    if (cfg->mode < 0 || cfg->mode > 2) return fail(TAME_EINVAL, "unknown mode %d", cfg->mode);
    if (!cfg->Phi || !cfg->Qinv || !cfg->S0inv) return fail(TAME_EINVAL, "Phi/Qinv/S0inv must be given");
    if (cfg->world < 1 || cfg->rank < 0 || cfg->rank >= cfg->world) return fail(TAME_EINVAL, "bad world/rank %d/%d", cfg->world, cfg->rank);
    int panel = cfg->panel > 0 ? cfg->panel : TAME_WIN;
    if (panel % TAME_WIN) return fail(TAME_EINVAL, "panel must be a multiple of %d", TAME_WIN);
    CK(cudaSetDevice(cfg->device));
    tame_handle* h = new tame_handle();
    h->cfg = *cfg;
    h->ops = tame_get_ops(cfg->r);
    h->d = 2 + 2 * cfg->r;
    h->panel = panel;
    const int n = cfg->n, T = cfg->T, d = h->d, world = cfg->world, rank = cfg->rank;
    // rows owned: panels b with b % world == rank
    int nloc = 0;
    for (int b = 0; b * panel < n; ++b)
        if (b % world == rank) nloc += std::min(panel, n - b * panel);
    if (world > 1 && n % panel) { delete h; return fail(TAME_EINVAL, "multi-GPU needs n %% panel == 0 (n=%d panel=%d)", n, panel); }
    h->nloc = nloc;
    if (T > h->ops->chain_max_T()) { delete h; return fail(TAME_EINVAL, "T=%d exceeds the co-resident capacity of the chain kernel", T); }

    // constant matrices: S0inv, Qinv, Phi'QinvPhi, QinvPhi, Phi'Qinv, Phi
    std::vector<double> c = constant_block(cfg, d);
    h->cfg.Phi = h->cfg.Qinv = h->cfg.S0inv = nullptr;             // host pointers are not retained

    const int TOT = h->ops->tot;
    h->NS = shape_ns(n);
    h->cap_n = n; h->cap_T = T;
    auto dalloc = [&](void** p, size_t bytes) { return cudaMalloc(p, std::max<size_t>(bytes, 16)); };
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = dalloc((void**)&h->cst, sizeof(double) * c.size());
    // column parts per streaming unit: split the (long) upper part so that the first sub-blocks are ready early
    h->nparts = shape_nparts(n);
    if (e == cudaSuccess) e = dalloc((void**)&h->H, sizeof(double) * (size_t)nloc * T * 2 * cfg->r * h->nparts);
    if (e == cudaSuccess) e = dalloc((void**)&h->Craw, sizeof(double) * (size_t)nloc * T * d * d);
    if (e == cudaSuccess) e = dalloc((void**)&h->hab, sizeof(double) * (size_t)nloc * T * 2);
    if (e == cudaSuccess) e = dalloc((void**)&h->tot, sizeof(double) * (size_t)T * TOT);
    if (e == cudaSuccess) e = dalloc((void**)&h->tot_partial, sizeof(double) * (size_t)T * h->NS * TOT);
    if (e == cudaSuccess) e = dalloc((void**)&h->progress, sizeof(int) * T);
    if (e == cudaSuccess) e = dalloc((void**)&h->abort_flag, sizeof(int));
    if (e == cudaSuccess) e = dalloc((void**)&h->sym_flag, sizeof(int));
    if (e == cudaSuccess) e = dalloc((void**)&h->cursor, sizeof(int) * TAME_MAX_PARTS);
    const size_t nunits = (size_t)((n + TAME_SB - 1) / TAME_SB) * ((T + 31) / 32);
    if (e == cudaSuccess) e = dalloc((void**)&h->unit_counter, sizeof(int));
    if (e == cudaSuccess) e = dalloc((void**)&h->dbg, sizeof(unsigned long long) * 16);
    if (getenv("TAME_TRACE")) {
        const size_t nb = sizeof(unsigned long long) * 22 * ((n + TAME_SB - 1) / TAME_SB);
        if (e == cudaSuccess) e = dalloc((void**)&h->trace, nb);
        if (e == cudaSuccess) e = cudaMemset(h->trace, 0, nb);
    }
    if (e == cudaSuccess) e = dalloc((void**)&h->hand, sizeof(double2) * (size_t)n * T * d);
    if (e == cudaSuccess) e = dalloc((void**)&h->unit_done, sizeof(int) * nunits * h->nparts * TAME_NG);
    if (e == cudaSuccess) e = dalloc((void**)&h->red6, sizeof(double) * 6);
    if (e == cudaSuccess) e = dalloc((void**)&h->fit_scratch, sizeof(double) * (FIT_PART_DOUBLES + 8));
    if (e == cudaSuccess) e = dalloc((void**)&h->out6, sizeof(double) * 6);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&h->out6_pinned, sizeof(double) * 6);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&h->abort_pinned, sizeof(int));
    if (e != cudaSuccess) { tame_destroy(h); return fail(TAME_ENOMEM, "allocation failed: %s", cudaGetErrorString(e)); }
    CK(cudaMemcpy(h->cst, c.data(), sizeof(double) * c.size(), cudaMemcpyHostToDevice));
    CK(cudaMemset(h->progress, 0, sizeof(int) * T));
    CK(cudaMemset(h->abort_flag, 0, sizeof(int)));
    CK(cudaMemset(h->unit_counter, 0, sizeof(int)));
    CK(cudaMemset(h->cursor, 0, sizeof(int) * TAME_MAX_PARTS));
    CK(cudaMemset(h->dbg, 0, sizeof(unsigned long long) * 16));
    CK(cudaMemset(h->hand, 0, sizeof(double2) * (size_t)n * T * d));
    CK(cudaMemset(h->unit_done, 0, sizeof(int) * nunits * h->nparts * TAME_NG));
    {
        const char* v = getenv("TAME_SWEEP");   // "panel" forces the stream-ordered per-panel path (debug / comparison)
        h->fused = (world == 1) && !(v && strcmp(v, "panel") == 0);
        h->fused_multi = !(v && strcmp(v, "panel") == 0);
        // the element type of Y is not known yet: the double instantiation is the binding one (the float one has the same
        // launch bounds and a smaller shared-memory footprint, so at least its capacity)
        if (h->fused && (T + TAME_CHAIN_WPC - 1) / TAME_CHAIN_WPC + 1 > h->ops->f64.sweep_capacity(1)) h->fused = false;
    }

    TameParams& P = h->P;
    P.n = n; P.T = T; P.nloc = nloc; P.world = world; P.rank = rank; P.panel = panel; P.mode = cfg->mode;
    P.lr = cfg->lr;
    P.p0 = cfg->Rinv[0]; P.p1 = cfg->Rinv[3]; P.q = 0.5 * (cfg->Rinv[1] + cfg->Rinv[2]);
    P.Craw = h->Craw; P.H = h->H; P.hab = h->hab; P.tot = h->tot; P.cst = h->cst; P.progress = h->progress; P.abort_flag = h->abort_flag;
    P.unit_counter = h->unit_counter; P.unit_done = h->unit_done; P.epoch = 0; P.n_chain_ctas = 0; P.hand = h->hand; P.dbg = h->dbg; P.trace = h->trace; P.nparts = h->nparts; P.cursor = h->cursor; P.npeers = 0;
    P.deterministic = 0;
    if (const char* v = getenv("TAME_DETERMINISTIC")) P.deterministic = atoi(v) ? 1 : 0;
    P.probe_t = T - 1;
    if (const char* v = getenv("TAME_PROBE_T")) P.probe_t = std::max(0, std::min(T - 1, atoi(v)));
    for (int k = 0; k < 7; ++k) P.hand_peer[k] = nullptr;
    // the zeroed hand-over slots / stamps must be in place before the first kernel on the handle's (possibly non-blocking)
    // stream, and -- multi-GPU -- before any peer can write into them
    if (world > 1) CK(cudaDeviceSynchronize());
    else CK(cudaStreamSynchronize(cudaStreamLegacy));

    h->nb_ll = h->ops->llmse_blocks(P);
    h->nb_cell = h->ops->cellterms_blocks(P);
    e = dalloc((void**)&h->part_ll, sizeof(double) * 2 * (size_t)h->nb_ll);
    if (e == cudaSuccess) e = dalloc((void**)&h->part_cell, sizeof(double) * 4 * (size_t)h->nb_cell);
    if (e != cudaSuccess) { tame_destroy(h); return fail(TAME_ENOMEM, "allocation failed: %s", cudaGetErrorString(e)); }
    *out = h;
    return TAME_OK;
}

int tame_destroy(tame_handle* h) {
    if (!h) return TAME_OK;
    cudaSetDevice(h->cfg.device);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    for (int k = 0; k < h->npeers; ++k) if (h->peer_base[k]) cudaIpcCloseMemHandle(h->peer_base[k]);
    for (void* p : {(void*)h->Craw, (void*)h->H, (void*)h->hab, (void*)h->tot, (void*)h->tot_partial, (void*)h->cst, (void*)h->part_ll,
                    (void*)h->part_cell, (void*)h->red6, (void*)h->out6, (void*)h->progress, (void*)h->abort_flag,
                    (void*)h->unit_counter, (void*)h->unit_done, (void*)h->hand, (void*)h->dbg, (void*)h->trace, (void*)h->fit_scratch, (void*)h->sym_flag, (void*)h->cursor})
        if (p) cudaFree(p);
    if (h->out6_pinned) cudaFreeHost(h->out6_pinned);
    if (h->abort_pinned) cudaFreeHost(h->abort_pinned);
    for (auto e : h->ev) cudaEventDestroy(e);
    delete h;
    return TAME_OK;
}

int tame_set_stream(tame_handle* h, void* s) {
    if (!h) return fail(TAME_EINVAL, "null handle");
    h->stream = (cudaStream_t)s;
    return TAME_OK;
}

int tame_y_symmetric(const tame_handle* h) { return (h && h->y_symmetric) ? 1 : 0; }

int tame_local_rows(const tame_handle* h, int32_t* out) {
    if (!h || !out) return fail(TAME_EINVAL, "null argument");
    *out = h->nloc;
    return TAME_OK;
}

int tame_bind_Y(tame_handle* h, const double* Y) { return bind_Y<double>(h, Y); }
int tame_bind_Y_f32(tame_handle* h, const float* Y) { return bind_Y<float>(h, Y); }

int tame_bind_state(tame_handle* h, double* Xm, double* Xc) {
    if (!h || !Xm || !Xc) return fail(TAME_EINVAL, "null argument");
    h->P.Xm = Xm;
    h->P.Xc = Xc;
    h->state_bound = true;
    return TAME_OK;
}

static int check_abort(tame_handle* h) {
    // called after a stream synchronisation
    if (*h->abort_pinned) {
        cudaMemset(h->abort_flag, 0, sizeof(int));
        *h->abort_pinned = 0;
        return fail(TAME_EHANG, "the chain kernel's watchdog fired (a time-step warp never saw its predecessor's progress)");
    }
    return TAME_OK;
}

int tame_sweep(tame_handle* h) {
    if (!h) return fail(TAME_EINVAL, "null handle");
    if (!h->y_bound || !h->state_bound) return fail(TAME_ESTATE, "tame_sweep before tame_bind_Y/tame_bind_state");
    CK(cudaSetDevice(h->cfg.device));
    const TameParams& P = h->P;
    const TameOps* ops = h->ops;
    const TameYOps& yops = h->yops();
    const int n = P.n, T = P.T, d = h->d, world = P.world, rank = P.rank;
    cudaStream_t st = h->stream;
    ev_mark(h, 0);
    // running totals of the partner moments from the current means; resets the progress counters
    ops->totals(P, h->tot_partial, h->NS, st);
    ev_mark(h, 1);
    h->P.epoch = ++h->epoch;   // stamps of this sweep (hand-over tags, unit_done)
    if (h->fused || (world > 1 && h->npeers == world - 1 && h->fused_multi)) {
        // single GPU: the whole sweep is one persistent cooperative launch (chain CTAs + streaming CTAs)
        ev_mark(h, 2);
        cudaError_t e = yops.sweep_fused(h->P, st);
        if (e != cudaSuccess) return fail(TAME_ECUDA, "fused sweep launch: %s", cudaGetErrorString(e));
        ev_mark(h, 0);
    } else {
        // static upper part: partners j > k still carry their old means when row k is updated
        yops.contract(P, 0, n, 0, n, /*tri=*/1, /*accumulate=*/0, st);
        ev_mark(h, 0);
        for (int lo = 0; lo < n; lo += TAME_WIN) {
            const int hi = std::min(n, lo + TAME_WIN);
            const int owner = (lo / h->panel) % world;
            if (owner == rank) {
                ev_mark(h, 2);
                cudaError_t e = yops.chain(P, lo, hi, st);
                if (e != cudaSuccess) return fail(TAME_ECUDA, "chain launch: %s", cudaGetErrorString(e));
                ev_mark(h, 0);
            }
            if (world > 1) {
                if (!h->comm) return fail(TAME_ESTATE, "world > 1 but tame_comm_init was not called");
                NK(g_nccl.GroupStart());
                NK(g_nccl.Broadcast(P.Xm + (size_t)lo * T * d, P.Xm + (size_t)lo * T * d, (size_t)(hi - lo) * T * d, ncclDouble, owner, h->comm, st));
                NK(g_nccl.Broadcast(P.tot, P.tot, (size_t)T * ops->tot, ncclDouble, owner, h->comm, st));
                NK(g_nccl.GroupEnd());
            }
            if (hi < n) {
                // right-looking push: the block's new means reach every later row
                ev_mark(h, 1);
                yops.contract(P, hi, n, lo, hi, /*tri=*/0, /*accumulate=*/1, st);
                ev_mark(h, 0);
            }
        }
    }
    ops->covblend(h->P, st);   // factorisation rule + damped write of the covariance blocks (chain -> Craw -> X_cov)
    ev_mark(h, 4);   // end of the sweep; folded at the next synchronisation (tame_elbo_mse)
    CK(cudaGetLastError());
    return TAME_OK;
}

int tame_elbo_mse(tame_handle* h, double* out6_host) {
    if (!h || !out6_host) return fail(TAME_EINVAL, "null argument");
    if (!h->y_bound || !h->state_bound) return fail(TAME_ESTATE, "tame_elbo_mse before tame_bind_Y/tame_bind_state");
    CK(cudaSetDevice(h->cfg.device));
    const TameParams& P = h->P;
    cudaStream_t st = h->stream;
    int nb = 0;
    ev_mark(h, 3);
    h->yops().llmse(P, h->part_ll, &nb, h->y_symmetric ? 1 : 0, st);
    ev_mark(h, 0);
    h->ops->cellterms(P, h->cfg.logdet_S0, h->cfg.logdet_Q, h->part_cell, h->nb_cell, st);
    k_reduce6<<<1, 256, 0, st>>>(h->part_ll, nb, h->part_cell, h->nb_cell, h->red6);
    if (P.world > 1) {
        if (!h->comm) return fail(TAME_ESTATE, "world > 1 but tame_comm_init was not called");
        NK(g_nccl.AllReduce(h->red6, h->red6, 6, ncclDouble, ncclSum, h->comm, st));
    }
    k_finalize<<<1, 1, 0, st>>>(h->red6, P.n, P.T, h->d, P.mode, P.p0, P.p1, h->cfg.logdet_R, h->out6);
    tame_count_launch(2);
    ev_mark(h, 0);
    CK(cudaMemcpyAsync(h->out6_pinned, h->out6, sizeof(double) * 6, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h->abort_pinned, h->abort_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (h->timing) ev_fold(h);
    memcpy(out6_host, h->out6_pinned, sizeof(double) * 6);
    return check_abort(h);
}

int tame_iterate(tame_handle* h, double* out6_host) {
    int rc = tame_sweep(h);
    if (rc != TAME_OK) return rc;
    return tame_elbo_mse(h, out6_host);
}

int tame_fit(tame_handle* h, int32_t max_iter, double tolerance, double* elbo_trace, double* mse_trace, int32_t* n_done) {
    if (!h || !n_done) return fail(TAME_EINVAL, "null argument");
    // base.py:166-203
    int patience = 0;
    double prev = -INFINITY;
    *n_done = 0;
    for (int it = 0; it < max_iter; ++it) {
        double o[6];
        int rc = tame_iterate(h, o);
        if (rc != TAME_OK) return rc;
        if (elbo_trace) elbo_trace[it] = o[0];
        if (mse_trace) mse_trace[it] = o[5];
        *n_done = it + 1;
        bool converged = false;
        if (it > 0) {
            const double rel = std::fabs(o[0] - prev) / (std::fabs(prev) + 1e-8);
            patience = (rel < tolerance) ? patience + 1 : 0;
            converged = patience >= 3;
        }
        prev = o[0];
        if (converged) break;
    }
    return TAME_OK;
}

int tame_fit_device(tame_handle* h, int32_t max_iter, double tolerance, double* elbo_dev, double* mse_dev, int32_t* n_done_dev) {
    if (!h || !elbo_dev || !mse_dev || !n_done_dev) return fail(TAME_EINVAL, "null argument");
    if (!h->y_bound || !h->state_bound) return fail(TAME_ESTATE, "tame_fit_device before tame_bind_Y/tame_bind_state");
    if (h->P.world != 1 || !h->fused) return fail(TAME_EINVAL, "tame_fit_device needs the single-GPU fused sweep");
    if (max_iter <= 0) return fail(TAME_EINVAL, "max_iter must be positive");
    CK(cudaSetDevice(h->cfg.device));
    if (h->yops().fit_grid(h->P) > 1024) return fail(TAME_EINVAL, "problem too large for the whole-fit kernel");
    cudaStream_t st = h->stream;
    CK(cudaMemsetAsync(h->fit_scratch + FIT_PART_DOUBLES, 0, sizeof(double) * 8, st));      // ctl[0..2], barrier counter
    CK(cudaMemsetAsync(n_done_dev, 0, sizeof(int32_t), st));
    TameFitArgs F;
    F.max_iter = max_iter;
    F.tolerance = tolerance;
    F.logdetS0 = h->cfg.logdet_S0; F.logdetQ = h->cfg.logdet_Q; F.logdetR = h->cfg.logdet_R;
    F.elbo_trace = elbo_dev; F.mse_trace = mse_dev; F.n_done = n_done_dev;
    F.part = h->fit_scratch;
    F.ctl = h->fit_scratch + FIT_PART_DOUBLES;
    F.bar = reinterpret_cast<unsigned int*>(h->fit_scratch + FIT_PART_DOUBLES + 4);
    h->P.epoch = h->epoch;               // iteration `it` of the kernel stamps with epoch + it + 1
    cudaError_t e = h->yops().fit_device(h->P, F, nullptr, st);
    h->epoch += max_iter;
    h->P.epoch = h->epoch;
    if (e != cudaSuccess) return fail(TAME_ECUDA, "whole-fit kernel launch: %s", cudaGetErrorString(e));
    return TAME_OK;
}

}  // extern "C"

static constexpr int BATCH_FALLBACK = 1;      // internal: the device-loop path declined before doing any work
// tame_fit_batch, device-loop path: every fit is ONE cooperative launch of k_fit (all its iterations and its stop rule on
// the device), queued round-robin on a few streams from this one host thread; nothing comes back to the host until the end.
template <class YT>
static int fit_batch_device(int32_t n_fits, const tame_config* cfgs, const YT* const* Y_dev, double* const* Xm_dev,
                            double* const* Xc_dev, int32_t max_iter, double tolerance, double* elbo_traces, double* mse_traces,
                            int32_t* n_done, int32_t n_streams) {
    if (n_streams <= 0) {
        const char* v = getenv("TAME_BATCH_STREAMS");
        n_streams = v ? atoi(v) : 16;
    }
    const int S = std::max(1, std::min(n_streams <= 0 ? 16 : n_streams, n_fits));
    const int dev0 = cfgs[0].device;
    CK(cudaSetDevice(dev0));
    std::vector<cudaStream_t> streams(S, nullptr);
    std::vector<std::vector<tame_handle*>> pool(S);
    double *el_d = nullptr, *ms_d = nullptr;
    int32_t* nd_d = nullptr;
    int rc = TAME_OK;
    auto cleanup = [&]() {
        std::string keep = g_err;
        for (auto& v : pool) for (tame_handle* q : v) tame_destroy(q);
        for (cudaStream_t s : streams) if (s) cudaStreamDestroy(s);
        cudaFree(el_d); cudaFree(ms_d); cudaFree(nd_d);
        g_err = keep;
    };
    cudaError_t e = cudaMalloc((void**)&el_d, sizeof(double) * (size_t)n_fits * max_iter);
    if (e == cudaSuccess) e = cudaMalloc((void**)&ms_d, sizeof(double) * (size_t)n_fits * max_iter);
    if (e == cudaSuccess) e = cudaMalloc((void**)&nd_d, sizeof(int32_t) * (size_t)n_fits);
    for (int s = 0; s < S && e == cudaSuccess; ++s) e = cudaStreamCreateWithFlags(&streams[s], cudaStreamNonBlocking);
    if (e != cudaSuccess) { cleanup(); return fail(TAME_ENOMEM, "tame_fit_batch set-up: %s", cudaGetErrorString(e)); }
    // largest fits first (a fit's cost grows with n * T; the stable sort keeps equal shapes adjacent for the handle pools):
    // the small ones fill the SMs the last large ones leave idle
    std::vector<int> order(n_fits);
    for (int f = 0; f < n_fits; ++f) order[f] = f;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        return (long)cfgs[a].n * cfgs[a].T > (long)cfgs[b].n * cfgs[b].T;
    });
    // one handle per (stream, r), sized for the largest n and the largest T of that r in the batch and re-pointed at each
    // fit: creating and destroying a handle per fit costs milliseconds of host time, more than a small fit takes
    int cap_n[TAME_MAX_R + 1] = {0}, cap_T[TAME_MAX_R + 1] = {0};
    for (int f = 0; f < n_fits; ++f) {
        cap_n[cfgs[f].r] = std::max(cap_n[cfgs[f].r], (int)cfgs[f].n);
        cap_T[cfgs[f].r] = std::max(cap_T[cfgs[f].r], (int)cfgs[f].T);
    }
    bool shared_cap[TAME_MAX_R + 1];
    for (int r = 1; r <= TAME_MAX_R; ++r) {
        if (!cap_n[r]) continue;
        // every fit needs the fused sweep (co-resident chain CTAs for all its time steps); otherwise the host loop takes over
        if ((cap_T[r] + TAME_CHAIN_WPC - 1) / TAME_CHAIN_WPC + 1 > tame_get_ops(r)->f64.sweep_capacity(1)) { cleanup(); return BATCH_FALLBACK; }
        // a batch of very different shapes (large n x small T next to small n x large T) would make the common capacity
        // much larger than any fit: keep one handle per shape then
        const double d = 2 + 2 * r, bytes = (double)S * cap_n[r] * cap_T[r] * (3.0 * d * d + 8.0 * d) * 8.0;
        shared_cap[r] = bytes <= 8e9;
    }
    for (int k = 0; k < n_fits && rc == TAME_OK; ++k) {
        const int f = order[k];
        const tame_config& cf = cfgs[f];
        const int s = k % S;
        tame_handle* h = nullptr;
        for (tame_handle* q : pool[s])
            if (q->cfg.r == cf.r && q->cap_n >= cf.n && q->cap_T >= cf.T) { h = q; break; }
        if (!h) {
            tame_config big = cf;
            if (shared_cap[cf.r]) { big.n = cap_n[cf.r]; big.T = cap_T[cf.r]; }
            rc = tame_create(&big, &h);
            if (rc == TAME_OK) { pool[s].push_back(h); rc = tame_set_stream(h, streams[s]); h->skip_symcheck = true; }
        }
        if (rc == TAME_OK) rc = tame_reconfigure(h, &cf);
        if (rc == TAME_OK && !h->fused) rc = fail(TAME_ESTATE, "tame_fit_batch: the fused sweep is unavailable for fit %d", f);
        if (rc == TAME_OK) rc = bind_Y<YT>(h, Y_dev[f]);
        if (rc == TAME_OK) rc = tame_bind_state(h, Xm_dev[f], Xc_dev[f]);
        if (rc == TAME_OK) rc = tame_fit_device(h, max_iter, tolerance, el_d + (size_t)f * max_iter, ms_d + (size_t)f * max_iter, nd_d + f);
    }
    for (int s = 0; s < S; ++s) {
        cudaError_t es = cudaStreamSynchronize(streams[s]);
        if (es != cudaSuccess && rc == TAME_OK) rc = fail(TAME_ECUDA, "tame_fit_batch: %s", cudaGetErrorString(es));
    }
    if (rc == TAME_OK) {
        for (auto& v : pool)
            for (tame_handle* q : v) {
                int ab = 0;
                cudaMemcpy(&ab, q->abort_flag, sizeof(int), cudaMemcpyDeviceToHost);
                if (ab) rc = fail(TAME_EHANG, "the chain kernel's watchdog fired inside tame_fit_batch");
            }
    }
    if (rc == TAME_OK) {
        std::vector<double> tmp((size_t)n_fits * max_iter);
        if (elbo_traces) { cudaMemcpy(tmp.data(), el_d, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost); memcpy(elbo_traces, tmp.data(), sizeof(double) * tmp.size()); }
        if (mse_traces) { cudaMemcpy(tmp.data(), ms_d, sizeof(double) * tmp.size(), cudaMemcpyDeviceToHost); memcpy(mse_traces, tmp.data(), sizeof(double) * tmp.size()); }
        e = cudaMemcpy(n_done, nd_d, sizeof(int32_t) * (size_t)n_fits, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(TAME_ECUDA, "tame_fit_batch read-back: %s", cudaGetErrorString(e));
    }
    cleanup();
    return rc;
}

template <class YT>
static int fit_host(const tame_config* cfg, const YT* Y_host, double* Xm_host, double* Xc_host, int32_t max_iter,
                  double tolerance, double* elbo_trace, double* mse_trace, int32_t* n_done) {
    if (!cfg || !Y_host || !Xm_host || !Xc_host) return fail(TAME_EINVAL, "null argument");
    if (cfg->world != 1) return fail(TAME_EINVAL, "tame_fit_host is single-GPU");
    tame_handle* h = nullptr;
    int rc = tame_create(cfg, &h);
    if (rc != TAME_OK) return rc;
    const size_t n = cfg->n, T = cfg->T, d = 2 + 2 * cfg->r;
    const size_t by = sizeof(YT) * n * n * T * 2, bm = sizeof(double) * n * T * d, bc = bm * d;
    YT* Y = nullptr;
    double *Xm = nullptr, *Xc = nullptr;
    cudaError_t e = cudaMalloc((void**)&Y, by);
    if (e == cudaSuccess) e = cudaMalloc((void**)&Xm, bm);
    if (e == cudaSuccess) e = cudaMalloc((void**)&Xc, bc);
    if (e == cudaSuccess) e = cudaMemcpyAsync(Y, Y_host, by, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(Xm, Xm_host, bm, cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(Xc, Xc_host, bc, cudaMemcpyHostToDevice, h->stream);
    if (e != cudaSuccess) rc = fail(TAME_ECUDA, "tame_fit_host staging: %s", cudaGetErrorString(e));
    if (rc == TAME_OK) rc = bind_Y<YT>(h, Y);
    if (rc == TAME_OK) rc = tame_bind_state(h, Xm, Xc);
    if (rc == TAME_OK) rc = tame_fit(h, max_iter, tolerance, elbo_trace, mse_trace, n_done);
    if (rc == TAME_OK) {
        e = cudaMemcpyAsync(Xm_host, Xm, bm, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(Xc_host, Xc, bc, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) rc = fail(TAME_ECUDA, "tame_fit_host read-back: %s", cudaGetErrorString(e));
    }
    std::string keep = g_err;
    cudaFree(Y); cudaFree(Xm); cudaFree(Xc);
    tame_destroy(h);
    g_err = keep;
    return rc;
}

template <class YT>
static int fit_batch(int32_t n_fits, const tame_config* cfgs, const YT* const* Y_dev, double* const* Xm_dev,
                   double* const* Xc_dev, int32_t max_iter, double tolerance, double* elbo_traces, double* mse_traces,
                   int32_t* n_done, int32_t n_streams) {
    if (n_fits < 0 || (n_fits > 0 && (!cfgs || !Y_dev || !Xm_dev || !Xc_dev || !n_done))) return fail(TAME_EINVAL, "null argument");
    for (int f = 0; f < n_fits; ++f) n_done[f] = 0;
    if (max_iter <= 0 || n_fits == 0) return TAME_OK;
    {
        // small single-GPU fits on one device: the whole fit loop runs on the device, one launch per fit (TAME_BATCH=host
        // keeps the host-driven loop below)
        bool eligible = true;
        for (int f = 0; f < n_fits; ++f)
            eligible = eligible && cfgs[f].world == 1 && cfgs[f].n <= 1024 && cfgs[f].device == cfgs[0].device && cfgs[f].r >= 1 && cfgs[f].r <= TAME_MAX_R;
        const char* v = getenv("TAME_BATCH");
        const char* sw = getenv("TAME_SWEEP");
        if (eligible && !(v && strcmp(v, "host") == 0) && !(sw && strcmp(sw, "panel") == 0)) {
            const int rc = fit_batch_device<YT>(n_fits, cfgs, Y_dev, Xm_dev, Xc_dev, max_iter, tolerance, elbo_traces, mse_traces, n_done, n_streams);
            if (rc != BATCH_FALLBACK) return rc;
        }
    }
    if (n_streams <= 0) n_streams = 8;
    n_streams = std::min(n_streams, std::max(n_fits, 1));
    // Small fits are bound by the host's launch rate, not by the device: one host thread per stream, each taking the next
    // unstarted fit and running the loop of base.py:166-203 on its own handle and stream.  Kernels of different fits
    // overlap on the device; nothing is shared between the workers but the fit counter.
    std::atomic<int> next{0};
    std::atomic<int> first_rc{TAME_OK};
    std::mutex err_mu;
    std::string err_msg;
    auto worker = [&]() {
        std::vector<std::pair<int, cudaStream_t>> streams;     // this worker's stream on every device it has met
        int rc = TAME_OK;
        std::vector<tame_handle*> pool;           // this worker's handles, one per shape it has met
        while (rc == TAME_OK && first_rc.load() == TAME_OK) {
            const int f = next.fetch_add(1);
            if (f >= n_fits) break;
            const tame_config& cf = cfgs[f];
            // a stream belongs to the device that was current when it was created (a new host thread starts on device 0)
            cudaStream_t st = nullptr;
            for (auto& ds : streams) if (ds.first == cf.device) st = ds.second;
            if (!st) {
                if (cudaSetDevice(cf.device) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) {
                    rc = fail(TAME_ECUDA, "cudaStreamCreate failed in tame_fit_batch (device %d)", cf.device);
                    break;
                }
                streams.emplace_back(cf.device, st);
            }
            tame_handle* h = nullptr;
            for (tame_handle* q : pool)
                if (q->cfg.n == cf.n && q->cfg.T == cf.T && q->cfg.r == cf.r && q->cfg.device == cf.device && cf.world == 1) { h = q; break; }
            if (h) rc = tame_reconfigure(h, &cf);
            else {
                rc = tame_create(&cf, &h);
                if (rc == TAME_OK) { pool.push_back(h); rc = tame_set_stream(h, st); }
            }
            if (rc == TAME_OK) rc = bind_Y<YT>(h, Y_dev[f]);
            if (rc == TAME_OK) rc = tame_bind_state(h, Xm_dev[f], Xc_dev[f]);
            if (rc == TAME_OK)
                rc = tame_fit(h, max_iter, tolerance, elbo_traces ? elbo_traces + (size_t)f * max_iter : nullptr,
                              mse_traces ? mse_traces + (size_t)f * max_iter : nullptr, &n_done[f]);
        }
        {
            std::string keep = g_err;
            for (tame_handle* q : pool) tame_destroy(q);
            g_err = keep;
        }
        if (rc != TAME_OK) {
            int expected = TAME_OK;
            if (first_rc.compare_exchange_strong(expected, rc)) {
                std::lock_guard<std::mutex> lk(err_mu);
                err_msg = g_err;
            }
        }
        for (auto& ds : streams) { cudaSetDevice(ds.first); cudaStreamDestroy(ds.second); }
    };
    std::vector<std::thread> pool;
    for (int w = 1; w < n_streams; ++w) pool.emplace_back(worker);
    worker();                                   // the calling thread is worker 0
    for (auto& t : pool) t.join();
    if (first_rc.load() != TAME_OK) {
        g_err = err_msg;
        return first_rc.load();
    }
    return TAME_OK;
}

extern "C" {

int tame_fit_host(const tame_config* cfg, const double* Y_host, double* Xm_host, double* Xc_host, int32_t max_iter,
                  double tolerance, double* elbo_trace, double* mse_trace, int32_t* n_done) {
    return fit_host<double>(cfg, Y_host, Xm_host, Xc_host, max_iter, tolerance, elbo_trace, mse_trace, n_done);
}
int tame_fit_host_f32(const tame_config* cfg, const float* Y_host, double* Xm_host, double* Xc_host, int32_t max_iter,
                      double tolerance, double* elbo_trace, double* mse_trace, int32_t* n_done) {
    return fit_host<float>(cfg, Y_host, Xm_host, Xc_host, max_iter, tolerance, elbo_trace, mse_trace, n_done);
}

int tame_fit_batch(int32_t n_fits, const tame_config* cfgs, const double* const* Y_dev, double* const* Xm_dev,
                   double* const* Xc_dev, int32_t max_iter, double tolerance, double* elbo_traces, double* mse_traces,
                   int32_t* n_done, int32_t n_streams) {
    return fit_batch<double>(n_fits, cfgs, Y_dev, Xm_dev, Xc_dev, max_iter, tolerance, elbo_traces, mse_traces, n_done, n_streams);
}
int tame_fit_batch_f32(int32_t n_fits, const tame_config* cfgs, const float* const* Y_dev, double* const* Xm_dev,
                       double* const* Xc_dev, int32_t max_iter, double tolerance, double* elbo_traces, double* mse_traces,
                       int32_t* n_done, int32_t n_streams) {
    return fit_batch<float>(n_fits, cfgs, Y_dev, Xm_dev, Xc_dev, max_iter, tolerance, elbo_traces, mse_traces, n_done, n_streams);
}

int tame_generate_Y(int32_t n, int32_t T, int32_t r, const double R[4], const double* X_dev, uint64_t seed,
                    int32_t row_begin, int32_t row_end, double* Y_dev, void* stream) {
    return generate_Y<double>(n, T, r, R, X_dev, seed, row_begin, row_end, Y_dev, stream);
}
int tame_generate_Y_f32(int32_t n, int32_t T, int32_t r, const double R[4], const double* X_dev, uint64_t seed,
                        int32_t row_begin, int32_t row_end, float* Y_dev, void* stream) {
    return generate_Y<float>(n, T, r, R, X_dev, seed, row_begin, row_end, Y_dev, stream);
}

int tame_comm_unique_id(void* id128) {
    if (!id128) return fail(TAME_EINVAL, "null argument");
    int rc = nccl_load();
    if (rc != TAME_OK) return rc;
    ncclUniqueId id;
    NK(g_nccl.GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, 128);
    return TAME_OK;
}

int tame_comm_init(tame_handle* h, const void* id128) {
    if (!h || !id128) return fail(TAME_EINVAL, "null argument");
    int rc = nccl_load();
    if (rc != TAME_OK) return rc;
    CK(cudaSetDevice(h->cfg.device));
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    NK(g_nccl.CommInitRank(&h->comm, h->P.world, id, h->P.rank));
    return TAME_OK;
}

int tame_ipc_export(tame_handle* h, void* handle64_host) {
    if (!h || !handle64_host) return fail(TAME_EINVAL, "null argument");
    CK(cudaSetDevice(h->cfg.device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    cudaIpcMemHandle_t mh;
    CK(cudaIpcGetMemHandle(&mh, h->hand));
    memcpy(handle64_host, &mh, 64);
    return TAME_OK;
}

int tame_ipc_import(tame_handle* h, const void* handles_host) {
    if (!h || !handles_host) return fail(TAME_EINVAL, "null argument");
    if (h->P.world == 1) return TAME_OK;
    if (h->P.world > 8) return fail(TAME_EINVAL, "the fused multi-GPU sweep supports up to 8 ranks");
    CK(cudaSetDevice(h->cfg.device));
    int k = 0;
    for (int r = 0; r < h->P.world; ++r) {
        if (r == h->P.rank) continue;
        cudaIpcMemHandle_t mh;
        memcpy(&mh, (const char*)handles_host + 64 * (size_t)r, 64);
        void* base = nullptr;
        CK(cudaIpcOpenMemHandle(&base, mh, cudaIpcMemLazyEnablePeerAccess));
        h->peer_base[k] = base;
        h->P.hand_peer[k] = (double2*)base;
        ++k;
    }
    h->npeers = k;
    h->P.npeers = h->fused_multi ? k : 0;
    return TAME_OK;
}

int tame_peer_attach(tame_handle* h, tame_handle* const* all_handles) {
    if (!h || !all_handles) return fail(TAME_EINVAL, "null argument");
    if (h->P.world == 1) return TAME_OK;
    if (h->P.world > 8) return fail(TAME_EINVAL, "the fused multi-GPU sweep supports up to 8 ranks");
    CK(cudaSetDevice(h->cfg.device));
    int k = 0;
    for (int r = 0; r < h->P.world; ++r) {
        if (r == h->P.rank) continue;
        tame_handle* o = all_handles[r];
        if (!o || o->P.world != h->P.world || o->P.rank != r || o->P.n != h->P.n || o->P.T != h->P.T || o->d != h->d)
            return fail(TAME_EINVAL, "tame_peer_attach: handle of rank %d does not belong to this fit", r);
        if (o->cfg.device != h->cfg.device) {
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, h->cfg.device, o->cfg.device));
            if (!can) return fail(TAME_ECUDA, "device %d cannot access device %d (no NVLink/P2P path)", h->cfg.device, o->cfg.device);
            cudaError_t e = cudaDeviceEnablePeerAccess(o->cfg.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(TAME_ECUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
            (void)cudaGetLastError();
        }
        h->P.hand_peer[k] = o->hand;
        ++k;
    }
    h->npeers = k;
    h->P.npeers = h->fused_multi ? k : 0;
    return TAME_OK;
}

int tame_gather_state(tame_handle* h) {
    if (!h) return fail(TAME_EINVAL, "null handle");
    if (h->P.world == 1) return TAME_OK;
    if (!h->comm) return fail(TAME_ESTATE, "tame_comm_init was not called");
    CK(cudaSetDevice(h->cfg.device));
    const size_t blk = (size_t)h->panel * h->P.T * h->d * h->d;
    NK(g_nccl.GroupStart());
    for (int b = 0; b * h->panel < h->P.n; ++b)
        NK(g_nccl.Broadcast(h->P.Xc + b * blk, h->P.Xc + b * blk, blk, ncclDouble, b % h->P.world, h->comm, h->stream));
    NK(g_nccl.GroupEnd());
    CK(cudaStreamSynchronize(h->stream));
    return TAME_OK;
}

int tame_debug_probes(tame_handle* h, uint64_t* out16_host) {
    if (!h || !out16_host) return fail(TAME_EINVAL, "null argument");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out16_host, h->dbg, sizeof(unsigned long long) * 16, cudaMemcpyDeviceToHost));
    return TAME_OK;
}

int tame_debug_trace(tame_handle* h, uint64_t* out_host, int32_t n_entries) {
    if (!h || !out_host) return fail(TAME_EINVAL, "null argument");
    if (!h->trace) return fail(TAME_ESTATE, "tracing is off (set TAME_TRACE=1 before tame_create)");
    CK(cudaSetDevice(h->cfg.device));
    CK(cudaStreamSynchronize(h->stream));
    const int have = 22 * ((h->P.n + TAME_SB - 1) / TAME_SB);
    CK(cudaMemcpy(out_host, h->trace, sizeof(unsigned long long) * std::min(have, (int)n_entries), cudaMemcpyDeviceToHost));
    return TAME_OK;
}

int tame_set_timing(tame_handle* h, int32_t enabled) {
    if (!h) return fail(TAME_EINVAL, "null handle");
    h->timing = enabled != 0;
    h->ev_used = 0;
    return TAME_OK;
}

int tame_last_timing(tame_handle* h, double* sweep_ms, double* elbo_ms, double* contract_ms, double* chain_ms, double* llmse_ms) {
    if (!h) return fail(TAME_EINVAL, "null handle");
    if (sweep_ms) *sweep_ms = h->sweep_ms;
    if (elbo_ms) *elbo_ms = h->elbo_ms;
    if (contract_ms) *contract_ms = h->contract_ms;
    if (chain_ms) *chain_ms = h->chain_ms;
    if (llmse_ms) *llmse_ms = h->llmse_ms;
    return TAME_OK;
}

}  // extern "C"
