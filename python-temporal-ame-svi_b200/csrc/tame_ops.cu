// tame_ops.cu -- instantiates the kernels of tame_kernels.cuh for one latent dimension (-DTAME_R=r) and
// exports their launchers through a function table; tame_api.cu picks the table by cfg.r.  The kernels that read Y are
// instantiated for both element types of Y (double, float): TameOps::f64 / TameOps::f32.
#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>

#include "tame_kernels.cuh"

#ifndef TAME_R
#error "compile with -DTAME_R=<latent dim>"
#endif

namespace {
constexpr int R = TAME_R;
constexpr int RW = 4;

// Kernel attributes (opt-in shared memory) and occupancy figures are per DEVICE: one flag / value per ordinal, so that a
// process driving several GPUs (drop-in `devices=`, tame_fit_batch over devices) configures each of them.
constexpr int MAX_DEV = 64;
struct PerDevice {
    std::atomic<int> v[MAX_DEV];
    PerDevice() { for (auto& x : v) x.store(-1); }
};
int current_device() {
    int dev = 0;
    cudaGetDevice(&dev);
    return (dev >= 0 && dev < MAX_DEV) ? dev : 0;
}
int device_sms(int dev) {
    static PerDevice sms;
    int s = sms.v[dev].load();
    if (s < 0) {
        cudaDeviceGetAttribute(&s, cudaDevAttrMultiProcessorCount, dev);
        sms.v[dev].store(s);
    }
    return s;
}
// runs `cfg` once per device (idempotent, so a race between two threads only repeats it)
template <class F>
void once_per_device(PerDevice& flag, F cfg) {
    const int dev = current_device();
    if (flag.v[dev].load() < 0) {
        cfg();
        flag.v[dev].store(1);
    }
}

void launch_totals(const TameParams& P, double* partial, int NS, cudaStream_t st) {
    k_totals_partial<R><<<dim3(P.T, NS), 320, 0, st>>>(P, partial, NS);
    k_totals_final<R><<<P.T, 128, 0, st>>>(P, partial, NS);
    tame_count_launch(2);
}

template <class YT>
void launch_contract(const TameParams& P, int k0, int k1, int j0, int j1, int tri, int accumulate, cudaStream_t st) {
    if (k1 <= k0 || j1 <= j0) return;
    dim3 grid((P.T + 31) / 32, (k1 - k0 + 8 * RW - 1) / (8 * RW));
    constexpr size_t smem = TameStream<R, RW, YT>::SMEM;
    static PerDevice configured;
    once_per_device(configured, [] { cudaFuncSetAttribute(k_contract<R, RW, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
    k_contract<R, RW, YT><<<grid, 256, smem, st>>>(P, k0, k1, j0, j1, tri, accumulate);
    tame_count_launch(1);
}

template <class YT = double>
size_t chain_smem_bytes() { return TAME_CHAIN_WPC * sizeof(TameChainSmem<R, 1, YT>); }

template <class YT>
cudaError_t launch_chain(const TameParams& P, int i0, int i1, cudaStream_t st) {
    static PerDevice configured;
    const size_t smem = chain_smem_bytes<YT>();
    cudaError_t ce = cudaSuccess;
    once_per_device(configured, [&] { ce = cudaFuncSetAttribute(k_chain<R, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
    if (ce != cudaSuccess) return ce;
    TameParams p = P;
    void* args[] = {(void*)&p, (void*)&i0, (void*)&i1};
    dim3 grid((P.T + TAME_CHAIN_WPC - 1) / TAME_CHAIN_WPC);
    tame_count_launch(1);
    return cudaLaunchCooperativeKernel((void*)k_chain<R, YT>, grid, dim3(2 * TAME_CHAIN_WPC * 32), args, smem, st);
}

void launch_covblend(const TameParams& P, cudaStream_t st) {
    const size_t cells = (size_t)P.nloc * P.T;
    if (cells == 0) return;
    const int blocks = (int)std::min<size_t>((cells + 7) / 8, (size_t)device_sms(current_device()) * 16);
    k_covblend<R><<<blocks, 256, 0, st>>>(P);
    tame_count_launch(1);
}

// the fused sweep in its two team shapes (NH = 1: 4 time steps per chain CTA; NH = 2: 2 time steps, separate totals / input warps)
template <int NH, class YT>
size_t sweep_smem_bytes() {
    const size_t chain = TameTeam<NH>::TPC * sizeof(TameChainSmem<R, NH, YT>);
    return chain > TameStream<R, RW, YT>::SMEM ? chain : TameStream<R, RW, YT>::SMEM;
}
template <int NH, class YT>
int sweep_capacity_nh() {
    static PerDevice cap;
    const int dev = current_device();
    int c = cap.v[dev].load();
    if (c < 0) {
        int per = 0;
        cudaFuncSetAttribute(k_sweep<R, RW, NH, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sweep_smem_bytes<NH, YT>());
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_sweep<R, RW, NH, YT>, 256, sweep_smem_bytes<NH, YT>());
        c = device_sms(dev) * per;
        cap.v[dev].store(c);
    }
    return c;
}
// co-resident CTAs of k_sweep on the current device
template <class YT>
int sweep_capacity(int nh) { return nh == 2 ? sweep_capacity_nh<2, YT>() : sweep_capacity_nh<1, YT>(); }

template <int NH, class YT>
cudaError_t launch_sweep_nh(const TameParams& P, cudaStream_t st) {
    const int capacity = sweep_capacity_nh<NH, YT>();
    TameParams p = P;
    p.n_chain_ctas = (P.T + TameTeam<NH>::TPC - 1) / TameTeam<NH>::TPC;
    const int nunits = ((P.n + TAME_SB - 1) / TAME_SB) * ((P.T + 31) / 32) * P.nparts;
    int workers = capacity - p.n_chain_ctas < nunits ? capacity - p.n_chain_ctas : nunits;
    if (workers < 1) return cudaErrorLaunchOutOfResources;
    // small problems: the chain (n nodes x ~1.5 us) outlasts the streaming (16 n^2 T bytes at ~30 GB/s per CTA) unless there
    // are fewer than ~n T / 2500 streaming CTAs; do not occupy many more SMs than that, so that independent fits
    // (tame_fit_batch) run side by side.  Any count >= 1 is correct: units are claimed dynamically and in order.
    const long want = ((long)P.n * P.T + 1499) / 1500 + 2;
    if ((long)workers > want) workers = (int)want;
    void* args[] = {(void*)&p};
    tame_count_launch(1);
    return cudaLaunchCooperativeKernel((void*)k_sweep<R, RW, NH, YT>, dim3(p.n_chain_ctas + workers), dim3(256), args, sweep_smem_bytes<NH, YT>(), st);
}

// grid of the fused sweep / whole-fit kernel for this problem: chain CTAs + streaming CTAs
template <int NH>
int sweep_grid_nh(const TameParams& P, int capacity, int* chain_ctas) {
    const int cc = (P.T + TameTeam<NH>::TPC - 1) / TameTeam<NH>::TPC;
    const int nunits = ((P.n + TAME_SB - 1) / TAME_SB) * ((P.T + 31) / 32) * P.nparts;
    int workers = capacity - cc < nunits ? capacity - cc : nunits;
    const long want = ((long)P.n * P.T + 1499) / 1500 + 2;
    if ((long)workers > want) workers = (int)want;
    *chain_ctas = cc;
    return workers < 1 ? -1 : cc + workers;
}

// k_fit: the whole fit loop in one cooperative launch (small problems; tame_fit_batch)
template <int NH, class YT>
size_t fit_smem_bytes() {
    const size_t a = sweep_smem_bytes<NH, YT>(), b = sizeof(TameCellSmem<R>);
    return a > b ? a : b;
}
template <int NH, class YT>
int fit_capacity_nh() {
    static PerDevice cap;
    const int dev = current_device();
    int c = cap.v[dev].load();
    if (c < 0) {
        int per = 0;
        cudaFuncSetAttribute(k_fit<R, RW, NH, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fit_smem_bytes<NH, YT>());
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_fit<R, RW, NH, YT>, 256, fit_smem_bytes<NH, YT>());
        c = device_sms(dev) * per;
        cap.v[dev].store(c);
    }
    return c;
}
template <int NH, class YT>
cudaError_t launch_fit_nh(const TameParams& P, const TameFitArgs& F, int* grid_out, cudaStream_t st) {
    TameParams p = P;
    const int grid = sweep_grid_nh<NH>(P, fit_capacity_nh<NH, YT>(), &p.n_chain_ctas);
    if (grid < 0) return cudaErrorLaunchOutOfResources;
    TameFitArgs f = F;
    void* args[] = {(void*)&p, (void*)&f};
    if (grid_out) *grid_out = grid;
    tame_count_launch(1);
    return cudaLaunchCooperativeKernel((void*)k_fit<R, RW, NH, YT>, dim3(grid), dim3(256), args, fit_smem_bytes<NH, YT>(), st);
}
template <class YT>
int pick_nh(const TameParams& P);
template <class YT>
cudaError_t launch_fit_device(const TameParams& P, const TameFitArgs& F, int* grid_out, cudaStream_t st) {
    return pick_nh<YT>(P) == 2 ? launch_fit_nh<2, YT>(P, F, grid_out, st) : launch_fit_nh<1, YT>(P, F, grid_out, st);
}
template <class YT>
int fit_grid(const TameParams& P) {
    int cc = 0;
    return pick_nh<YT>(P) == 2 ? sweep_grid_nh<2>(P, fit_capacity_nh<2, YT>(), &cc) : sweep_grid_nh<1>(P, fit_capacity_nh<1, YT>(), &cc);
}

// Team shape: the wide team (NH = 2) needs twice the chain CTAs; it pays when the chain, not the streaming, bounds the
// sweep -- several GPUs (the streaming shrinks with the rank count, the chain does not) or a small problem -- and
// when enough SMs are left for the streaming CTAs.  TAME_NH=1|2 overrides.
template <class YT>
int pick_nh(const TameParams& P) {
    int nh = (P.world >= 2 || (long)P.n * P.n * P.T <= (long)4096 * 4096 * 64) ? 2 : 1;
    if (const char* v = getenv("TAME_NH")) nh = (atoi(v) == 2) ? 2 : 1;
    if (nh == 2 && (P.T + 1) / 2 + 8 > sweep_capacity_nh<2, YT>()) nh = 1;
    return nh;
}

template <class YT>
cudaError_t launch_sweep_fused(const TameParams& P, cudaStream_t st) {
    return pick_nh<YT>(P) == 2 ? launch_sweep_nh<2, YT>(P, st) : launch_sweep_nh<1, YT>(P, st);
}

int chain_max_T() {
    static PerDevice cap;
    const int dev = current_device();
    int c = cap.v[dev].load();
    if (c < 0) {
        int per = 0;
        cudaFuncSetAttribute(k_chain<R, double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chain_smem_bytes());
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_chain<R, double>, 2 * TAME_CHAIN_WPC * 32, chain_smem_bytes());
        c = device_sms(dev) * per * TAME_CHAIN_WPC;
        cap.v[dev].store(c);
    }
    return c;
}

int llmse_blocks(const TameParams& P) { return 4 * ((P.T + 31) / 32) * ((P.nloc + 15) / 16); }   // upper bound over all variants (x4: grid.z split)

template <int RR, class YT, bool OK = (RR % 4 == 0)>
struct LlmseMma {
    static bool launch(const TameParams&, double*, int*, int, cudaStream_t) { return false; }
    static int blocks(const TameParams&) { return 0; }
};
template <int RR, class YT>
struct LlmseMma<RR, YT, true> {
    static int blocks(const TameParams& P) { return ((P.T + 31) / 32) * ((P.nloc + 15) / 16); }
    static bool launch(const TameParams& P, double* partial, int* nblocks, int symmetric, cudaStream_t st) {
        dim3 grid((P.T + 31) / 32, (P.nloc + 15) / 16);
        constexpr size_t smem = TameMma<RR, YT>::SMEM;
        static PerDevice configured;
        once_per_device(configured, [] {
            cudaFuncSetAttribute(k_llmse_mma<RR, false, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            cudaFuncSetAttribute(k_llmse_mma<RR, true, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        });
        if (symmetric) k_llmse_mma<RR, true, YT><<<grid, 256, smem, st>>>(P, partial);
        else k_llmse_mma<RR, false, YT><<<grid, 256, smem, st>>>(P, partial);
        *nblocks = grid.x * grid.y;
        tame_count_launch(1);
        return true;
    }
};
// default: DMMA tile where it wins (r = 4: -23 % on config 3), DFMA ring for r = 8 (the DMMA tile's chunk-granular double
// buffer keeps half as many bytes in flight and re-reads the partner records per 16 rows: +10 % at config 4).
// TAME_LLMSE=mma|dfma overrides (read per call so that tests can cover both).
bool llmse_use_mma() {
    if (R % 4 != 0) return false;
    const char* v = getenv("TAME_LLMSE");
    if (v && strcmp(v, "dfma") == 0) return false;
    if (v && strcmp(v, "mma") == 0) return true;
    return R == 4;
}

// DFMA ring with a 32-row tile of LL_NW warps x LL_RW rows (same ring footprint for every shape).  The tile reads each
// partner record from shared memory once per WARP, so the shared-memory pipe carries 144 B x LL_NW of records next to the
// 512 B x 2 of Y per partner and lane: 8 warps x 4 rows halves the record share (ncu, 16 x 2: l1tex data pipe 79 % busy,
// short_scoreboard the top stall; config 4: 16.9 -> 14.1 ms; n = 512 ... 4096, r = 2 ... 8: 0 ... -16 %).
template <int LL_RW, int LL_NW, class YT>
void launch_llmse_tile(const TameParams& P, double* partial, int* nblocks, int symmetric, cudaStream_t st) {
    dim3 grid((P.T + 31) / 32, (P.nloc + 31) / 32);
    constexpr size_t smem = TameStream<R, RW, YT>::SMEM;  // ring PD x LL_RW x (LL_NW x 32) dyads == PD x RW x 256 dyads
    static_assert(LL_RW * LL_NW == RW * 8, "same ring footprint");
    static PerDevice configured;
    once_per_device(configured, [] {
        cudaFuncSetAttribute(k_llmse<R, LL_RW, LL_NW, false, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        cudaFuncSetAttribute(k_llmse<R, LL_RW, LL_NW, true, YT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    });
    // split the partner range over grid.z when the (row tile x time slice) grid alone would leave SMs idle
    const int sms = device_sms(current_device());
    const int base = grid.x * grid.y;
    grid.z = (base >= 3 * sms) ? 1 : std::min(4, (3 * sms + base - 1) / base);
    if (symmetric) k_llmse<R, LL_RW, LL_NW, true, YT><<<grid, LL_NW * 32, smem, st>>>(P, partial);
    else k_llmse<R, LL_RW, LL_NW, false, YT><<<grid, LL_NW * 32, smem, st>>>(P, partial);
    *nblocks = grid.x * grid.y * grid.z;
    tame_count_launch(1);
}

template <class YT>
void launch_llmse(const TameParams& P, double* partial, int* nblocks, int symmetric, cudaStream_t st) {
    if (llmse_use_mma() && LlmseMma<R, YT>::launch(P, partial, nblocks, symmetric, st)) return;
    launch_llmse_tile<4, 8, YT>(P, partial, nblocks, symmetric, st);
}

// one resident wave: the kernel is latency-bound per warp (a serial elimination per cell), so a partial second wave at a
// third of the occupancy would cost as much as the first
int cellterms_blocks(const TameParams& P) {
    static PerDevice cap;
    const int dev = current_device();
    int c = cap.v[dev].load();
    if (c < 0) {
        int per = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k_cellterms<R>, 256, 0);
        c = device_sms(dev) * std::max(per, 1);
        cap.v[dev].store(c);
    }
    const long cells = (long)P.nloc * P.T, per_block = 8 * TameCellSmem<R>::G;
    return (int)std::max(1L, std::min((long)c, (cells + per_block - 1) / per_block));
}

void launch_cellterms(const TameParams& P, double logdetS0, double logdetQ, double* partial, int nblocks, cudaStream_t st) {
    k_cellterms<R><<<nblocks, 256, 0, st>>>(P, logdetS0, logdetQ, partial);
    tame_count_launch(1);
}
}  // namespace

#define TAME_CAT2(a, b) a##b
#define TAME_CAT(a, b) TAME_CAT2(a, b)
#define TAME_YOPS(YT) {launch_contract<YT>, launch_chain<YT>, launch_sweep_fused<YT>, launch_fit_device<YT>, fit_grid<YT>, sweep_capacity<YT>, launch_llmse<YT>}
extern const TameOps TAME_CAT(tame_ops_r, TAME_R) = {
    R, chain_smem_bytes(), TameTot<R>::TOT, launch_totals, launch_covblend, chain_max_T, launch_cellterms, llmse_blocks, cellterms_blocks,
    TAME_YOPS(double), TAME_YOPS(float)};
