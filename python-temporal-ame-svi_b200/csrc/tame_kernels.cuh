// tame_kernels.cuh -- sm_100a FP64 kernels of the Temporal-AME variational update loop.
//
// Reference formulas (file:line under /root/reference, see SURVEY.md section 8a):
//   observation terms   src/inference/structured_mf.py:289-326 (== naive_mf.py:284-376)
//   node update         src/inference/structured_mf.py:220-287, src/inference/naive_mf.py:207-282
//   ELBO                src/inference/structured_mf.py:115-209, src/inference/naive_mf.py:89-191
//   reconstruction MSE  src/models/temporal_ame.py:255-291, src/models/static_ame.py:189-238
//
// Data layout in HBM (row-major; FP64 except Y, which may be FP32):
//   Y    (nloc, n, T, 2)   the reference layout, stored as double or float (template parameter YT of every kernel that reads
//                          it; each dyad is widened to FP64 right after the load, all arithmetic is FP64).  For a fixed row
//                          the (j,t) pairs are contiguous 16-byte (8-byte) dyads, so a warp with lane <-> t streams 512
//                          (256) contiguous bytes per partner j.
//   Xm   (n, T, D)         D = 2 + 2R, x = [a, b, U(R), V(R)]
//   Xc   (n, T, D, D)
//   H    (nloc, T, 2R)     partner contraction  [ sum_j w0*V_j (R) , sum_j w1*U_j (R) ]  ("z order")
//   hab  (nloc, T, 2)      sum_j w0, sum_j w1  (sweep invariant)
//   tot  (T, 2R + 4R^2)    g = sum_j z_j, G = sum_j z_j z_j'  with z_j = [V_j, U_j]
//
// The Gauss-Seidel schedule of the reference is kept exactly: cell (i,t) sees new means of (j<i, t) and
// (i, t-1), old means of (j>i, t) and (i, t+1).  Parallelism comes from (a) the partner reductions
// (k_contract), (b) a systolic pipeline over time (k_chain: warp t owns time step t and walks the nodes in
// order, handing its new mean to warp t+1), (c) the streaming ELBO pass.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <type_traits>

#define TAME_WIN 64          // node block of the stand-alone chain launches (multi-GPU path)
#define TAME_RING 128        // ring of new partner vectors kept per time-step warp (>= the widest inline window)
#define TAME_CHAIN_WPC 4     // warps (time steps) per chain CTA: one per SM sub-partition, no issue/FP64 contention
#define TAME_SPIN_LIMIT (1 << 24)   // streaming workers' poll bound (the chain's waits are time-bounded, TAME_WATCHDOG_NS)
#define TAME_SB 32           // sub-block of the fused sweep: rows per streaming unit, push granularity
#define TAME_MAX_PARTS 4     // column parts per streaming unit (k_sweep): 1..TAME_MAX_PARTS
#define TAME_NG 4            // a streaming unit's 32 time steps are released / stamped as TAME_NG groups of 8
#define TAME_REFRESH 64      // the chain re-inverts the precision from scratch every TAME_REFRESH nodes (rank-2 updates between)

struct TameParams {
    int n, T, nloc, world, rank, panel, mode;
    double lr, p0, p1, q;     // R_inv = [[p0,q],[q,p1]]
    const void* Y;            // local rows, double or float (TameY<YT>::ptr)
    double* Xm;
    double* Xc;
    double* Craw;             // (nloc, T, D, D) raw covariance of the sweep (chain) -> k_covblend applies the rule + damping into Xc
    double* H;
    double* hab;
    double* tot;
    const double* cst;        // 6 DxD matrices: S0inv, Qinv, Phi'QinvPhi, QinvPhi, Phi'Qinv, Phi
    int* progress;            // (T) nodes finished in this sweep by the warp of time t
    int* abort_flag;
    // fused sweep (k_sweep): work distribution between the chain CTAs and the streaming CTAs
    unsigned long long* trace; // (2 * sub-blocks) optional: when the helper of t=0 started / stopped waiting for each sub-block's unit
    unsigned long long* dbg;  // 16 timing slots (ns / cycles) written by the first and last time-step warps
    double2* hand;            // (n,T,D) hand-over slots {new mean, tag}: the flag travels with the data
    double2* hand_peer[7];    // the other ranks' `hand` buffers (CUDA IPC peer pointers over NVLink); npeers entries
    int npeers;               // > 0: fused multi-GPU sweep (owners publish into every peer, the peers follow)
    int* unit_counter;        // next (sub-block, t-slice) unit to hand to a streaming CTA
    int* unit_done;           // (nsb * nslices) epoch stamp written when a unit's H rows are complete
    int epoch;                // sweep number (stamps are compared against it; never reset)
    int* cursor;              // (TAME_MAX_PARTS) column position last published by a streaming CTA of each column part
    int nparts;               // column parts per streaming unit (H holds nparts slabs of nloc*T*2R partial sums)
    int n_chain_ctas;
    int probe_t;              // time step of the second probe slot (dbg[8..15]); default T-1
    int deterministic;        // 1: fixed summation order of H (no convoy start: TAME_DETERMINISTIC=1), bitwise reproducible sweeps
};

// ------------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double2 tame_ld_stream2(const double* p) {
    double2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ float2 tame_ld_stream2(const float* p) {
    float2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double tame_ld_cg(const double* p) { return __ldcg(p); }
__device__ __forceinline__ void tame_st_cg(double* p, double v) { __stcg(p, v); }
__device__ __forceinline__ int tame_ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long tame_globaltimer() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ double2 tame_ld_volatile2(const double2* p) {
    double2 v;
    asm volatile("ld.volatile.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void tame_st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// local row of global node i / global node of local row (panel-cyclic ownership)
__device__ __forceinline__ int tame_lrow(int i, int panel, int world) {
    int b = i / panel;
    return (b / world) * panel + (i - b * panel);
}
__device__ __forceinline__ int tame_grow(int l, int panel, int world, int rank) {
    int lb = l / panel;
    return (lb * world + rank) * panel + (l - lb * panel);
}
__device__ __forceinline__ bool tame_owned(int i, int panel, int world, int rank) { return ((i / panel) % world) == rank; }

// ------------------------------------------------------------------------------------------------------
// moment totals per time step:  g[x] = sum_j z_j[x],  G[x][y] = sum_j z_j[x] z_j[y],  z_j = [V_j, U_j]
// (the partner sums of structured_mf.py:310-323 in closed form, SURVEY.md section 8a row A2)
// k_totals_partial: grid (T, NS), block 320 (>= TOT for R=8: 272); k_totals_final: grid T.
// ------------------------------------------------------------------------------------------------------
template <int R>
struct TameTot {
    static constexpr int NV = 2 * R;
    static constexpr int TOT = NV + NV * NV;
};

template <int R>
__device__ __forceinline__ int tame_zidx(int x) {  // index into x=[a,b,U,V] of component x of z=[V,U]
    return x < R ? 2 + R + x : 2 + (x - R);
}

template <int R>
__global__ void __launch_bounds__(320) k_totals_partial(TameParams P, double* partial, int NS) {
    constexpr int D = 2 + 2 * R, NV = 2 * R, TOT = TameTot<R>::TOT;
    const int t = blockIdx.x, s = blockIdx.y, e = threadIdx.x;
    const int chunk = (P.n + NS - 1) / NS;
    const int jb = s * chunk, je = min(P.n, jb + chunk);
    if (e >= TOT) return;
    int xa, xb = -1;
    if (e < NV) {
        xa = tame_zidx<R>(e);
    } else {
        int f = e - NV;
        xa = tame_zidx<R>(f / NV);
        xb = tame_zidx<R>(f % NV);
    }
    double acc = 0.0;
    for (int j = jb; j < je; ++j) {
        const double* m = P.Xm + ((size_t)j * P.T + t) * D;
        double va = m[xa];
        acc += (xb < 0) ? va : va * m[xb];
    }
    partial[((size_t)t * NS + s) * TOT + e] = acc;
}

template <int R>
__global__ void k_totals_final(TameParams P, const double* partial, int NS) {
    constexpr int TOT = TameTot<R>::TOT;
    const int t = blockIdx.x;
    for (int e = threadIdx.x; e < TOT; e += blockDim.x) {
        double acc = 0.0;
        for (int s = 0; s < NS; ++s) acc += partial[((size_t)t * NS + s) * TOT + e];
        P.tot[(size_t)t * TOT + e] = acc;
    }
    if (threadIdx.x == 0) {
        P.progress[t] = 0;
        if (t == 0) *P.unit_counter = 0;
    }
}

// ------------------------------------------------------------------------------------------------------
// asynchronous-copy helpers (LDGSTS): 16-byte global -> shared copies, zero-filled when !valid
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tame_cp_async16(void* smem_dst, const void* gsrc, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
// 8-byte variant (float dyads of Y): cp.async.cg only takes a cp-size of 16, so this one goes through L1 (.ca)
__device__ __forceinline__ void tame_cp_async8(void* smem_dst, const void* gsrc, bool valid) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int sz = valid ? 8 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void tame_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tame_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Element type of Y: one dyad (y_ij, y_ji) is a V2 in HBM and in the shared-memory staging buffers; `wide` turns it into
// the FP64 pair all arithmetic runs on (exact for float).  `bits` is the raw bit pattern (mirror check / hash).
template <class YT>
struct TameY;
template <>
struct TameY<double> {
    using V2 = double2;
    static __host__ __device__ __forceinline__ const double* ptr(const TameParams& P) { return static_cast<const double*>(P.Y); }
    static __device__ __forceinline__ void cp_async(void* dst, const double* src, bool valid) { tame_cp_async16(dst, src, valid); }
    static __device__ __forceinline__ double2 ld_stream(const double* p) { return tame_ld_stream2(p); }
    static __device__ __forceinline__ double2 wide(const double2& v) { return v; }
    static __device__ __forceinline__ double2 lds(const double2* p) { return *p; }
    static __device__ __forceinline__ unsigned long long bits(double v) { return (unsigned long long)__double_as_longlong(v); }
};
template <>
struct TameY<float> {
    using V2 = float2;
    static __host__ __device__ __forceinline__ const float* ptr(const TameParams& P) { return static_cast<const float*>(P.Y); }
    static __device__ __forceinline__ void cp_async(void* dst, const float* src, bool valid) { tame_cp_async8(dst, src, valid); }
    static __device__ __forceinline__ float2 ld_stream(const float* p) { return tame_ld_stream2(p); }
    static __device__ __forceinline__ double2 wide(const float2& v) { return make_double2((double)v.x, (double)v.y); }
    // a ring slot read where it is used (an ordered shared load): left to itself the compiler hoists the cheaper float
    // loads of later partners and the widened values then exceed the streaming loop's register budget at r = 8
    static __device__ __forceinline__ double2 lds(const float2* p) {
        float2 v;
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"((unsigned)__cvta_generic_to_shared(p)));
        return wide(v);
    }
    static __device__ __forceinline__ unsigned long long bits(float v) { return (unsigned long long)__float_as_uint(v); }
};

// shared-memory stride (doubles) of one staged X_mean record: D, or D+2 when D/2 is even, so that the 8 lanes of
// a quarter-warp reading 16-byte pieces of consecutive records hit distinct bank groups
template <int D>
struct TameRec {
    static constexpr int RS = ((D / 2) % 2) ? D : D + 2;
};

// Streaming tile shared by k_contract and k_llmse.
//   CTA = 8 warps; lane <-> time step t (32 consecutive t: 512 contiguous bytes of Y per partner), warp <-> RW rows.
//   Y goes global -> shared through a per-thread ring of PD partners (cp.async, RW*PD 16-byte (float Y: 8-byte) copies in
//   flight per thread, 128 KB (64 KB) per CTA at RW=4): every thread later reads back exactly the dyads it copied, so the ring
//   needs no block-level synchronisation.  The partners' X_mean records (a,b,U,V at the CTA's 32 time steps) are
//   staged in their natural layout, JC partners per chunk, double buffered, one __syncthreads per chunk.
template <int R, int RW, class YT = double>
struct TameStream {
    static constexpr int D = 2 + 2 * R, JC = 8, PD = 8, RS = TameRec<D>::RS, PIECES = D / 2;
    static constexpr size_t Y_BYTES = (size_t)PD * RW * 256 * sizeof(typename TameY<YT>::V2);
    static constexpr size_t M_BYTES = (size_t)2 * JC * 32 * RS * sizeof(double);
    static constexpr size_t SMEM = Y_BYTES + M_BYTES;
};

// ------------------------------------------------------------------------------------------------------
// tame_stream_cols: acc += sum_{j in [jb,je), (tri ? j>k : j!=k)} ( w0(k,j,t) * V_j(t) , w1(k,j,t) * U_j(t) )
// for the CTA's 8*RW rows (warp <-> RW rows starting at kw) and 32 time steps (lane <-> t), with
// w0 = p0*y0 + q*y1, w1 = q*y0 + p1*y1  -- the [U,V] rows of sum_j J'R^-1 y_ij (structured_mf.py:324).
// Software pipeline described at TameStream.  Must be called by all 256 threads of the CTA.
// ------------------------------------------------------------------------------------------------------
template <int R, int RW, class YT>
__device__ __forceinline__ void tame_stream_cols(const TameParams& P, unsigned char* smem_raw, const YT* const (&yrow)[RW],
                                                 const bool (&rv)[RW], int kw, int t0, int jb, int je, bool tri,
                                                 double (&accA)[RW][R], double (&accB)[RW][R], int* cursor = nullptr,
                                                 bool lane_on = true) {
    using TS = TameStream<R, RW, YT>;
    using Y2 = typename TameY<YT>::V2;
    constexpr int D = TS::D, JC = TS::JC, PD = TS::PD, RS = TS::RS;
    static_assert(JC == PD, "ring slot == position in chunk");
    Y2 (*Yr)[RW][256] = reinterpret_cast<Y2 (*)[RW][256]>(smem_raw);                                 // [PD][RW][256]
    double (*Mb)[JC][32][RS] = reinterpret_cast<double (*)[JC][32][RS]>(smem_raw + TS::Y_BYTES);     // [2][JC][32][RS]
    const int tid = threadIdx.x, lane = tid & 31;
    const size_t jstride = (size_t)P.T * 2;
    const int nchunks = (je > jb) ? (je - jb + JC - 1) / JC : 0;
    if (nchunks == 0) return;

    auto issue_y = [&](int j, int slot) {
#pragma unroll
        for (int rr = 0; rr < RW; ++rr) {
            const int k = kw + rr;
            const bool ok = lane_on && rv[rr] && (j < je) && (tri ? (j > k) : (j != k));
            TameY<YT>::cp_async(&Yr[slot][rr][tid], yrow[rr] + (size_t)min(j, P.n - 1) * jstride, ok);
        }
    };
    // fast path of the record staging: with the natural record pitch (RS == D) and a full 32-step slice, partner j's records
    // are one contiguous block of 32*D doubles in global AND shared memory, so 16-byte piece e of the chunk goes from
    // base + 2e + jj*(T*D - 32*D) to Mb[buf] + 2e with jj = e / (32*PIECES): no per-piece modulo / clamp / predicate.
    const bool m_fast = (RS == D) && (t0 + 32 <= P.T);
    const size_t m_gap = (size_t)P.T * D - 32 * D;
    auto issue_m = [&](int buf, int jc) {
        if (m_fast && jc + JC <= P.n) {
            const double* base = P.Xm + ((size_t)jc * P.T + t0) * D;
            double* dst = &Mb[buf][0][0][0];
#pragma unroll
            for (int it = 0; it < (JC * 32 * TS::PIECES + 255) / 256; ++it) {
                const int e = tid + it * 256;
                if ((it + 1) * 256 <= JC * 32 * TS::PIECES || e < JC * 32 * TS::PIECES) {
                    const int jj = e / (32 * TS::PIECES);
                    tame_cp_async16(dst + 2 * e, base + 2 * e + jj * m_gap, true);
                }
            }
            return;
        }
        for (int e = tid; e < JC * 32 * TS::PIECES; e += 256) {
            const int piece = e % TS::PIECES, tl = (e / TS::PIECES) & 31, jj = e / (TS::PIECES * 32);
            const int j = jc + jj, tt = t0 + tl;
            const bool ok = (j < je) && (tt < P.T);
            const double* src = P.Xm + ((size_t)min(j, P.n - 1) * P.T + min(tt, P.T - 1)) * D + piece * 2;
            tame_cp_async16(&Mb[buf][jj][tl][piece * 2], src, ok);
        }
    };

    __syncthreads();            // the staging buffers may still be read by a previous call
    issue_m(0, jb);
#pragma unroll
    for (int s = 0; s < PD; ++s) {
        issue_y(jb + s, s);
        tame_cp_async_commit();
    }
    for (int c = 0; c < nchunks; ++c) {
        const int jc = jb + c * JC, buf = c & 1;
#pragma unroll
        for (int jj = 0; jj < JC; ++jj) {
            tame_cp_async_wait<PD - 1>();
            if (jj == 0) {
                __syncthreads();                               // chunk c's partner records are visible to the CTA
                if (c + 1 < nchunks) issue_m(buf ^ 1, jc + JC);
                if (cursor != nullptr && (c & 15) == 0 && tid == 0) *((volatile int*)cursor) = jc;   // convoy position
            }
            double w0[RW], w1[RW];
#pragma unroll
            for (int rr = 0; rr < RW; ++rr) {
                const double2 y = TameY<YT>::lds(&Yr[jj][rr][tid]);
                w0[rr] = P.p0 * y.x + P.q * y.y;
                w1[rr] = P.q * y.x + P.p1 * y.y;
            }
            const double* rec = &Mb[buf][jj][lane][0];
#pragma unroll
            for (int a = 0; a < R; ++a) {
                const double zu = rec[2 + a];        // U_j[a]
                const double zv = rec[2 + R + a];    // V_j[a]
#pragma unroll
                for (int rr = 0; rr < RW; ++rr) {
                    accA[rr][a] = fma(w0[rr], zv, accA[rr][a]);
                    accB[rr][a] = fma(w1[rr], zu, accB[rr][a]);
                }
            }
            issue_y(jc + jj + PD, jj);
            tame_cp_async_commit();
        }
    }
    tame_cp_async_wait<0>();
}

// ------------------------------------------------------------------------------------------------------
// k_contract: H[k,t,:] (+)= contraction over partners j in [j0,j1) for rows [k0,k1) (stand-alone launches: the
// multi-GPU sweep's static upper part and right-looking pushes).  One pass over Y[k0:k1, j0:j1].
// grid (ceil(T/32), ceil((k1-k0)/(8*RW))), block 256, TameStream::SMEM dynamic smem.
// ------------------------------------------------------------------------------------------------------
template <int R, int RW, class YT>
__global__ void __launch_bounds__(256, 1) k_contract(TameParams P, int k0, int k1, int j0, int j1, int tri, int accumulate) {
    constexpr int NV = 2 * R, JC = TameStream<R, RW, YT>::JC, RT = 8 * RW;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int t0 = blockIdx.x * 32, t = t0 + lane;
    const bool tv = t < P.T;
    const int kbase = k0 + blockIdx.y * RT;
    if (!tame_owned(kbase, P.panel, P.world, P.rank)) return;   // RT divides the panel size
    const int kw = kbase + warp * RW;

    double accA[RW][R], accB[RW][R];
#pragma unroll
    for (int rr = 0; rr < RW; ++rr)
#pragma unroll
        for (int a = 0; a < R; ++a) accA[rr][a] = accB[rr][a] = 0.0;
    const YT* yrow[RW];
    bool rv[RW];
#pragma unroll
    for (int rr = 0; rr < RW; ++rr) {
        const int k = kw + rr;
        rv[rr] = (k < k1) && tv;
        const int l = tame_lrow(min(k, P.n - 1), P.panel, P.world);
        yrow[rr] = TameY<YT>::ptr(P) + ((size_t)l * P.n * P.T + (tv ? t : 0)) * 2;
    }
    const int jstart = tri ? max(j0, ((kbase + 1) / JC) * JC) : j0;
    tame_stream_cols<R, RW, YT>(P, smem_raw, yrow, rv, kw, t0, jstart, j1, tri != 0, accA, accB);
#pragma unroll
    for (int rr = 0; rr < RW; ++rr) {
        const int k = kw + rr;
        if (k < k1 && tv) {
            double* h = P.H + ((size_t)tame_lrow(k, P.panel, P.world) * P.T + t) * NV;
#pragma unroll
            for (int a = 0; a < R; ++a) {
                h[a] = accumulate ? h[a] + accA[rr][a] : accA[rr][a];
                h[R + a] = accumulate ? h[R + a] + accB[rr][a] : accB[rr][a];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// warp-level in-place Gauss-Jordan inverse of a symmetric positive-definite DxD matrix.
// lane c (< D) holds column c in col[0..D-1].  At step k every lane publishes its element of pivot row k, the
// whole row is read back as a shared-memory broadcast, and column k is reconstructed from the row by the
// (anti)symmetry of the partially swept matrix ( M[r][k] = -M[k][r] for swept r<k, +M[k][r] otherwise; the
// publishing lane applies the sign ).  The loop over pivots is ROLLED (one step is ~100 instructions, so the
// chain's inner loop stays inside the instruction cache): the row registers rotate by one position per step so the
// pivot row is always col[0] and all register indices stay compile-time; the published row is stored twice so the
// rotated read needs no modulo.  After D steps the rows are back in place.
// Returns sum_k log(pivot_k) = logdet when WANT_LOGDET.  rowb: 4*D doubles of per-warp shared memory.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ double tame_rcp(double x) {
    // rcp.approx.ftz.f64 carries ~20 bits (measured 9.9e-7 on B200); one cubic (Halley) step reaches 2.2e-16
    // (tools/ubench_fp64.cu): r' = r (1 + e + e^2), e = 1 - x r.  24 + 3*8.8 cycles instead of 76 for IEEE division.
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double e = fma(-x, r, 1.0);
    const double e2 = fma(e, e, e);
    return fma(r, e2, r);
}

#define TAME_GJ_ROWB(D) (2 * (2 * (D) + 32))   // doubles of per-warp shared memory used by tame_gj_inverse

template <int D, bool WANT_LOGDET>
__device__ __forceinline__ double tame_gj_inverse(double (&col)[D], double* rowb, int lane) {
    constexpr int RB = 2 * D + 32;
    double logdet = 0.0;
    // every lane publishes (lanes >= D into a scratch slot) so the loop body has no divergent region
    const int slot0 = (lane < D) ? lane : 2 * D + (lane - D), slot1 = (lane < D) ? lane + D : 2 * D + (lane - D);
    rowb[slot0] = col[0];
    rowb[slot1] = col[0];
#pragma unroll 1
    for (int k = 0; k < D; ++k) {
        const double* rr = rowb + (k & 1) * RB + k;   // rr[p]: signed pivot-row element of original index (k+p) mod D
        __syncwarp();
        const double pivv = rr[0];
        double rk[D];
#pragma unroll
        for (int p = 1; p < D; ++p) rk[p] = rr[p];
        // in the shadow of the reciprocal: the pivot column restarts from zero (its new entries are -f_r * piv) and
        // its own pivot-row element counts as 1 (so that s = piv there)
        const bool isk = (lane == k);
        const double a0 = isk ? 1.0 : col[0];
#pragma unroll
        for (int p = 1; p < D; ++p) col[p] = isk ? 0.0 : col[p];
        const unsigned flip = (lane <= k) ? 0x80000000u : 0u;    // rows 0..k are swept from the next step on
        const double piv = tame_rcp(pivv);
        if (WANT_LOGDET) logdet += log(pivv);
        const double s = a0 * piv;                                // new pivot-row element of this column
        // the next pivot row's element first, published at once: the broadcast round trip of step k+1 overlaps the
        // rest of this step's update
        col[0] = fma(-rk[1], s, col[1]);
        if (k + 1 < D) {
            double* nb = rowb + ((k + 1) & 1) * RB;
            const double v = __hiloint2double(__double2hiint(col[0]) ^ flip, __double2loint(col[0]));
            nb[slot0] = v;
            nb[slot1] = v;
        }
#pragma unroll
        for (int p = 2; p < D; ++p) col[p - 1] = fma(-rk[p], s, col[p]);
        col[D - 1] = s;
    }
    return logdet;
}

// logdet of a symmetric positive-definite DxD matrix (lane c holds column c): forward elimination only -- at step k just
// the rows below the pivot are updated (half the work of the inverse) -- and the pivots are multiplied in groups of four
// so that 18 pivots cost 5 logarithms.  A GROUP of lanes owns the matrix (lane c of the group <-> column c, `act` = c < D and
// the group has a matrix); all 32 lanes must call.  rb2: 2*D doubles of shared memory per group (double-buffered pivot row).
template <int D>
__device__ __forceinline__ double tame_logdet_spd(double (&col)[D], double* rb2 /* this lane group's 2 * D doubles */, int c, bool act) {
    double logdet = 0.0, prod = 1.0;
#pragma unroll
    for (int k = 0; k < D; ++k) {
        double* rb = rb2 + (k & 1) * D;
        if (act) rb[c] = col[k];
        __syncwarp();
        const double pivv = rb[k];
        prod *= pivv;
        if ((k & 3) == 3 || k == D - 1) { logdet += log(prod); prod = 1.0; }
        if (k + 1 < D) {
            const double s = col[k] * tame_rcp(pivv);
#pragma unroll
            for (int r = k + 1; r < D; ++r) col[r] = fma(-rb[r], s, col[r]);
        }
    }
    return logdet;
}

// ------------------------------------------------------------------------------------------------------
// The Gauss-Seidel chain (structured_mf.py:211-287, naive_mf.py:193-282).
//
// Warp pair <-> time step t: a CHAIN warp and a HELPER warp walk the nodes in order.  For cell (i,t)
//   P_i = const_t + sum_{j != i} G(z_j),  G(z) = J_z' R^-1 J_z (rank 2),  z_j = [V_j, U_j] at time t (new for j<i, old for j>i)
//   C_i = P_i^-1 (then mask / symmetrise / jitter, :270-277),  mu = C_i h_i,  damped write (:282-287).
// The only loop-carried work is the inverse: P_i = P_{i-1} - G(z_i^old) + G(z_{i-1}^new).  The chain warp carries the raw
// inverse in registers (lane c <-> column c) and applies the two rank-2 Woodbury corrections (2x2 capacitance matrix, one
// reciprocal each) at the start of the node in ONE rolled loop -- the code exists once (instruction cache) and the chain
// needs nothing of node i+1.  Every TAME_REFRESH nodes (and at the first node after foreign nodes) the HELPER side rebuilds
// the inverse from the running moment totals (in-place Gauss-Jordan) without the last TAME_NL partners, which the chain
// re-enters by up-dates in the same loop.
// Everything else is the helper's: ALL global loads TAME_LA nodes ahead (cp.async staging: the inline window's Y entries,
// old means, the static partner part H, the hand-over slot of (i,t-1)), the inline window's partner sum, the AR(1) terms
// with the NEW mean of (i,t-1) and the OLD mean of (i,t+1), the running totals, and -- multi-GPU -- the nodes of other ranks.
// The chain warp stores its raw covariance column straight to the global scratch Craw; the factorisation rule, the
// symmetrisation, the jitter and the damped write into X_cov happen in a streaming post-pass (k_covblend).
// Mailboxes (shared memory):  helper -> chain  inp[k] {h without the last TAME_NL partners, old mean, those partners'
// weights}, pdt[k] (diag(P), naive rule), pcol (the inverse at refresh nodes);  chain -> helper  ring[k] (new z), mring[k]
// (new mean for the next time step's helper in the same CTA).
// Counters: ready[slot] (inputs of the node in that mailbox slot), t_ready (totals-side data), f_done (foreign nodes),
// c_done (chain).
// Two shapes of the warp team per time step (template NH):
//   NH = 1  chain warp + ONE helper that does everything above; 4 time steps per CTA (streaming-bound problems: the
//           chain CTAs take few SMs)
//   NH = 2  chain warp + a TOTALS warp (running moments, precision column at refresh nodes, diag(P), foreign nodes) + TWO
//           INPUT warps that prepare alternate nodes; 2 time steps per CTA (chain-bound problems: small n, multi-GPU)
// ------------------------------------------------------------------------------------------------------
#define TAME_NL 3            // trailing partners (i-NL..i-1) whose terms the chain warp adds itself: the helpers run NL nodes ahead
#define TAME_LA 4            // look-ahead of a helper's global loads, in its own loop iterations (NH = 1)
#define TAME_LA2 3           // same for the input warps of NH = 2 (an iteration is two nodes there)
#define TAME_NINP 8          // depth of the helper -> chain mailbox (power of two, >= TAME_NL + 2)
#define TAME_MR 16           // depth of the intra-CTA hand-over ring (self-validating slots; the global slot is the fallback)
// inline window of the fused sweep: the TAME_WBACK(NH) previous + the current 32-node sub-block are summed by the helpers,
// everything older by the streaming CTAs.  The wide team can afford one more sub-block, which takes the streaming CTAs'
// reaction to a group's final release (one 32-column pass, ~15 us) off the chain's critical path.
#define TAME_WBACK(NH) ((NH) == 1 ? 2 : 3)
#define TAME_WATCHDOG_NS 4000000000ull
enum { TAME_ROLE_ALL = 0, TAME_ROLE_TOTALS = 1, TAME_ROLE_INPUT = 2 };

template <int R, int NH, class YT = double>
struct __align__(16) TameChainSmem {
    static constexpr int D = 2 + 2 * R, NV = 2 * R, TOT = TameTot<R>::TOT, DP = D + 1;
    static constexpr int NSLOT = (NH == 1) ? 8 : 16;   // staging ring of the input side (power of two)
    static constexpr int WMAX = 32 * (TAME_WBACK(NH) + 1);          // widest inline window (partners)
    static constexpr int RING = (NH == 1) ? TAME_RING : 2 * TAME_RING;   // rows of the z ring (>= WMAX + look-ahead, power of two)
    static constexpr int NTS = (NH == 1) ? 1 : 8;      // staging ring of the totals warp (NH = 2)
    struct Stage {                                  // one node's global inputs (cp.async destinations, 16-byte aligned)
        typename TameY<YT>::V2 ywin[WMAX];          // Y[i, wlo + s, t, :] of the inline window
        double2 hand[D];                            // hand-over slot {new mean, tag} of (i, t-1); foreign nodes (NH = 1): of (i, t)
        double mold[D], mnext[D];                   // old means of (i,t) and (i,t+1)
        double H[TAME_MAX_PARTS][NV];               // static partner part (per column part)
        double hab[2];
    };
    struct TStage {                                 // the totals warp's own staging (NH = 2)
        double2 hand[D];                            // foreign nodes: hand-over slot of (i, t)
        double mold[D];
    };
    struct Inp {                                    // helper -> chain
        double hrest[D];                            // h of the cell without the trailing partners' terms
        double mold[D];
        double wl[TAME_NL][2];                      // (w0, w1) of the trailing partners: wl[q] <-> partner i-1-q
    };
    double ring[RING][NV];                     // z = [V,U] (new) of the last TAME_RING nodes at this time step
    Stage st[NSLOT];
    TStage tst[NTS];
    double pcol[D * DP];                            // totals side -> chain at refresh nodes: the precision without the trailing partners
    double pdt[TAME_NINP][D];                       // totals side -> chain: diag(P) without the trailing partners (naive rule)
    Inp inp[TAME_NINP];
    double2 wbuf[NH][WMAX];                    // (w0, w1) of the window, per input warp
    double2 Fs[2][32];                              // F = M J' of the up-date / down-date, one row per lane
    double rowb[TAME_GJ_ROWB(D)];
    double hvec[D], mprev[NH][D], hin[NH][NV];
    double2 mring[TAME_MR][D];                      // chain -> helper of the next time step in the same CTA: {new mean, tag}
    int ready[TAME_NINP];                           // node whose inputs sit in mailbox slot s
    int t_ready;                                    // last node whose totals-side data (pcol, pdt) is published
    int f_done;                                     // last foreign node taken over (X_mean replica, ring)
    int c_done;                                     // last node the chain warp has finished
    int pad_;
};
static_assert(sizeof(TameChainSmem<1, 1>) % 16 == 0 && sizeof(TameChainSmem<2, 1>) % 16 == 0 && sizeof(TameChainSmem<3, 1>) % 16 == 0 &&
              sizeof(TameChainSmem<4, 2>) % 16 == 0 && sizeof(TameChainSmem<8, 2>) % 16 == 0 &&
              sizeof(TameChainSmem<1, 1, float>) % 16 == 0 && sizeof(TameChainSmem<3, 2, float>) % 16 == 0, "per-time-step chain block must stay 16-byte aligned");
static_assert(TAME_LA + 2 <= 8 && 2 * (TAME_LA2 + 1) + 4 <= 16 && TAME_NL + 2 <= TAME_NINP, "mailbox depth");

// panel-cyclic ownership of consecutive nodes without integer divisions: rem = k % panel, pw = (k / panel) % world,
// lb = (k / panel) / world; owned = (pw == rank), local row = lb * panel + rem
struct TameOwn {
    int rem, pw, lb;
    __device__ __forceinline__ void init(int k, int panel, int world) {
        const int b = k / panel;
        rem = k - b * panel; pw = b % world; lb = b / world;
    }
    __device__ __forceinline__ void next(int panel, int world) {
        if (++rem == panel) { rem = 0; if (++pw == world) { pw = 0; ++lb; } }
    }
    __device__ __forceinline__ int lrow(int panel) const { return lb * panel + rem; }
};

// time-bounded spinning: every 1024 failed polls look at the abort flag and at the clock
struct TameSpin {
    unsigned spins = 0;
    unsigned long long t0 = 0;
    // the slow check: abort raised by anyone, or this wait older than the watchdog (which then raises it)
    __device__ __forceinline__ bool check(int* abort_flag) {
        if (*((volatile int*)abort_flag)) return true;
        const unsigned long long now = tame_globaltimer();
        if (t0 == 0) t0 = now;
        else if (now - t0 > TAME_WATCHDOG_NS) { atomicExch(abort_flag, 1); return true; }
        return false;
    }
    __device__ __forceinline__ bool expired(int* abort_flag) { return ((++spins & 1023u) == 0) && check(abort_flag); }
};

// wait until a shared-memory counter written by the partner warp reaches `target`; false = abort.  Every lane polls the same
// word (one broadcast LDS per poll), so the branch is warp-uniform and the ready case costs one load.
__device__ __forceinline__ bool tame_wait_smem(const int* flag, int target, int lane, int* abort_flag) {
    if (*((volatile const int*)flag) < target) {
        TameSpin sp;
        for (;;) {
            if (*((volatile const int*)flag) >= target) break;
            if ((++sp.spins & 1023u) == 0) {
                const int ex = (lane == 0 && sp.check(abort_flag)) ? 1 : 0;
                if (__any_sync(0xffffffffu, ex)) return false;
            }
        }
    }
    __syncwarp();
    return true;
}

// F = M J_z' for the symmetric matrix whose column (= row) c is cw[]:  f0 = (M g0)[c], f1 = (M g1)[c],
// g0 = (1,0,V,0), g1 = (0,1,0,U), z = [V,U]
template <int R>
__device__ __forceinline__ void tame_rank2_F(const double (&cw)[2 + 2 * R], const double (&z)[2 * R], double& f0, double& f1) {
    double a0 = cw[0], a1 = 0.0, b0 = cw[1], b1 = 0.0;
#pragma unroll
    for (int x = 0; x < R; ++x) {
        if (x & 1) a1 = fma(cw[2 + x], z[x], a1); else a0 = fma(cw[2 + x], z[x], a0);
        if (x & 1) b1 = fma(cw[2 + R + x], z[R + x], b1); else b0 = fma(cw[2 + R + x], z[R + x], b0);
    }
    f0 = a0 + a1;
    f1 = b0 + b1;
}
// cw <- (M + sigma J_z' R^-1 J_z)^-1 = M^-1... in inverse form: cw - F (sigma R + J_z F)^-1 F'   (Woodbury; Rxx = (R^-1)^-1)
template <int R>
__device__ __forceinline__ void tame_rank2_apply(double (&cw)[2 + 2 * R], const double (&z)[2 * R], double f0, double f1,
                                                 const double2* Fs, double sigma, double R00, double R01, double R11) {
    constexpr int D = 2 + 2 * R;
    double2 F[D];
#pragma unroll
    for (int k = 0; k < D; ++k) F[k] = Fs[k];
    double K00 = fma(sigma, R00, F[0].x), K01 = fma(sigma, R01, F[0].y), K11 = fma(sigma, R11, F[1].y);
    double a1 = 0.0, b1 = 0.0, c1 = 0.0;
#pragma unroll
    for (int x = 0; x < R; ++x) {
        if (x & 1) { a1 = fma(z[x], F[2 + x].x, a1); b1 = fma(z[x], F[2 + x].y, b1); c1 = fma(z[R + x], F[2 + R + x].y, c1); }
        else { K00 = fma(z[x], F[2 + x].x, K00); K01 = fma(z[x], F[2 + x].y, K01); K11 = fma(z[R + x], F[2 + R + x].y, K11); }
    }
    K00 += a1; K01 += b1; K11 += c1;
    const double rd = tame_rcp(fma(K00, K11, -K01 * K01));
    const double v0 = fma(K11, f0, -K01 * f1) * rd, v1 = fma(K00, f1, -K01 * f0) * rd;
#pragma unroll
    for (int k = 0; k < D; ++k) cw[k] = fma(-F[k].x, v0, fma(-F[k].y, v1, cw[k]));
}

// ------------------------------------------------------------------------------------------------------
// helper warp(s) of time step t.  ROLE_ALL: the one helper of NH = 1.  ROLE_TOTALS / ROLE_INPUT (hi = 0,1): the team of NH = 2;
// an input warp takes the nodes i0 + hi, i0 + hi + 2, ...
// ------------------------------------------------------------------------------------------------------
template <int R, bool FUSED, int NH, int ROLE, class YT>
__device__ __forceinline__ void tame_chain_helper(const TameParams& P, TameChainSmem<R, NH, YT>& sm, const TameChainSmem<R, NH, YT>* pv,
                                                  int lane, int t, int hi, int i0, int i1) {
    using S = TameChainSmem<R, NH, YT>;
    constexpr bool DO_TOT = (ROLE != TAME_ROLE_INPUT), DO_INP = (ROLE != TAME_ROLE_TOTALS);
    constexpr int STEP = (ROLE == TAME_ROLE_INPUT) ? NH : 1;
    constexpr int D = S::D, NV = S::NV, TOT = S::TOT, DP = S::DP;
    constexpr int WSB = FUSED ? TAME_SB : TAME_WIN, WBACK = FUSED ? TAME_WBACK(NH) : 0, NWS = FUSED ? TAME_WBACK(NH) + 1 : 2;
    constexpr int NL = TAME_NL, LA = (NH == 1) ? TAME_LA : ((ROLE == TAME_ROLE_INPUT) ? TAME_LA2 : TAME_LA);
    constexpr int SMASK = (DO_INP ? S::NSLOT : S::NTS) - 1, IMASK = TAME_NINP - 1, RMASK = S::RING - 1;
    const int T = P.T, c = lane, cc = min(c, D - 1);
    const bool act = c < D, has_prev = t > 0, has_next = t < T - 1;
    const bool multi = FUSED && P.npeers > 0;
    const int nslices = (T + 31) / 32, nparts = FUSED ? P.nparts : 1;
    const double m1 = (double)(P.n - 1);
    const unsigned long long magic = 0x5AFE000000000000ull + (unsigned long long)(unsigned)P.epoch;
    const size_t slab = (size_t)P.nloc * T * NV;
    const double2* hand_prev = P.hand + (size_t)max(t - 1, 0) * D + cc;     // + i*T*D : slot of (i, t-1), component cc
    const double2* hand_mine = P.hand + (size_t)t * D + cc;
    auto window_lo = [&](int k) { return max(i0, (k / WSB - WBACK) * WSB); };
    auto tag_ok = [&](const double2& v) {
        return ((unsigned long long)__double_as_longlong(v.x) ^ (unsigned long long)__double_as_longlong(v.y)) == magic;
    };
    // (i, t-1) from a chain warp of the same CTA comes through its shared-memory ring (tag keyed by the node as well)
    const bool use_ring = (pv != nullptr);
    auto rtag_ok = [&](const double2& v, int k) {
        return ((unsigned long long)__double_as_longlong(v.x) ^ (unsigned long long)__double_as_longlong(v.y)) ==
               magic + (unsigned long long)(unsigned)k * 0x9E3779B97F4A7C15ull;
    };
    // ownership of the node streams this warp walks: k (current), k-1-NL (its ring row must be there), the staged node
    const int kfirst = i0 + ((ROLE == TAME_ROLE_INPUT) ? hi : 0);
    TameOwn own_k, own_f, own_s;
    own_k.init(min(kfirst, P.n - 1), P.panel, P.world);
    own_f.init(i0, P.panel, P.world);
    own_s = own_k;
    int f_at = i0;                                                    // node own_f stands at
    auto is_mine = [&](const TameOwn& o) { return !multi || o.pw == P.rank; };
    auto own_step = [&](TameOwn& o) {
#pragma unroll
        for (int q = 0; q < STEP; ++q) o.next(P.panel, P.world);
    };

    // rows cc of Qinv Phi and Phi' Qinv (AR(1) terms of h, structured_mf.py:258,264) and the constant part of diag(P)
    double qp[DO_INP ? D : 1], pq[DO_INP ? D : 1];
    if (DO_INP) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            qp[k] = P.cst[3 * D * D + cc * D + k];
            pq[k] = P.cst[4 * D * D + cc * D + k];
        }
    }
    const double cdiag = (has_prev ? P.cst[1 * D * D + cc * D + cc] : P.cst[cc * D + cc]) + (has_next ? P.cst[2 * D * D + cc * D + cc] : 0.0);
    // running partner moments of this time step: lane c >= 2 owns column y = c-2 of G = sum_j z_j z_j' (and g[y], G[y][y]);
    // lanes 0,1 hold g = sum_j z_j -- exactly what the lane needs to form its column of the observation precision
    double Gc[DO_TOT ? NV : 1], gy = 0.0, gd = 0.0;
    if (DO_TOT) {
#pragma unroll
        for (int x = 0; x < NV; ++x) {
            double v = 0.0;
            if (c < 2) v = P.tot[(size_t)t * TOT + x];
            else if (act) v = P.tot[(size_t)t * TOT + NV + x * NV + (c - 2)];
            Gc[x] = v;
        }
        if (c >= 2 && act) {
            gy = P.tot[(size_t)t * TOT + (c - 2)];
            gd = P.tot[(size_t)t * TOT + NV + (c - 2) * NV + (c - 2)];
        }
    }
    // tot += sign * (z, z z'); z read from shared memory in z order (ring row) or from a mean vector in x order
    using TrueT = std::true_type;
    using FalseT = std::false_type;
    auto tot_update = [&](const double* m, auto xorder, double sign) {
        constexpr bool XO = decltype(xorder)::value;
        if (DO_TOT) {
            double zy = 0.0;
            if (c < 2) zy = sign;
            else if (act) zy = sign * m[XO ? tame_zidx<R>(c - 2) : c - 2];
#pragma unroll
            for (int x = 0; x < (DO_TOT ? NV : 1); ++x) Gc[x] = fma(m[XO ? tame_zidx<R>(x) : x], zy, Gc[x]);
            if (c >= 2) { gy += zy; gd = fma(zy * zy, sign, gd); }
        }
    };
    double sA, sB;   // scale pattern of P_obs: rows x<R of the z-block use sA, rows x>=R use sB
    if (c == 0) { sA = P.p0; sB = P.q; }
    else if (c == 1) { sA = P.q; sB = P.p1; }
    else if (c - 2 < R) { sA = P.p0; sB = P.q; }
    else { sA = P.q; sB = P.p1; }

    long long wait_unit = 0, wait_hand = 0, wait_chain = 0;
    bool alive = true;

    // stage the global inputs of node k this role needs (cp.async; the caller commits one group per loop iteration).  At
    // the first node of a sub-block the stamp of its streaming unit (static partner part H) is awaited first.
    auto stage = [&](int k, bool mine_s, int l) {
        const size_t cell = (size_t)k * T + t;
        const double* xm = P.Xm + cell * D;
        if (!DO_INP) {                                          // totals warp: old mean of every node, hand-over slot of foreign ones
            typename S::TStage& s = sm.tst[k & SMASK];
            if (lane < D / 2) tame_cp_async16(&s.mold[2 * lane], xm + 2 * lane, true);
            if (!mine_s && act) tame_cp_async16(&s.hand[c], hand_mine + (size_t)k * T * D, true);
            return;
        }
        typename S::Stage& s = sm.st[k & SMASK];
        if (!mine_s) {
            if (DO_TOT) {
                if (lane < D / 2) tame_cp_async16(&s.mold[2 * lane], xm + 2 * lane, true);
                if (act) tame_cp_async16(&s.hand[c], hand_mine + (size_t)k * T * D, true);
            }
            return;
        }
        if (lane < D / 2) tame_cp_async16(&s.mold[2 * lane], xm + 2 * lane, true);
        if (has_prev && act) tame_cp_async16(&s.hand[c], hand_prev + (size_t)k * T * D, true);
        if (has_next && lane >= 16 && lane < 16 + D / 2) tame_cp_async16(&s.mnext[2 * (lane - 16)], xm + D + 2 * (lane - 16), true);
        const int wlo = window_lo(k);
        const YT* yb = TameY<YT>::ptr(P) + (((size_t)l * P.n + wlo) * T + t) * 2;
#pragma unroll
        for (int u = 0; u < NWS; ++u) {
            const int sl = lane + 32 * u;
            if (wlo + sl < k) TameY<YT>::cp_async(&s.ywin[sl], yb + (size_t)sl * T * 2, true);
        }
        if (FUSED && ((k % TAME_SB) < STEP)) {                   // this warp's first node of the sub-block
            const long long c0 = clock64();
            if (P.trace != nullptr && t == 0 && lane == 0 && (k % TAME_SB) == 0) P.trace[2 * (k / TAME_SB)] = tame_globaltimer();
            int ok = 1;
            if (lane == 0) {
                const int* flag = P.unit_done + (size_t)((l / TAME_SB) * nslices + (t >> 5)) * P.nparts * TAME_NG + ((t >> 3) & (TAME_NG - 1));
                TameSpin sp;
                for (int part = 0; part < P.nparts && ok; ++part)
                    while (tame_ld_acquire(flag + part * TAME_NG) != P.epoch)
                        if (sp.expired(P.abort_flag)) { ok = 0; break; }
            }
            ok = __shfl_sync(0xffffffffu, ok, 0);
            __syncwarp();
            wait_unit += clock64() - c0;
            if (P.trace != nullptr && t == 0 && lane == 0 && (k % TAME_SB) == 0) P.trace[2 * (k / TAME_SB) + 1] = tame_globaltimer();
            if (!ok) { alive = false; return; }
        }
        const size_t lcell = (size_t)l * T + t;
        if (lane == 31) tame_cp_async16(&s.hab[0], P.hab + lcell * 2, true);
        if (lane < nparts * R) {
            const int part = lane / R, piece = lane - part * R;
            tame_cp_async16(&s.H[part][2 * piece], P.H + part * slab + lcell * NV + 2 * piece, true);
        }
    };

    {
        int ks = kfirst;
        for (int u = 0; u <= LA; ++u, ks += STEP) {
            if (alive && ks < i1) stage(ks, is_mine(own_s), own_s.lrow(P.panel));
            own_step(own_s);
            tame_cp_async_commit();
        }
    }
    for (int k = kfirst; k < i1 && alive; k += STEP) {
        const bool mine = is_mine(own_k);
        tame_cp_async_wait<LA>();
        __syncwarp();

        // ---- the ring must hold every node up to k-1-NL (chain: its own nodes, totals side: foreign nodes); the totals
        // side folds them into the running moments as it passes: node k-1-NL enters with its new mean, node k leaves
        // with its old one
        const int jf = k - 1 - NL;
        if (jf >= i0) {
            while (f_at < jf) { own_f.next(P.panel, P.world); ++f_at; }
            const long long c0 = clock64();
            if (is_mine(own_f)) {
                if (!tame_wait_smem(&sm.c_done, jf, lane, P.abort_flag)) { alive = false; break; }
            } else if (!DO_TOT) {
                if (!tame_wait_smem(&sm.f_done, jf, lane, P.abort_flag)) { alive = false; break; }
            }
            wait_chain += clock64() - c0;
            tot_update(sm.ring[jf & RMASK], FalseT{}, 1.0);
        }
        if (DO_TOT) tot_update(DO_INP ? sm.st[k & SMASK].mold : sm.tst[k & SMASK].mold, TrueT{}, -1.0);

        if (!mine) {
            if (DO_TOT) {
                // ---- node of another rank: its owner wrote {new mean, tag} straight into this rank's hand-over slots over
                // NVLink; keep the replicated X_mean, the window ring and the progress counter in step
                double2 hf = DO_INP ? sm.st[k & SMASK].hand[cc] : sm.tst[k & SMASK].hand[cc];
                TameSpin sp;
                for (;;) {
                    if (__all_sync(0xffffffffu, !act || tag_ok(hf))) break;
                    int ex = 0;
                    if (lane == 0) ex = sp.expired(P.abort_flag) ? 1 : 0;
                    if (__shfl_sync(0xffffffffu, ex, 0)) { alive = false; break; }
                    if (act) hf = tame_ld_volatile2(hand_mine + (size_t)k * T * D);
                }
                if (!alive) break;
                if (act) {
                    tame_st_cg(P.Xm + ((size_t)k * T + t) * D + c, hf.x);
                    if (c >= 2) sm.ring[k & RMASK][(c - 2 < R) ? c - 2 + R : c - 2 - R] = hf.x;
                }
                if (((k + 1) % TAME_SB) == 0 || k + 1 == i1) {
                    __threadfence();
                    __syncwarp();
                    if (lane == 0) tame_st_release(P.progress + t, k + 1);
                }
                __threadfence_block();
                __syncwarp();
                if (lane == 0) *((volatile int*)&sm.f_done) = k;
            }
        } else {
            double hval = 0.0;
            int wlo = 0, nle = 0, cnt = 0;
            if (DO_INP) {
                const typename S::Stage& s = sm.st[k & SMASK];
                double2* wbuf = sm.wbuf[hi];
                double* hin = sm.hin[hi];
                double* mprev = sm.mprev[hi];
                // ---- the window's weights  w0 = p0 y0 + q y1, w1 = q y0 + p1 y1  (structured_mf.py:324)
                wlo = window_lo(k); nle = min(NL, k - i0); cnt = (k - nle) - wlo;     // the helper sums partners wlo .. k-nle-1
#pragma unroll
                for (int u = 0; u < NWS; ++u) {
                    const int sl = lane + 32 * u;
                    if (wlo + sl < k) {
                        const double2 y = TameY<YT>::wide(s.ywin[sl]);
                        wbuf[sl] = make_double2(P.p0 * y.x + P.q * y.y, P.q * y.x + P.p1 * y.y);
                    }
                }
                // ---- AR(1) term of the successor (old mean) + static partner part
                if (c < 2) hval = s.hab[c];
                else if (act) {
                    for (int pp = 0; pp < nparts; ++pp) hval += s.H[pp][c - 2];
                }
                if (has_next) {
                    double n0 = 0.0, n1 = 0.0, n2 = 0.0;
#pragma unroll
                    for (int q = 0; q + 2 < D; q += 3) {
                        n0 = fma(pq[q], s.mnext[q], n0);
                        n1 = fma(pq[q + 1], s.mnext[q + 1], n1);
                        n2 = fma(pq[q + 2], s.mnext[q + 2], n2);
                    }
#pragma unroll
                    for (int q = (D / 3) * 3; q < D; ++q) n0 = fma(pq[q], s.mnext[q], n0);
                    hval += (n0 + n1) + n2;                                  // Phi' Qinv mu_{t+1}     (structured_mf.py:264)
                }
                // ---- (k, t-1), cheapest source first: the ring of the neighbouring chain warp (same CTA) if it is already
                // there; the staged look at the global hand-over slot (valid when the predecessor is LA+ nodes ahead, which
                // also covers a ring slot that has been overwritten since); wait for the ring; poll the global slot
                if (has_prev) {
                    double2 hv = make_double2(0.0, 0.0);
                    bool got = false;
                    const long long c0 = clock64();
                    if (use_ring && *((volatile const int*)&pv->c_done) >= k) {
                        hv = pv->mring[k & (TAME_MR - 1)][cc];
                        got = __all_sync(0xffffffffu, !act || rtag_ok(hv, k));
                    }
                    if (!got) {
                        hv = s.hand[cc];
                        got = __all_sync(0xffffffffu, !act || tag_ok(hv));
                    }
                    if (!got && use_ring) {
                        if (!tame_wait_smem(&pv->c_done, k, lane, P.abort_flag)) { alive = false; break; }
                        hv = pv->mring[k & (TAME_MR - 1)][cc];
                        got = __all_sync(0xffffffffu, !act || rtag_ok(hv, k));
                    }
                    if (!got) {
                        TameSpin sp;
                        for (;;) {
                            if (act) hv = tame_ld_volatile2(hand_prev + (size_t)k * T * D);
                            if (__all_sync(0xffffffffu, !act || tag_ok(hv))) break;
                            int ex = 0;
                            if (lane == 0) ex = sp.expired(P.abort_flag) ? 1 : 0;
                            if (__shfl_sync(0xffffffffu, ex, 0)) { alive = false; break; }
                        }
                        if (!alive) break;
                    }
                    wait_hand += clock64() - c0;
                    if (act) mprev[c] = hv.x;
                }
                __syncwarp();        // wbuf, mprev
                // ---- partial window sum over the ring
                if (R % 4 == 0) {
                    // lane = (partner phase, component quad): NGR quads x PH phases = 32 lanes; a quad lies in one half of z
                    constexpr int NGR = (NV / 4 > 0) ? NV / 4 : 1, PH = 32 / NGR;
                    const int gq = lane % NGR, ph = lane / NGR, x0 = 4 * gq;
                    const double* wsel = reinterpret_cast<const double*>(wbuf) + ((x0 < R) ? 0 : 1);
                    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0, b0 = 0.0, b1 = 0.0, b2 = 0.0, b3 = 0.0;
                    int jj = ph;
                    for (; jj + PH < cnt; jj += 2 * PH) {
                        const double wa = wsel[2 * jj], wb = wsel[2 * (jj + PH)];
                        const double2* za = reinterpret_cast<const double2*>(&sm.ring[(wlo + jj) & RMASK][x0]);
                        const double2* zb = reinterpret_cast<const double2*>(&sm.ring[(wlo + jj + PH) & RMASK][x0]);
                        const double2 za0 = za[0], za1 = za[1], zb0 = zb[0], zb1 = zb[1];
                        a0 = fma(wa, za0.x, a0); a1 = fma(wa, za0.y, a1); a2 = fma(wa, za1.x, a2); a3 = fma(wa, za1.y, a3);
                        b0 = fma(wb, zb0.x, b0); b1 = fma(wb, zb0.y, b1); b2 = fma(wb, zb1.x, b2); b3 = fma(wb, zb1.y, b3);
                    }
                    if (jj < cnt) {
                        const double wa = wsel[2 * jj];
                        const double2* za = reinterpret_cast<const double2*>(&sm.ring[(wlo + jj) & RMASK][x0]);
                        const double2 za0 = za[0], za1 = za[1];
                        a0 = fma(wa, za0.x, a0); a1 = fma(wa, za0.y, a1); a2 = fma(wa, za1.x, a2); a3 = fma(wa, za1.y, a3);
                    }
                    a0 += b0; a1 += b1; a2 += b2; a3 += b3;
#pragma unroll
                    for (int o = NGR; o < 32; o <<= 1) {
                        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
                        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
                        a2 += __shfl_xor_sync(0xffffffffu, a2, o);
                        a3 += __shfl_xor_sync(0xffffffffu, a3, o);
                    }
                    if (lane < NGR) { hin[x0] = a0; hin[x0 + 1] = a1; hin[x0 + 2] = a2; hin[x0 + 3] = a3; }
                } else {
                    // lane = (partner phase, component pair); NPP pairs x PH phases = 32 lanes
                    constexpr int NPP = (R <= 1) ? 1 : (R <= 2) ? 2 : (R <= 4) ? 4 : 8, PH = 32 / NPP;
                    const int xp = min(lane % NPP, R - 1), ph = lane / NPP, x0 = 2 * xp;
                    const bool a0 = x0 < R, a1 = x0 + 1 < R;
                    double s0 = 0.0, s1 = 0.0, u0 = 0.0, u1 = 0.0;
                    int jj = ph;
                    for (; jj + PH < cnt; jj += 2 * PH) {
                        const double2 wa = wbuf[jj], wb = wbuf[jj + PH];
                        const double2 za = *reinterpret_cast<const double2*>(&sm.ring[(wlo + jj) & RMASK][x0]);
                        const double2 zb = *reinterpret_cast<const double2*>(&sm.ring[(wlo + jj + PH) & RMASK][x0]);
                        s0 = fma(a0 ? wa.x : wa.y, za.x, s0);
                        u0 = fma(a1 ? wa.x : wa.y, za.y, u0);
                        s1 = fma(a0 ? wb.x : wb.y, zb.x, s1);
                        u1 = fma(a1 ? wb.x : wb.y, zb.y, u1);
                    }
                    if (jj < cnt) {
                        const double2 wa = wbuf[jj];
                        const double2 za = *reinterpret_cast<const double2*>(&sm.ring[(wlo + jj) & RMASK][x0]);
                        s0 = fma(a0 ? wa.x : wa.y, za.x, s0);
                        u0 = fma(a1 ? wa.x : wa.y, za.y, u0);
                    }
                    s0 += s1;
                    u0 += u1;
#pragma unroll
                    for (int o = NPP; o < 32; o <<= 1) {
                        s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                        u0 += __shfl_xor_sync(0xffffffffu, u0, o);
                    }
                    if (lane < NPP && lane < R) { hin[x0] = s0; hin[x0 + 1] = u0; }
                }
                if (has_prev) {
                    double p0 = 0.0, p1 = 0.0, p2 = 0.0;
#pragma unroll
                    for (int q = 0; q + 2 < D; q += 3) {
                        p0 = fma(qp[q], mprev[q], p0);
                        p1 = fma(qp[q + 1], mprev[q + 1], p1);
                        p2 = fma(qp[q + 2], mprev[q + 2], p2);
                    }
#pragma unroll
                    for (int q = (D / 3) * 3; q < D; ++q) p0 = fma(qp[q], mprev[q], p0);
                    hval += (p0 + p1) + p2;                                  // Qinv Phi mu_{t-1}      (structured_mf.py:258)
                }
                __syncwarp();        // hin
                if (c >= 2 && act) hval += hin[c - 2];
                // ---- node k's inputs
                typename S::Inp& in = sm.inp[k & IMASK];
                if (act) {
                    in.hrest[c] = hval;
                    in.mold[c] = s.mold[c];
                }
                if (lane < 2 * nle) {               // wl[q] <-> partner k-1-q
                    const int q = lane >> 1;
                    const double2 w = wbuf[cnt + nle - 1 - q];
                    in.wl[q][lane & 1] = (lane & 1) ? w.y : w.x;
                }
            }
            if (DO_TOT) {
                // ---- totals side: diag(P) for the naive rule, the precision column at refresh nodes (both without the
                // trailing partners: the chain adds those)
                if (P.mode == 0 && act)
                    sm.pdt[k & IMASK][c] = cdiag + ((c < 2) ? ((c == 0) ? P.p0 : P.p1) * m1 : ((c - 2 < R) ? P.p0 : P.p1) * gd);
                if (k == i0 || (k % TAME_REFRESH) == 0) {
                    // refresh node: the precision without the trailing partners, from the running totals, inverted here
                    // (in-place Gauss-Jordan); the chain warp re-enters the trailing partners by rank-2 up-dates
                    double col[D];
                    const size_t cb = (size_t)(has_prev ? 1 : 0) * D * D;
                    double c0v, c1v;
                    // the (a,b) block of P_obs is R^-1 times the partner count: the trailing partners' share is left out
                    // here, their rank-2 up-dates in the chain warp bring it back
                    const double m1r = m1 - (double)min(NL, k - i0);
                    if (c < 2) { c0v = ((c == 0) ? P.p0 : P.q) * m1r; c1v = ((c == 0) ? P.q : P.p1) * m1r; }
                    else { c0v = sA * gy; c1v = sB * gy; }
#pragma unroll
                    for (int q = 0; q < D; ++q) {
                        double v = (q == 0) ? c0v : (q == 1) ? c1v : ((q - 2 < R) ? sA : sB) * Gc[(DO_TOT && q >= 2) ? q - 2 : 0];
                        v += P.cst[cb + q * D + cc];
                        if (has_next) v += P.cst[2 * D * D + q * D + cc];
                        col[q] = act ? v : 0.0;
                    }
                    tame_gj_inverse<D, false>(col, sm.rowb, lane);
                    if (act) {
#pragma unroll
                        for (int q = 0; q < D; ++q) sm.pcol[q * DP + c] = col[q];
                    }
                }
            }
            __threadfence_block();
            __syncwarp();
            if (lane == 0) {
                if (DO_TOT) *((volatile int*)&sm.t_ready) = k;
                if (DO_INP) *((volatile int*)&sm.ready[k & IMASK]) = k;
            }
        }
        // ---- next inputs
        __syncwarp();
        {
            const int ks = k + STEP * (1 + LA);
            if (ks < i1) stage(ks, is_mine(own_s), own_s.lrow(P.panel));
        }
        own_step(own_s);
        own_step(own_k);
        tame_cp_async_commit();
    }
    // ---- drain: the last nodes' totals
    tame_cp_async_wait<0>();
    __syncwarp();
    if (ROLE == TAME_ROLE_INPUT && hi == 0 && FUSED && lane == 0 && (t == 0 || t == P.probe_t)) {      // probes of the first input warp
        unsigned long long* dbg = P.dbg + (t == 0 ? 0 : 8);
        dbg[3] = (unsigned long long)wait_unit;
        dbg[4] = (unsigned long long)wait_hand;
        dbg[5] = (unsigned long long)wait_chain;
    }
    if (!DO_TOT) return;
    for (int jf = max(i0, i1 - 1 - NL); jf < i1 && alive; ++jf) {
        while (f_at < jf) { own_f.next(P.panel, P.world); ++f_at; }
        if (is_mine(own_f) && !tame_wait_smem(&sm.c_done, jf, lane, P.abort_flag)) { alive = false; break; }
        tot_update(sm.ring[jf & RMASK], FalseT{}, 1.0);
    }
    if (!alive) return;            // watchdog: leave the running totals alone, the caller reports TAME_EHANG
    if (c >= 2 && act) {
        P.tot[(size_t)t * TOT + (c - 2)] = gy;
#pragma unroll
        for (int x = 0; x < (DO_TOT ? NV : 1); ++x) P.tot[(size_t)t * TOT + NV + x * NV + (c - 2)] = Gc[x];
    }
    if (ROLE == TAME_ROLE_ALL && FUSED && lane == 0 && (t == 0 || t == P.probe_t)) {
        unsigned long long* dbg = P.dbg + (t == 0 ? 0 : 8);
        dbg[3] = (unsigned long long)wait_unit;
        dbg[4] = (unsigned long long)wait_hand;
        dbg[5] = (unsigned long long)wait_chain;
    }
}

// ------------------------------------------------------------------------------------------------------
// chain warp of time step t
// ------------------------------------------------------------------------------------------------------
template <int R, bool FUSED, int NH, class YT>
__device__ __forceinline__ void tame_chain_warp(const TameParams& P, TameChainSmem<R, NH, YT>& sm, int lane, int t, int i0, int i1) {
    using S = TameChainSmem<R, NH, YT>;
    constexpr int D = S::D, NV = S::NV, DP = S::DP;
    constexpr int NL = TAME_NL, IMASK = TAME_NINP - 1, RMASK = S::RING - 1;
    const int T = P.T, c = lane, cc = min(c, D - 1);
    const bool act = c < D, has_next = t < T - 1;
    const bool multi = FUSED && P.npeers > 0;
    const int mode = P.mode;
    const double lr = P.lr, om = 1.0 - P.lr;
    const double rdetR = 1.0 / (P.p0 * P.p1 - P.q * P.q);
    const double R00 = P.p1 * rdetR, R11 = P.p0 * rdetR, R01 = -P.q * rdetR;      // R = (R^-1)^-1
    const unsigned long long magic = 0x5AFE000000000000ull + (unsigned long long)(unsigned)P.epoch;
    auto refresh_at = [&](int k) { return k == i0 || (k % TAME_REFRESH) == 0; };
    TameOwn own_i;
    own_i.init(i0, P.panel, P.world);
    auto is_mine = [&](const TameOwn& o) { return !multi || o.pw == P.rank; };
    // component c of x = [a,b,U,V] sits at zpos in z = [V,U]; its h entry takes w0 (U rows) or w1 (V rows)
    const int zc = (cc >= 2) ? cc - 2 : 0;                       // index of this lane's component in h[2:], H, hin, ring rows
    const int zpos = (zc < R) ? zc + R : zc - R;                 // where its own new value goes in a ring row
    const int wsel = (zc < R) ? 0 : 1;
    const bool zlane = act && c >= 2;
    const double sdiag = (zc < R) ? P.p0 : P.p1;
    const bool lo = c < 2;

    double cw[D];            // raw inverse, column (= row) c; after a down-date it is B_{i+1}^-1
#pragma unroll
    for (int k = 0; k < D; ++k) cw[k] = 0.0;
    const bool probe = FUSED && lane == 0 && (t == 0 || t == P.probe_t);     // timing probes (dbg[0..7]: t=0, [8..15]: t=probe_t)
    unsigned long long* dbg = P.dbg + (t == 0 ? 0 : 8);
    long long wait_in = 0, wait_next = 0;
    int ncell = 0;
    if (probe) dbg[0] = tame_globaltimer();
    // the other ranks' hand-over buffers (kernel parameters -> registers: no indexed constant loads inside the node loop)
    const int npeers = FUSED ? P.npeers : 0;
    double2* peer[7];
#pragma unroll
    for (int pr = 0; pr < 7; ++pr) peer[pr] = P.hand_peer[pr];
    // running addresses of (i, t, c)
    const size_t nstride = (size_t)T * D;
    size_t xoff = ((size_t)i0 * T + t) * D + cc;

    bool prev_mine = true;
    for (int i = i0; i < i1; ++i, xoff += nstride, own_i.next(P.panel, P.world)) {
        if (!is_mine(own_i)) { prev_mine = false; continue; }
        const bool refresh = refresh_at(i);
        {
            const long long c0 = clock64();
            if (!tame_wait_smem(&sm.ready[i & IMASK], i, lane, P.abort_flag)) return;
            if ((refresh || mode == 0) && !tame_wait_smem(&sm.t_ready, i, lane, P.abort_flag)) return;
            // the trailing partners' ring rows: written by this warp, or -- foreign nodes with a separate totals warp -- awaited
            if (NH > 1 && !prev_mine && i > i0 && !tame_wait_smem(&sm.f_done, i - 1, lane, P.abort_flag)) return;
            wait_in += clock64() - c0;
        }
        prev_mine = true;
        const typename S::Inp& in = sm.inp[i & IMASK];
        const int nle = min(NL, i - i0);
        const double mo = in.mold[cc];
        // ---- h: the helper's part + the trailing partners i-1-q (new z in the ring)
        double hval = in.hrest[cc];
        double pdiag = (mode == 0) ? sm.pdt[i & IMASK][cc] : 0.0;
#pragma unroll
        for (int q = 0; q < NL; ++q) {
            const double zj = sm.ring[(i - 1 - q) & RMASK][zc];
            const double w = in.wl[q][wsel];
            if (q < nle && zlane) {
                hval = fma(w, zj, hval);
                pdiag = fma(sdiag * zj, zj, pdiag);
            }
        }
        if (act) sm.hvec[c] = hval;

        // ---- the inverse.  Between refreshes P_i = P_{i-1} - G(z_i^old) + G(z_{i-1}^new): node i leaves with its old mean
        // (pass 0), node i-1 re-enters with its new mean (pass 1).  At a refresh node the helper hands over the inverse of
        // the precision without the trailing partners (built from the running totals, Gauss-Jordan) and passes 1..nle
        // re-enter those partners.  One rolled loop: the rank-2 code exists once (instruction cache).
        int pass = 0, pass_end = 2;
        if (refresh) {
#pragma unroll
            for (int k = 0; k < D; ++k) cw[k] = act ? sm.pcol[k * DP + c] : 0.0;
            pass = 1;
            pass_end = nle + 1;
        }
#pragma unroll 1
        for (; pass < pass_end; ++pass) {
            double z[NV];
            if (pass == 0) {
                const double* mn = in.mold;
                if (R % 2 == 0) {
                    const double2* mu2 = reinterpret_cast<const double2*>(mn + 2);          // U block
                    const double2* mv2 = reinterpret_cast<const double2*>(mn + 2 + R);      // V block
#pragma unroll
                    for (int x = 0; x < R / 2; ++x) {
                        const double2 v = mv2[x], u = mu2[x];
                        z[2 * x] = v.x; z[2 * x + 1] = v.y; z[R + 2 * x] = u.x; z[R + 2 * x + 1] = u.y;
                    }
                } else {
#pragma unroll
                    for (int x = 0; x < NV; ++x) z[x] = mn[tame_zidx<R>(x)];
                }
            } else {
                const double2* zr = reinterpret_cast<const double2*>(sm.ring[(i - pass) & RMASK]);
#pragma unroll
                for (int x = 0; x < R; ++x) { const double2 v = zr[x]; z[2 * x] = v.x; z[2 * x + 1] = v.y; }
            }
            double f0, f1;
            tame_rank2_F<R>(cw, z, f0, f1);
            __syncwarp();                                   // the previous pass has read Fs
            sm.Fs[0][lane] = make_double2(f0, f1);
            __syncwarp();
            tame_rank2_apply<R>(cw, z, f0, f1, sm.Fs[0], pass == 0 ? -1.0 : 1.0, R00, R01, R11);
        }
        __syncwarp();                                       // hvec
        // ---- cw = raw C_i.  Mean (factorisation rule applied to the row), damped write, hand-over
        {
            double h[D];
            const double2* hv2 = reinterpret_cast<const double2*>(sm.hvec);
#pragma unroll
            for (int k = 0; k < D / 2; ++k) { const double2 v = hv2[k]; h[2 * k] = v.x; h[2 * k + 1] = v.y; }
            double m0 = 0.0, m1 = 0.0, m2 = 0.0;
            if (mode == 2) {                                                         // structured_mf.py:270-273
                if (lo) { m0 = cw[0] * h[0]; m1 = cw[1] * h[1]; }
                else {
#pragma unroll
                    for (int k = 2; k < D; ++k) {
                        if (k % 3 == 0) m0 = fma(cw[k], h[k], m0); else if (k % 3 == 1) m1 = fma(cw[k], h[k], m1); else m2 = fma(cw[k], h[k], m2);
                    }
                }
            } else {
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    if (k % 3 == 0) m0 = fma(cw[k], h[k], m0); else if (k % 3 == 1) m1 = fma(cw[k], h[k], m1); else m2 = fma(cw[k], h[k], m2);
                }
            }
            double mu = (m0 + m1) + m2;
            if (mode != 0) mu = fma(1e-6, hval, mu);                                 // (C + 1e-6 I) h   :277-279
            const double mnew = lr * mu + om * mo;                                   // :282-284
            if (act) {
                tame_st_cg(P.Xm + xoff, mnew);
                if (has_next || multi) {
                    const unsigned long long tag = (unsigned long long)__double_as_longlong(mnew) ^ magic;
                    const double2 slotv = make_double2(mnew, __longlong_as_double((long long)tag));
                    __stcg(P.hand + xoff, slotv);
                    if (FUSED) {
#pragma unroll
                        for (int pr = 0; pr < 7; ++pr)
                            if (pr < npeers) __stcg(peer[pr] + xoff, slotv);                            // NVLink peer stores
                    }
                }
                if (c >= 2) sm.ring[i & RMASK][zpos] = mnew;
                {   // the next time step's helper, if it lives in this CTA, takes the mean from here
                    const unsigned long long rtag = (unsigned long long)__double_as_longlong(mnew) ^
                                                    (magic + (unsigned long long)(unsigned)i * 0x9E3779B97F4A7C15ull);
                    sm.mring[i & (TAME_MR - 1)][c] = make_double2(mnew, __longlong_as_double((long long)rtag));
                }
                // raw covariance column -> global scratch; k_covblend applies mask / symmetrisation / jitter / damping
                // (naive: only the diagonal 1 / (diag(P) + 1e-8) is kept, naive_mf.py:271-274)
                const int l = own_i.lrow(P.panel);
                double* cr = P.Craw + ((size_t)l * T + t) * (D * D) + c;
                if (mode != 0) {
#pragma unroll
                    for (int k = 0; k < D; ++k) __stcs(cr + k * D, cw[k]);
                } else {
                    __stcs(cr + c * D, 1.0 / (pdiag + 1e-8));
                }
            }
        }
        __threadfence_block();
        __syncwarp();
        if (lane == 0) *((volatile int*)&sm.c_done) = i;
        ++ncell;
        // progress is only consumed by the streaming CTAs, at sub-block granularity: one fence per 32 nodes
        if (((i + 1) % TAME_SB) == 0 || i + 1 == i1) {
            __threadfence();
            __syncwarp();
            if (lane == 0) tame_st_release(P.progress + t, i + 1);
            if (FUSED && P.trace != nullptr && lane == 0 && t < 16) {      // when time step t released sub-block i / 32
                const int nsb = (P.n + TAME_SB - 1) / TAME_SB;
                P.trace[6 * nsb + 16 * (i / TAME_SB) + t] = tame_globaltimer();
            }
        }
    }
    if (probe) {
        dbg[2] = tame_globaltimer();
        dbg[1] = (unsigned long long)wait_next;
        dbg[6] = (unsigned long long)ncell;
        dbg[7] = (unsigned long long)wait_in;
    }
}

// One chain CTA (8 warps).  NH = 1: warps 0..3 are the chain warps of 4 consecutive time steps (one per SM sub-partition),
// warps 4..7 their helpers.  NH = 2: two time steps, each with a chain warp, a totals warp and two input warps; the roles of
// the second time step are rotated by one so that every sub-partition carries one chain-or-totals warp and one input warp.
template <int NH>
struct TameTeam {
    static constexpr int TPC = (NH == 1) ? 4 : 2;        // time steps per chain CTA
};
template <int R, bool FUSED, int NH, class YT>
__device__ __forceinline__ void tame_chain_body(const TameParams& P, unsigned char* smem_raw, int cta, int i0, int i1) {
    using S = TameChainSmem<R, NH, YT>;
    constexpr int TPC = TameTeam<NH>::TPC;
    S* team = reinterpret_cast<S*>(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < TPC) {
        S& q = team[threadIdx.x];
        for (int k = 0; k < TAME_NINP; ++k) q.ready[k] = i0 - 1;
        q.t_ready = i0 - 1; q.f_done = i0 - 1; q.c_done = i0 - 1;
    }
    __syncthreads();
    if (NH == 1) {
        const bool is_helper = warp >= TPC;
        const int tg = warp - (is_helper ? TPC : 0);
        if (tg >= TPC) return;
        const int t = cta * TPC + tg;
        if (t >= P.T) return;
        if (is_helper) tame_chain_helper<R, FUSED, NH, TAME_ROLE_ALL, YT>(P, team[tg], (tg > 0) ? &team[tg - 1] : nullptr, lane, t, 0, i0, i1);
        else tame_chain_warp<R, FUSED, NH, YT>(P, team[tg], lane, t, i0, i1);
    } else {
        const int tg = warp >> 2;
        if (tg >= TPC) return;
        const int role = ((warp & 3) + 4 - tg) & 3;           // 0 chain, 1 totals, 2/3 input warps
        const int t = cta * TPC + tg;
        if (t >= P.T) return;
        const S* pv = (tg > 0) ? &team[tg - 1] : nullptr;
        if (role == 0) tame_chain_warp<R, FUSED, NH, YT>(P, team[tg], lane, t, i0, i1);
        else if (role == 1) tame_chain_helper<R, FUSED, NH, TAME_ROLE_TOTALS, YT>(P, team[tg], pv, lane, t, 0, i0, i1);
        else tame_chain_helper<R, FUSED, NH, TAME_ROLE_INPUT, YT>(P, team[tg], pv, lane, t, role - 2, i0, i1);
    }
}


// ------------------------------------------------------------------------------------------------------
// k_covblend: X_cov[i,t] = lr * rule(C_raw) + (1 - lr) * X_cov[i,t] for the rank's own nodes, one thread per element.
//   good : rule(C) = (C + C')/2 + 1e-6 I                        structured_mf.py:276-277, damping :285-287
//   bad  : the 2 x 2r cross blocks are zeroed first             :270-273
//   naive: rule = diag(1 / (diag(P) + 1e-8)), kept on the diagonal of the scratch     naive_mf.py:271-274, 280-282
// ------------------------------------------------------------------------------------------------------
template <int R>
__device__ __forceinline__ void tame_covblend_impl(const TameParams& P, double* tile_all, int bid, int nb) {
    // one warp per (own node, t) block: the raw block goes through shared memory once (coalesced), the transposed partner
    // of every element is read from there.  tile_all: 8 * D * (D+1) doubles of shared memory.
    constexpr int D = 2 + 2 * R, DD = D * D, DP = D + 1, NE = (DD + 31) / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* tile = tile_all + warp * (D * DP);
    const double lr = P.lr, om = 1.0 - P.lr;
    const long ncell = (long)P.nloc * P.T;
    for (long cell = (long)bid * 8 + warp; cell < ncell; cell += (long)nb * 8) {
        const int l = (int)(cell / P.T), t = (int)(cell - (long)l * P.T);
        const int i = tame_grow(l, P.panel, P.world, P.rank);
        const double* cr = P.Craw + (size_t)cell * DD;
        double* xc = P.Xc + ((size_t)i * P.T + t) * DD;
        double old[NE];
#pragma unroll
        for (int m = 0; m < NE; ++m) {
            const int e = lane + 32 * m;
            if (e < DD) {
                const int row = e / D, col = e - row * D;
                tile[row * DP + col] = __ldcs(cr + e);
                old[m] = xc[e];
            }
        }
        __syncwarp();
#pragma unroll
        for (int m = 0; m < NE; ++m) {
            const int e = lane + 32 * m;
            if (e < DD) {
                const int row = e / D, col = e - row * D;
                double cf;
                if (P.mode == 0) cf = (row == col) ? tile[row * DP + col] : 0.0;
                else {
                    const bool masked = (P.mode == 2) && ((row < 2) != (col < 2));
                    cf = masked ? 0.0 : 0.5 * (tile[row * DP + col] + tile[col * DP + row]);
                    if (row == col) cf += 1e-6;
                }
                __stcs(xc + e, lr * cf + om * old[m]);
            }
        }
        __syncwarp();
    }
}
template <int R>
__global__ void __launch_bounds__(256) k_covblend(TameParams P) {
    constexpr int D = 2 + 2 * R;
    __shared__ double tile[8 * D * (D + 1)];
    tame_covblend_impl<R>(P, tile, blockIdx.x, gridDim.x);
}

// stand-alone chain launch over one 64-node block (multi-GPU path); cooperative, grid = ceil(T/8)
template <int R, class YT>
__global__ void __launch_bounds__(2 * TAME_CHAIN_WPC * 32, 1) k_chain(TameParams P, int i0, int i1) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    tame_chain_body<R, false, 1, YT>(P, smem_raw, blockIdx.x, i0, i1);
}

// ------------------------------------------------------------------------------------------------------
// k_sweep: one whole Gauss-Seidel sweep in ONE persistent cooperative launch (single-GPU path).
//   CTAs [0, n_chain_ctas)   run the chain over all nodes 0..n-1 (tame_chain_body<FUSED>): no pipeline refill.
//   the remaining CTAs       are streaming workers.  A unit = (32-row sub-block sb, 32-step time slice).  A worker
//       takes units in ascending order from an atomic counter, keeps the unit's 32 x 32 x 2R partner sums in
//       registers, streams  (a) the static upper part j > k (partners still carrying their old means when row k
//       is updated) immediately and (b) its share of the lower columns j < (sb-WBACK)*32 (new means) as the chain's progress
//       counters release them, then writes H once (no read-modify-write, no atomics) and stamps unit_done.
//   The chain's helpers wait for a sub-block's stamps (one per group of 8 time steps) before entering it and cover the last
//   (up to) 96 / 128 partners (narrow / wide team) inline.
// Every Y entry is read exactly once per sweep; the schedule is the reference's.
// grid = n_chain_ctas + workers (all co-resident), block 256, dynamic smem = max of the two roles.
// ------------------------------------------------------------------------------------------------------
template <int R, int RW, int NH, class YT>
__device__ __forceinline__ void tame_sweep_body(const TameParams& P, unsigned char* smem_raw) {
    static_assert(8 * RW == TAME_SB, "a streaming unit is one sub-block of rows");
    if ((int)blockIdx.x < P.n_chain_ctas) {
        tame_chain_body<R, true, NH, YT>(P, smem_raw, blockIdx.x, 0, P.n);
        return;
    }
    constexpr int NV = 2 * R, JC = TameStream<R, RW, YT>::JC;
    __shared__ int s_val;
    __shared__ int s_dg[TAME_NG], s_plan[3];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nslices = (P.T + 31) / 32, nsb = (P.nloc + TAME_SB - 1) / TAME_SB, nunits = nsb * nslices * P.nparts;   // local sub-blocks
    for (;;) {
        if (tid == 0) s_val = atomicAdd(P.unit_counter, 1);
        __syncthreads();
        const int u = s_val;
        __syncthreads();
        if (u >= nunits) break;
        const int part = u % P.nparts, us = u / P.nparts;            // unit = (sub-block, time slice, column part)
        const int lsb = us / nslices, slice = us - lsb * nslices;                 // local sub-block (storage order)
        const int kbase = tame_grow(lsb * TAME_SB, P.panel, P.world, P.rank);    // its first node
        const int sb = kbase / TAME_SB, kw = kbase + warp * RW;
        const int t0 = slice * 32, t = t0 + lane;
        const bool tv = t < P.T;
        double accA[RW][R], accB[RW][R];
#pragma unroll
        for (int rr = 0; rr < RW; ++rr)
#pragma unroll
            for (int a = 0; a < R; ++a) accA[rr][a] = accB[rr][a] = 0.0;
        const YT* yrow[RW];
        bool rv[RW];
#pragma unroll
        for (int rr = 0; rr < RW; ++rr) {
            const int k = kw + rr;
            rv[rr] = (k < P.n) && tv;
            yrow[rr] = TameY<YT>::ptr(P) + ((size_t)tame_lrow(min(k, P.n - 1), P.panel, P.world) * P.n * P.T + (tv ? t : 0)) * 2;
        }
        // optional trace of the unit (sub-block, slice 0, part 0): claim, upper part done, group 0 urgent, group 0 stamped
        unsigned long long* utr = (P.trace != nullptr && slice == 0 && part == P.nparts - 1 && tid == 0) ? P.trace + 2 * nsb + 4 * lsb : nullptr;
        if (utr) utr[0] = tame_globaltimer();
        // (a) static upper part: this part's share of the columns j > k
        {
            const int ub = ((kbase + 1) / JC) * JC;
            const int len = (((P.n - ub + P.nparts - 1) / P.nparts + JC - 1) / JC) * JC;
            const int jb = ub + part * len, je = min(P.n, jb + len);
            // convoy: start where the other streaming CTAs of this column part currently are and wrap around, so that a
            // partner-record chunk fetched from HBM by one CTA is L2-hot for the rest (the records are re-read by every
            // row tile: 151 MB at config 4, more than L2 can hold next to the Y stream)
            int start = jb;
            if (je - jb > 64 * JC && !P.deterministic) {
                if (tid == 0) s_val = *((volatile int*)(P.cursor + part));
                __syncthreads();
                const int cur = s_val;
                __syncthreads();
                if (cur > jb && cur < je) start = jb + ((cur - jb) / JC) * JC;
            }
            tame_stream_cols<R, RW, YT>(P, smem_raw, yrow, rv, kw, t0, start, je, true, accA, accB, P.cursor + part);
            if (start > jb) tame_stream_cols<R, RW, YT>(P, smem_raw, yrow, rv, kw, t0, jb, start, true, accA, accB, P.cursor + part);
        }
        // (b) lower columns, released by the chain (carried by part 0).  The unit's 32 time steps are followed as TAME_NG
        // groups of 8: the chain warps of a slice are skewed by ~2 us per time step, so the first group of a slice reaches
        // the unit's rows long before the last group has released the final columns.  Far from the diagonal all groups
        // advance together (one full-width pass per release); a group whose final columns are out goes alone (the other
        // lanes are masked), writes its part of H and is stamped separately -- its chain warps wait for nothing else.
        if (utr) utr[1] = tame_globaltimer();
        // the lower columns [0, (sb - WBACK) * 32) are dealt to the unit's column parts in contiguous 32-aligned ranges
        // [lowbeg, lowend): a late sub-block's backlog (everything the chain released before the unit was claimed) is
        // worked off by all parts in parallel; the last part carries the final release
        const int lowall = max(0, (sb - TAME_WBACK(NH)) * TAME_SB);
        const int lowq = ((lowall / TAME_SB + P.nparts - 1) / P.nparts) * TAME_SB;
        const int lowbeg = min(lowall, part * lowq), lowend = min(lowall, lowbeg + lowq);
        // CTA-uniform bookkeeping lives in shared memory (the accumulators own the registers): s_dg[g] = columns done by
        // group g, s_plan = {c0, c1, active mask} of the next pass; `stamped` is a bit mask
        if (tid < TAME_NG) s_dg[tid] = (t0 + 8 * tid < P.T) ? lowbeg : lowend;
        int stamped = 0, spins = 0;
        __syncthreads();
        for (;;) {
            // ---- groups that are complete: write their H rows once, stamp
            int newly = 0, all_done = 1;
#pragma unroll
            for (int g = 0; g < TAME_NG; ++g) {
                const bool fin = s_dg[g] >= lowend;
                if (fin && !((stamped >> g) & 1)) newly |= 1 << g;
                all_done &= fin ? 1 : 0;
            }
            if (newly) {
                if ((newly >> (lane >> 3)) & 1) {
#pragma unroll
                    for (int rr = 0; rr < RW; ++rr) {
                        const int k = kw + rr;
                        if (k < P.n && tv) {
                            double* h = P.H + (size_t)part * P.nloc * P.T * NV + ((size_t)tame_lrow(k, P.panel, P.world) * P.T + t) * NV;
#pragma unroll
                            for (int a = 0; a < R; ++a) {
                                __stcg(h + a, accA[rr][a]);
                                __stcg(h + R + a, accB[rr][a]);
                            }
                        }
                    }
                }
                __threadfence();
                __syncthreads();
                if (tid < TAME_NG && ((newly >> tid) & 1)) tame_st_release(P.unit_done + (size_t)u * TAME_NG + tid, P.epoch);
                if (utr && (newly & 1)) utr[3] = tame_globaltimer();
                stamped |= newly;
            }
            if (all_done) break;
            // ---- what the chain has released per group -> plan of the next pass (thread 0 decides, everybody follows)
            if (warp == 0) {
                int v = (t0 + lane < P.T) ? tame_ld_acquire(P.progress + t0 + lane) : 0x7fffffff;
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
                int tg[TAME_NG];
#pragma unroll
                for (int g = 0; g < TAME_NG; ++g) tg[g] = min(lowend, max(lowbeg, (__shfl_sync(0xffffffffu, v, 8 * g) / TAME_SB) * TAME_SB));
                if (lane == 0) {
                    if (++spins > TAME_SPIN_LIMIT / 8) atomicExch(P.abort_flag, 1);
                    int c0 = -1, c1 = 0, mask = 0;
                    if (*((volatile int*)P.abort_flag)) c0 = -2;
                    else {
#pragma unroll
                        for (int g = 0; g < TAME_NG; ++g)            // urgent: a group whose final columns are released
                            if (c0 < 0 && s_dg[g] < lowend && tg[g] >= lowend) { c0 = s_dg[g]; c1 = lowend; }
                        if (c0 >= 0) {
#pragma unroll
                            for (int g = 0; g < TAME_NG; ++g) if (s_dg[g] == c0 && tg[g] >= lowend) mask |= 1 << g;
                        } else {
                            // otherwise, of the groups WITH released columns, those furthest behind advance together (a
                            // worker that is behind finds every group far ahead and makes one full-width pass; a parked
                            // worker has nothing better to do than to follow each group eagerly, so that a group's final
                            // pass is one 32-column slab: the chain warps of a launch drift apart until this coupling
                            // stops them, so that final pass sits on the chain's critical path)
                            int dmin = 0x7fffffff, tmin = 0x7fffffff;
#pragma unroll
                            for (int g = 0; g < TAME_NG; ++g) if (tg[g] > s_dg[g]) dmin = min(dmin, s_dg[g]);
#pragma unroll
                            for (int g = 0; g < TAME_NG; ++g) if (tg[g] > s_dg[g] && s_dg[g] == dmin) tmin = min(tmin, tg[g]);
                            if (dmin != 0x7fffffff) {
                                c0 = dmin; c1 = tmin;
#pragma unroll
                                for (int g = 0; g < TAME_NG; ++g) if (tg[g] > s_dg[g] && s_dg[g] == dmin) mask |= 1 << g;
                            }
                        }
                    }
                    s_plan[0] = c0; s_plan[1] = c1; s_plan[2] = mask;
                    if (utr && c1 == lowend && (mask & 1) && c0 >= 0) utr[2] = tame_globaltimer();
                }
            }
            __syncthreads();
            const int c0 = s_plan[0], c1 = s_plan[1], mask = s_plan[2];
            __syncthreads();
            if (c0 == -2) break;                             // abort: leave without stamping
            if (c0 < 0) { __nanosleep(128); continue; }
            const bool lane_on = (mask >> (lane >> 3)) & 1;      // lanes of the other groups copy nothing and add zeros
            tame_stream_cols<R, RW, YT>(P, smem_raw, yrow, rv, kw, t0, c0, c1, false, accA, accB, nullptr, lane_on);
            if (tid < TAME_NG && ((mask >> tid) & 1)) s_dg[tid] = c1;
            __syncthreads();
        }
    }
}

template <int R, int RW, int NH, class YT>
__global__ void __launch_bounds__(256, 1) k_sweep(TameParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    tame_sweep_body<R, RW, NH, YT>(P, smem_raw);
}

// ------------------------------------------------------------------------------------------------------
// k_llmse: fused expected-log-likelihood quadratic form + reconstruction error, one pass over Y.
//   e0 = y0 - (a_i + b_j + U_i.V_j), e1 = y1 - (a_j + b_i + U_j.V_i)        static_ame.py:226-236
//   sq   += e0^2 + e1^2                        for all i != j               temporal_ame.py:284-290
//   quad += p0 e0^2 + 2 q e0 e1 + p1 e1^2      for i < j only               structured_mf.py:136-139
// Same streaming tile as k_contract (TameStream).  grid (ceil(T/32), ceil(nloc/(8*RW))), block 256;
// partial (grid.y*grid.x, 2).
// ------------------------------------------------------------------------------------------------------
// NW warps x RW rows = 32 rows per CTA at the same ring size.  Every warp reads each partner's record (144 B per lane at
// r = 8) from shared memory, so the record traffic of the shared-memory pipe grows with NW: at 16 x 2 that pipe was 79 % busy
// (ncu l1tex__data_pipe_lsu_wavefronts, short_scoreboard the top stall); 8 x 4 halves the record share (16.9 -> 14.1 ms).
// SYM: Y was verified mirror-consistent at bind time (Y[j,i,t,:] == swap(Y[i,j,t,:]) bit for bit, which the reference's
// generate_data guarantees, temporal_ame.py:209-216): the residuals of (j,i) are those of (i,j) swapped, so the pass only
// streams the partners j > i and doubles the squared error.  Otherwise the full pass runs.
template <int R, int RW, int NW, bool SYM, class YT>
__global__ void __launch_bounds__(NW * 32, 1) k_llmse(TameParams P, double* partial) {
    using TS = TameStream<R, RW, YT>;
    using Y2 = typename TameY<YT>::V2;
    constexpr int D = TS::D, JC = TS::JC, PD = TS::PD, RS = TS::RS, RT = NW * RW, NT = NW * 32;
    static_assert(NW * RW == 32, "32-row tile");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Y2 (*Yr)[RW][NT] = reinterpret_cast<Y2 (*)[RW][NT]>(smem_raw);
    double (*Mb)[JC][32][RS] = reinterpret_cast<double (*)[JC][32][RS]>(smem_raw + (size_t)PD * RW * NT * sizeof(Y2));
    __shared__ double red[2][NW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int t0 = blockIdx.x * 32, t = t0 + lane;
    const bool tv = t < P.T;
    const int lw = blockIdx.y * RT + warp * RW;

    double oa[RW], ob[RW], oU[RW][R], oV[RW][R];
    const YT* yrow[RW];
    int gi[RW];
    bool rv[RW];
#pragma unroll
    for (int rr = 0; rr < RW; ++rr) {
        int l = lw + rr;
        rv[rr] = (l < P.nloc) && tv;
        l = min(l, P.nloc - 1);
        gi[rr] = tame_grow(l, P.panel, P.world, P.rank);
        const double* m = P.Xm + ((size_t)gi[rr] * P.T + (tv ? t : 0)) * D;
        oa[rr] = m[0];
        ob[rr] = m[1];
#pragma unroll
        for (int a = 0; a < R; ++a) { oU[rr][a] = m[2 + a]; oV[rr][a] = m[2 + R + a]; }
        yrow[rr] = TameY<YT>::ptr(P) + ((size_t)l * P.n * P.T + (tv ? t : 0)) * 2;
    }
    const size_t jstride = (size_t)P.T * 2;
    // per-row moment accumulators: upper partners (j > i) feed S00 = sum e0^2, S01 = sum e0 e1, S11 = sum e1^2 (the
    // quadratic form is p0 S00 + 2q S01 + p1 S11), lower partners only the squared error SL.  Invalid rows / time steps
    // are dropped in the epilogue, so the inner loop carries no per-element predicate outside the diagonal chunks.
    double S00[RW], S01[RW], S11[RW], SL[RW];
#pragma unroll
    for (int rr = 0; rr < RW; ++rr) S00[rr] = S01[rr] = S11[rr] = SL[rr] = 0.0;
    const int gfirst = tame_grow(min(blockIdx.y * RT, P.nloc - 1), P.panel, P.world, P.rank);   // first node of the tile
    // partner range of this CTA: SYM skips the partners below the tile; gridDim.z splits the range when the grid would not
    // fill the GPU otherwise (few rows per rank on many GPUs)
    const int jlo = SYM ? (gfirst / JC) * JC : 0;
    const int zlen = (((P.n - jlo + (int)gridDim.z - 1) / (int)gridDim.z + JC - 1) / JC) * JC;
    const int jbeg = jlo + (int)blockIdx.z * zlen, jend = min(P.n, jbeg + zlen);
    const int nchunks = (jend > jbeg) ? (jend - jbeg + JC - 1) / JC : 0;

    auto issue_y = [&](int j, int slot) {
#pragma unroll
        for (int rr = 0; rr < RW; ++rr) {
            const bool ok = rv[rr] && (j < jend) && (SYM ? (j > gi[rr]) : (j != gi[rr]));
            TameY<YT>::cp_async(&Yr[slot][rr][tid], yrow[rr] + (size_t)min(j, P.n - 1) * jstride, ok);
        }
    };
    // fast path of the record staging (see tame_stream_cols)
    const bool m_fast = (RS == D) && (t0 + 32 <= P.T);
    const size_t m_gap = (size_t)P.T * D - 32 * D;
    auto issue_m = [&](int buf, int jc) {
        if (m_fast && jc + JC <= P.n) {
            const double* base = P.Xm + ((size_t)jc * P.T + t0) * D;
            double* dst = &Mb[buf][0][0][0];
#pragma unroll
            for (int it = 0; it < (JC * 32 * TS::PIECES + NT - 1) / NT; ++it) {
                const int e = tid + it * NT;
                if ((it + 1) * NT <= JC * 32 * TS::PIECES || e < JC * 32 * TS::PIECES) {
                    const int jj = e / (32 * TS::PIECES);
                    tame_cp_async16(dst + 2 * e, base + 2 * e + jj * m_gap, true);
                }
            }
            return;
        }
        for (int e = tid; e < JC * 32 * TS::PIECES; e += NT) {
            const int piece = e % TS::PIECES, tl = (e / TS::PIECES) & 31, jj = e / (TS::PIECES * 32);
            const int j = jc + jj, tt = t0 + tl;
            const bool ok = (j < jend) && (tt < P.T);
            const double* src = P.Xm + ((size_t)min(j, P.n - 1) * P.T + min(tt, P.T - 1)) * D + piece * 2;
            tame_cp_async16(&Mb[buf][jj][tl][piece * 2], src, ok);
        }
    };
    if (nchunks > 0) issue_m(0, jbeg);
#pragma unroll
    for (int s = 0; s < PD; ++s) {
        issue_y(jbeg + s, s);
        tame_cp_async_commit();
    }
    for (int c = 0; c < nchunks; ++c) {
        const int jc = jbeg + c * JC, buf = c & 1;
        // chunk-uniform case: 0 all partners below the tile's rows, 1 all above, 2 touches the tile's own nodes / the tail
        const int kind = (jc + JC <= gfirst) ? 0 : ((jc > gfirst + RT - 1 && jc + JC <= jend) ? 1 : 2);
#pragma unroll
        for (int jj = 0; jj < JC; ++jj) {
            const int j = jc + jj;
            tame_cp_async_wait<PD - 1>();
            if (jj == 0) {
                __syncthreads();
                if (c + 1 < nchunks) issue_m(buf ^ 1, jc + JC);
            }
            const double* rec = &Mb[buf][jj][lane][0];
            const double aj = rec[0], bj = rec[1];
            double d0[RW], d1[RW];
#pragma unroll
            for (int rr = 0; rr < RW; ++rr) { d0[rr] = oa[rr] + bj; d1[rr] = aj + ob[rr]; }   // (a_i + b_j), (a_j + b_i)
#pragma unroll
            for (int a = 0; a < R; ++a) {
                const double uj = rec[2 + a], vj = rec[2 + R + a];
#pragma unroll
                for (int rr = 0; rr < RW; ++rr) {
                    d0[rr] = fma(oU[rr][a], vj, d0[rr]);
                    d1[rr] = fma(uj, oV[rr][a], d1[rr]);
                }
            }
#pragma unroll
            for (int rr = 0; rr < RW; ++rr) {
                const double2 y = TameY<YT>::wide(Yr[jj][rr][tid]);
                const double e0 = y.x - d0[rr], e1 = y.y - d1[rr];
                if (kind == 1) {
                    S00[rr] = fma(e0, e0, S00[rr]);
                    S01[rr] = fma(e0, e1, S01[rr]);
                    S11[rr] = fma(e1, e1, S11[rr]);
                } else if (kind == 0) {
                    SL[rr] = fma(e0, e0, SL[rr]);
                    SL[rr] = fma(e1, e1, SL[rr]);
                } else if (j < jend && j != gi[rr]) {
                    if (j > gi[rr]) {
                        S00[rr] = fma(e0, e0, S00[rr]);
                        S01[rr] = fma(e0, e1, S01[rr]);
                        S11[rr] = fma(e1, e1, S11[rr]);
                    } else if (!SYM) {
                        SL[rr] = fma(e0, e0, SL[rr]);
                        SL[rr] = fma(e1, e1, SL[rr]);
                    }
                }
            }
            issue_y(j + PD, jj);
            tame_cp_async_commit();
        }
    }
    tame_cp_async_wait<0>();
    double sq = 0.0, quad = 0.0;
#pragma unroll
    for (int rr = 0; rr < RW; ++rr) {
        if (rv[rr]) {
            sq += SYM ? 2.0 * (S00[rr] + S11[rr]) : (S00[rr] + S11[rr]) + SL[rr];
            quad += P.p0 * S00[rr] + 2.0 * P.q * S01[rr] + P.p1 * S11[rr];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
        quad += __shfl_xor_sync(0xffffffffu, quad, o);
    }
    if (lane == 0) { red[0][warp] = sq; red[1][warp] = quad; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0, qd = 0.0;
#pragma unroll
        for (int w = 0; w < NW; ++w) { s += red[0][w]; qd += red[1][w]; }
        size_t b = ((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        partial[b * 2 + 0] = s;
        partial[b * 2 + 1] = qd;
    }
}

// ------------------------------------------------------------------------------------------------------
// k_llmse_mma: the same pass with the bilinear terms on the FP64 tensor cores (mma.sync.m8n8k4.f64 = DMMA).
//   For a fixed time step the 8x8 blocks  d0[i][j] = U_i.V_j  and  d1[i][j] = V_i.U_j  of an (8 rows x 8 partners) tile
//   are R/4 DMMA each: A = the tile's own rows (kept in registers for the whole pass), B = the partners' records staged
//   in shared memory.  The accumulator fragment gives every lane two dyads (row g, partners 2q, 2q+1), whose Y entries
//   it reads from the cp.async ring (padded pitches 517/257 so that a quarter-warp's 16-byte reads hit distinct banks; the
//   float-Y ring keeps the same pitches in 8-byte units).
//   CTA = 8 warps = 16 rows x 32 time steps; warp w owns time steps t0+4w..+3 and both 8-row tiles.  ~0.36 issued
//   instructions per dyad instead of ~1.25.  R must be a multiple of 4.
// grid (ceil(T/32), ceil(nloc/16)), block 256; partial (grid.y*grid.x, 2).
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tame_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <int R, class YT = double>
struct TameMma {
    static constexpr int D = 2 + 2 * R, JC = 8, RS = TameRec<D>::RS, PIECES = D / 2, KS = R / 4;
    static constexpr int PR = 257, PJ = 517;                       // ring pitches in dyads (see header)
    static constexpr int MJ = 32 * RS + 4;                         // partner pitch of the staged records (doubles)
    static constexpr size_t Y_BYTES = (size_t)2 * JC * PJ * sizeof(typename TameY<YT>::V2);
    static constexpr size_t M_BYTES = (size_t)2 * JC * MJ * sizeof(double);
    static constexpr size_t SMEM = Y_BYTES + M_BYTES;
};

template <int R, bool SYM, class YT>
__global__ void __launch_bounds__(256, 1) k_llmse_mma(TameParams P, double* partial) {
    using TM = TameMma<R, YT>;
    using Y2 = typename TameY<YT>::V2;
    constexpr int D = TM::D, JC = TM::JC, RS = TM::RS, KS = TM::KS, PR = TM::PR, PJ = TM::PJ, MJ = TM::MJ, RT = 16;
    static_assert(R % 4 == 0, "DMMA k-step is 4");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Y2* Yr = reinterpret_cast<Y2*>(smem_raw);                                    // [2][JC*PJ]
    double* Mb = reinterpret_cast<double*>(smem_raw + TM::Y_BYTES);              // [2][JC*MJ]
    __shared__ double red[2][8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int t0 = blockIdx.x * 32;
    const int lrow0 = blockIdx.y * RT;
    const int gfirst = tame_grow(min(lrow0, P.nloc - 1), P.panel, P.world, P.rank);   // first node of the tile (16 | panel)

    // ---- copy role: this thread moves the dyads of rows lrow0 + 2*warp + {0,1} at time t0 + lane
    const YT* yrow[2];
    bool rvc[2];
    int gic[2];
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
        int l = lrow0 + 2 * warp + rr;
        rvc[rr] = (l < P.nloc) && (t0 + lane < P.T);
        l = min(l, P.nloc - 1);
        gic[rr] = tame_grow(l, P.panel, P.world, P.rank);
        yrow[rr] = TameY<YT>::ptr(P) + ((size_t)l * P.n * P.T + min(t0 + lane, P.T - 1)) * 2;
    }
    const size_t jstride = (size_t)P.T * 2;
    auto issue_chunk = [&](int buf, int jc) {
        Y2* yb = Yr + (size_t)buf * JC * PJ;
#pragma unroll
        for (int jj = 0; jj < JC; ++jj) {
            const int j = jc + jj;
#pragma unroll
            for (int rr = 0; rr < 2; ++rr) {
                const bool ok = rvc[rr] && (j < P.n) && (SYM ? (j > gic[rr]) : (j != gic[rr]));
                TameY<YT>::cp_async(yb + jj * PJ + rr * PR + tid, yrow[rr] + (size_t)min(j, P.n - 1) * jstride, ok);
            }
        }
        double* mb = Mb + (size_t)buf * JC * MJ;
        for (int e = tid; e < JC * 32 * TM::PIECES; e += 256) {
            const int piece = e % TM::PIECES, tl = (e / TM::PIECES) & 31, jj = e / (TM::PIECES * 32);
            const int j = jc + jj, tt = t0 + tl;
            const bool ok = (j < P.n) && (tt < P.T);
            const double* src = P.Xm + ((size_t)min(j, P.n - 1) * P.T + min(tt, P.T - 1)) * D + piece * 2;
            tame_cp_async16(mb + jj * MJ + tl * RS + piece * 2, src, ok);
        }
        tame_cp_async_commit();
    };

    // ---- tensor-core role: time steps t0 + 4*warp + tt, row tiles 0/1 (rows lrow0 + 8*tile + g)
    double aU[4][2][KS], aV[4][2][KS], oa[4][2], ob[4][2];
    int grow[2];
    bool rowok[2];
#pragma unroll
    for (int tile = 0; tile < 2; ++tile) {
        int l = lrow0 + 8 * tile + g;
        rowok[tile] = l < P.nloc;
        l = min(l, P.nloc - 1);
        grow[tile] = tame_grow(l, P.panel, P.world, P.rank);
#pragma unroll
        for (int tt = 0; tt < 4; ++tt) {
            const int t = min(t0 + 4 * warp + tt, P.T - 1);
            const double* m = P.Xm + ((size_t)grow[tile] * P.T + t) * D;
            oa[tt][tile] = m[0];
            ob[tt][tile] = m[1];
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                aU[tt][tile][ks] = m[2 + 4 * ks + q];          // A[row g][k q] = U_i[k]
                aV[tt][tile][ks] = m[2 + R + 4 * ks + q];      // A[row g][k q] = V_i[k]
            }
        }
    }
    double S00 = 0.0, S01 = 0.0, S11 = 0.0, SL = 0.0;

    const int jbeg = SYM ? (gfirst / JC) * JC : 0;
    const int nchunks = (P.n - jbeg + JC - 1) / JC;
    issue_chunk(0, jbeg);
    if (nchunks > 1) issue_chunk(1, jbeg + JC);
    for (int c = 0; c < nchunks; ++c) {
        const int jc = jbeg + c * JC, buf = c & 1;
        if (c + 1 < nchunks) tame_cp_async_wait<1>(); else tame_cp_async_wait<0>();
        __syncthreads();                                       // chunk c (Y dyads + partner records) is visible to the CTA
        const Y2* yb = Yr + (size_t)buf * JC * PJ;
        const double* mb = Mb + (size_t)buf * JC * MJ;
        // 0: all partners below the tile's rows, 1: all above (and inside the matrix), 2: mixed / tail
        const int kind = (jc + JC <= gfirst) ? 0 : ((jc > gfirst + RT - 1 && jc + JC <= P.n) ? 1 : 2);
        const int j0 = jc + 2 * q, j1 = j0 + 1;               // this lane's two partners
#pragma unroll
        for (int tt = 0; tt < 4; ++tt) {
            const int tl = 4 * warp + tt;
            const bool tok = (t0 + tl) < P.T;
            // B fragments: B[k q][partner g]
            double bV[KS], bU[KS];
            const double* recg = mb + g * MJ + tl * RS;
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                bU[ks] = recg[2 + 4 * ks + q];
                bV[ks] = recg[2 + R + 4 * ks + q];
            }
            const double2 ab0 = *reinterpret_cast<const double2*>(mb + (2 * q) * MJ + tl * RS);        // (a_j, b_j) of partner j0
            const double2 ab1 = *reinterpret_cast<const double2*>(mb + (2 * q + 1) * MJ + tl * RS);    // partner j1
#pragma unroll
            for (int tile = 0; tile < 2; ++tile) {
                double d00 = 0.0, d01 = 0.0, d10 = 0.0, d11 = 0.0;      // d0/d1 for partners j0, j1
#pragma unroll
                for (int ks = 0; ks < KS; ++ks) {
                    tame_dmma(d00, d01, aU[tt][tile][ks], bV[ks]);      // U_i . V_j
                    tame_dmma(d10, d11, aV[tt][tile][ks], bU[ks]);      // V_i . U_j
                }
                // the two dyads of this lane: row (8*tile + g) -> copied by warp (4*tile + g/2), rr = g & 1
                const int slot = (g & 1) * PR + (4 * tile + (g >> 1)) * 32 + tl;
                const double2 y0 = TameY<YT>::wide(yb[(2 * q) * PJ + slot]);
                const double2 y1 = TameY<YT>::wide(yb[(2 * q + 1) * PJ + slot]);
                const int gi = grow[tile];
                const double e00 = y0.x - ((oa[tt][tile] + ab0.y) + d00), e01 = y0.y - ((ab0.x + ob[tt][tile]) + d10);
                const double e10 = y1.x - ((oa[tt][tile] + ab1.y) + d01), e11 = y1.y - ((ab1.x + ob[tt][tile]) + d11);
                const bool base = rowok[tile] && tok;
                if (kind == 1) {
                    if (base) {
                        S00 = fma(e00, e00, S00); S01 = fma(e00, e01, S01); S11 = fma(e01, e01, S11);
                        S00 = fma(e10, e10, S00); S01 = fma(e10, e11, S01); S11 = fma(e11, e11, S11);
                    }
                } else if (kind == 0) {
                    if (base && !SYM) { SL = fma(e00, e00, SL); SL = fma(e01, e01, SL); SL = fma(e10, e10, SL); SL = fma(e11, e11, SL); }
                } else {
                    if (base && j0 < P.n && j0 != gi) {
                        if (j0 > gi) { S00 = fma(e00, e00, S00); S01 = fma(e00, e01, S01); S11 = fma(e01, e01, S11); }
                        else if (!SYM) { SL = fma(e00, e00, SL); SL = fma(e01, e01, SL); }
                    }
                    if (base && j1 < P.n && j1 != gi) {
                        if (j1 > gi) { S00 = fma(e10, e10, S00); S01 = fma(e10, e11, S01); S11 = fma(e11, e11, S11); }
                        else if (!SYM) { SL = fma(e10, e10, SL); SL = fma(e11, e11, SL); }
                    }
                }
            }
        }
        __syncthreads();                                       // every warp is done with buffer `buf`
        if (c + 2 < nchunks) issue_chunk(buf, jc + 2 * JC);
    }
    double sq = SYM ? 2.0 * (S00 + S11) : (S00 + S11) + SL;
    double quad = P.p0 * S00 + 2.0 * P.q * S01 + P.p1 * S11;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
        quad += __shfl_xor_sync(0xffffffffu, quad, o);
    }
    if (lane == 0) { red[0][warp] = sq; red[1][warp] = quad; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0, qd = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { s += red[0][w]; qd += red[1][w]; }
        size_t b = (size_t)blockIdx.y * gridDim.x + blockIdx.x;
        partial[b * 2 + 0] = s;
        partial[b * 2 + 1] = qd;
    }
}

// ------------------------------------------------------------------------------------------------------
// k_cellterms: per (i,t) block terms of the ELBO, one lane group (8, 16 or 32 lanes) per owned cell.
//   ent   = 0.5 (d (1+log 2pi) + logdet X_cov[i,t])                                    structured_mf.py:202-209
//   t==0 : lp0 = -0.5 (logdet S0 + mu' S0inv mu + tr(S0inv X_cov) + d log 2pi)         :152-173
//   t>0  : lpt = -0.5 (logdet Q + (mu_t - Phi mu_{t-1})' Qinv (..) + tr(Qinv X_cov) + d log 2pi)   :175-200
//   tr    = trace X_cov[i,t]   (for the "simplified" correction, :142-144)
// block 256 (8 warps); partial (gridDim.x, 4) = {lp0, lpt, ent, tr}.
// ------------------------------------------------------------------------------------------------------
template <int R>
struct TameCellSmem {
    static constexpr int D = 2 + 2 * R;
    static constexpr int DP = D <= 8 ? 8 : (D <= 16 ? 16 : 32);      // lanes per cell
    static constexpr int G = 32 / DP;                                  // cells per warp and pass
    double Cm[8][G * D * D];
    double rowb[8][G * 2 * D];
    double vec[8][G * 2 * D];
    double red[8][4];
    double cT[3][D * D];      // S0inv, Qinv, Phi transposed: cT[m][k * D + c] = M[c][k]
};
// A warp takes G = 32 / DP cells per pass (DP = 8, 16 or 32 lanes per cell, lane c of a group <-> column c): for the small
// blocks of r <= 3 that is 4 cells per pass instead of 1 with 26 idle lanes.
template <int R>
__device__ __forceinline__ void tame_cellterms_impl(const TameParams& P, double logdetS0, double logdetQ, double* partial,
                                                    TameCellSmem<R>& sh, int bid, int nb) {
    using CS = TameCellSmem<R>;
    constexpr int D = 2 + 2 * R, DD = D * D, DP = CS::DP, G = CS::G, NE = (G * DD + 31) / 32;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane / DP, c = lane % DP;
    for (int e = threadIdx.x; e < 3 * DD; e += blockDim.x) {
        const int m = e / DD, rc = e % DD;
        sh.cT[m][(rc % D) * D + rc / D] = P.cst[(m == 2 ? 5 : m) * DD + rc];
    }
    __syncthreads();
    const double LOG2PI = 1.8378770664093454835606594728112;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    const long ncell = (long)P.nloc * P.T;
    for (long cell0 = ((long)bid * 8 + warp) * G; cell0 < ncell; cell0 += (long)nb * 8 * G) {
#pragma unroll
        for (int m = 0; m < NE; ++m) {
            const int e = lane + 32 * m;
            if (e < G * DD) {
                const long ce = cell0 + e / DD;
                double v = 0.0;
                if (ce < ncell) {
                    const int le = (int)(ce / P.T), te = (int)(ce % P.T);
                    v = P.Xc[((size_t)tame_grow(le, P.panel, P.world, P.rank) * P.T + te) * DD + e % DD];
                }
                sh.Cm[warp][e] = v;
            }
        }
        const long cell = cell0 + g;
        const bool valid = cell < ncell, act = valid && c < D;
        const int l = valid ? (int)(cell / P.T) : 0, t = valid ? (int)(cell % P.T) : 0;
        const int i = tame_grow(l, P.panel, P.world, P.rank);
        double* vec = sh.vec[warp] + g * 2 * D;
        const double* Cg = sh.Cm[warp] + g * DD;
        if (act) {
            vec[c] = P.Xm[((size_t)i * P.T + t) * D + c];
            vec[D + c] = (t > 0) ? P.Xm[((size_t)i * P.T + t - 1) * D + c] : 0.0;
        }
        __syncwarp();
        const double* A = sh.cT[t == 0 ? 0 : 1];                 // S0inv or Qinv, A[k * D + c] = M[c][k]
        const double* Phi = sh.cT[2];
        double col[D];
        double tr = 0.0, trA = 0.0, resid = 0.0;
        if (act) {
#pragma unroll
            for (int k = 0; k < D; ++k) {
                col[k] = Cg[k * D + c];
                trA = fma(A[k * D + c], col[k], trA);       // sum_k A[c][k] * cov[k][c]
                tr = (k == c) ? col[k] : tr;
            }
            resid = vec[c];
            if (t > 0) {
                double pm = 0.0;
#pragma unroll
                for (int k = 0; k < D; ++k) pm = fma(Phi[k * D + c], vec[D + k], pm);
                resid -= pm;
            }
        } else {
#pragma unroll
            for (int k = 0; k < D; ++k) col[k] = 0.0;
        }
        __syncwarp();
        if (act) vec[c] = resid;
        __syncwarp();
        double quad = 0.0;
        if (act) {
            double a = 0.0;
#pragma unroll
            for (int k = 0; k < D; ++k) a = fma(A[k * D + c], vec[k], a);
            quad = resid * a;
        }
        const double logdet = tame_logdet_spd<D>(col, sh.rowb[warp] + g * 2 * D, c, act);
#pragma unroll
        for (int o = DP / 2; o > 0; o >>= 1) {
            tr += __shfl_xor_sync(0xffffffffu, tr, o);
            trA += __shfl_xor_sync(0xffffffffu, trA, o);
            quad += __shfl_xor_sync(0xffffffffu, quad, o);
        }
        if (valid && c == 0) {
            const double lp = -0.5 * ((t == 0 ? logdetS0 : logdetQ) + quad + trA + D * LOG2PI);
            if (t == 0) acc[0] += lp; else acc[1] += lp;
            acc[2] += 0.5 * (D * (1.0 + LOG2PI) + logdet);
            acc[3] += tr;
        }
        __syncwarp();
    }
    // the group leaders' sums -> lane 0 (the other lanes hold zeros)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int o = 16; o >= DP; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) sh.red[warp][k] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        double sum = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) sum += sh.red[w][threadIdx.x];
        partial[(size_t)bid * 4 + threadIdx.x] = sum;
    }
    __syncthreads();
}
template <int R>
__global__ void __launch_bounds__(256) k_cellterms(TameParams P, double logdetS0, double logdetQ, double* partial) {
    __shared__ TameCellSmem<R> sh;
    tame_cellterms_impl<R>(P, logdetS0, logdetQ, partial, sh, blockIdx.x, gridDim.x);
}

// ------------------------------------------------------------------------------------------------------
// k_fit: a WHOLE fit in one persistent cooperative launch (BASELINE config 5: many small independent fits) -- the loop of
// src/inference/base.py:166-203 on the device: per iteration  totals -> sweep (chain + streaming CTAs, exactly k_sweep) ->
// covariance blend -> ELBO / MSE partial sums -> reduction + the convergence test of base.py:183-203 by block 0, separated
// by grid-wide barriers; the traces stay in device memory until the host asks for them.  No host involvement per iteration.
// Meant for small n (the ELBO pass here is a plain one-warp-per-(row, time-slice) loop without the cp.async ring).
// ------------------------------------------------------------------------------------------------------
struct TameFitArgs {
    int max_iter;
    double tolerance, logdetS0, logdetQ, logdetR;
    double* elbo_trace;       // device, max_iter
    double* mse_trace;        // device, max_iter
    int* n_done;              // device
    double* part;             // device scratch: (grid, 6) partial sums {sq, quad, lp0, lpt, ent, tr}
    double* ctl;              // device: [0] previous ELBO, [1] patience, [2] stop flag
    unsigned int* bar;        // device: grid barrier counter (zero at launch)
};

__device__ __forceinline__ void tame_grid_sync(unsigned int* bar, unsigned int nblk, unsigned int& phase) {
    __syncthreads();
    if (threadIdx.x == 0) {
        ++phase;
        __threadfence();
        atomicAdd(bar, 1u);
        const unsigned int target = phase * nblk;
        while (*((volatile unsigned int*)bar) < target) { }
        __threadfence();
    }
    __syncthreads();
}

// moment totals of the current means, one CTA per time step (strided), fixed summation order: thread <-> (entry e, node
// part p), part p sums the nodes p, p + PARTS, ... and the parts are added in order (red: PARTS * TOT doubles of smem)
template <int R>
__device__ __forceinline__ void tame_totals_small(const TameParams& P, double* red, int bid, int nb) {
    constexpr int D = 2 + 2 * R, NV = 2 * R, TOT = TameTot<R>::TOT;
    constexpr int PARTS = (256 / TOT) > 0 ? (256 / TOT) : 1, EPT = (TOT + 255) / 256;     // r = 2: 12 parts of 20 entries
    for (int t = bid; t < P.T; t += nb) {
#pragma unroll
        for (int q = 0; q < EPT; ++q) {
            const int slot = threadIdx.x + 256 * q, e = slot % TOT, part = slot / TOT;
            if (part < PARTS) {
                int xa, xb = -1;
                if (e < NV) xa = tame_zidx<R>(e);
                else { const int f = e - NV; xa = tame_zidx<R>(f / NV); xb = tame_zidx<R>(f % NV); }
                double acc = 0.0;
                for (int j = part; j < P.n; j += PARTS) {
                    const double* m = P.Xm + ((size_t)j * P.T + t) * D;
                    const double va = __ldcg(m + xa);
                    acc += (xb < 0) ? va : va * __ldcg(m + xb);
                }
                if (PARTS == 1) P.tot[(size_t)t * TOT + e] = acc;
                else red[part * TOT + e] = acc;
            }
        }
        if (PARTS > 1) {
            __syncthreads();
            if (threadIdx.x < TOT) {
                double acc = 0.0;
#pragma unroll
                for (int p = 0; p < PARTS; ++p) acc += red[p * TOT + threadIdx.x];
                P.tot[(size_t)t * TOT + threadIdx.x] = acc;
            }
            __syncthreads();
        }
    }
}

// quadratic form of the expected log-likelihood (i<j) + squared reconstruction error (i != j): one warp per (row, W-step
// time slice), lane <-> (t, partner subgroup): W = 8, 16 or 32 time steps per slice, whichever pads T least, and the 32 / W
// lane groups take every (32/W)-th partner (a short T would otherwise leave most lanes idle).  Fixed summation order
// (structured_mf.py:124-146, temporal_ame.py:255-291); per-block sums -> part[bid][0..1]
template <int R, class YT>
__device__ __forceinline__ void tame_llmse_small(const TameParams& P, double* part, double* red /* 16 doubles smem */, int bid, int nb) {
    constexpr int D = 2 + 2 * R;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int W = 32;
    if (((P.T + 15) / 16) * 16 < ((P.T + W - 1) / W) * W) W = 16;
    if (((P.T + 7) / 8) * 8 < ((P.T + W - 1) / W) * W) W = 8;
    const int G = 32 / W, tl = lane & (W - 1), js = lane / W;
    const int nslices = (P.T + W - 1) / W;
    const long nitems = (long)P.n * nslices;
    double sq = 0.0, quad = 0.0;
    for (long item = (long)bid * 8 + warp; item < nitems; item += (long)nb * 8) {
        const int i = (int)(item / nslices), t = (int)(item - (long)i * nslices) * W + tl;
        if (t < P.T) {
            const double* mi = P.Xm + ((size_t)i * P.T + t) * D;
            double ai = mi[0], bi = mi[1], Ui[R], Vi[R];
#pragma unroll
            for (int a = 0; a < R; ++a) { Ui[a] = mi[2 + a]; Vi[a] = mi[2 + R + a]; }
            const YT* yrow = TameY<YT>::ptr(P) + ((size_t)i * P.n * P.T + t) * 2;
            double s = 0.0, q = 0.0;
            // partners four at a time: the loads of a group are issued before the first use (L2 latency, no ring here)
            for (int j0 = js; j0 < P.n; j0 += 4 * G) {
                double2 y[4];
                double rec[4][D];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = min(j0 + u * G, P.n - 1);
                    y[u] = TameY<YT>::wide(TameY<YT>::ld_stream(yrow + (size_t)j * P.T * 2));
                    const double* mj = P.Xm + ((size_t)j * P.T + t) * D;
#pragma unroll
                    for (int k = 0; k < D; ++k) rec[u][k] = __ldcg(mj + k);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = j0 + u * G;
                    if (j < P.n && j != i) {
                        double d0 = ai + rec[u][1], d1 = rec[u][0] + bi;
#pragma unroll
                        for (int a = 0; a < R; ++a) { d0 = fma(Ui[a], rec[u][2 + R + a], d0); d1 = fma(rec[u][2 + a], Vi[a], d1); }
                        const double e0 = y[u].x - d0, e1 = y[u].y - d1;
                        s = fma(e0, e0, fma(e1, e1, s));
                        if (j > i) q += P.p0 * e0 * e0 + 2.0 * P.q * e0 * e1 + P.p1 * e1 * e1;
                    }
                }
            }
            sq += s;
            quad += q;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
        quad += __shfl_xor_sync(0xffffffffu, quad, o);
    }
    if (lane == 0) { red[warp] = sq; red[8 + warp] = quad; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { a += red[w]; b += red[8 + w]; }
        part[(size_t)bid * 6 + 0] = a;
        part[(size_t)bid * 6 + 1] = b;
    }
    __syncthreads();
}

template <int R, int RW, int NH, class YT>
__global__ void __launch_bounds__(256, 1) k_fit(TameParams P0, TameFitArgs F) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int D = 2 + 2 * R;
    const unsigned int nblk = gridDim.x;
    const int bid = blockIdx.x, tid = threadIdx.x;
    unsigned int phase = 0;
    double* part4 = F.part + (size_t)nblk * 6;            // cell terms go through a (grid, 4) block of their own
    for (int it = 0; it < F.max_iter; ++it) {
        TameParams P = P0;
        P.epoch = P0.epoch + it + 1;                       // stamps of this sweep (hand-over tags, unit_done)
        // ---- running totals of the partner moments from the current means; reset of the sweep's counters
        tame_totals_small<R>(P, reinterpret_cast<double*>(smem_raw), bid, (int)nblk);
        if (bid == 0) {
            for (int t = tid; t < P.T; t += blockDim.x) P.progress[t] = 0;
            if (tid == 0) *P.unit_counter = 0;
        }
        tame_grid_sync(F.bar, nblk, phase);
        // ---- the sweep: chain CTAs + streaming CTAs, exactly as in k_sweep
        tame_sweep_body<R, RW, NH, YT>(P, smem_raw);
        tame_grid_sync(F.bar, nblk, phase);
        // ---- factorisation rule + damped write of the covariance blocks
        tame_covblend_impl<R>(P, reinterpret_cast<double*>(smem_raw), bid, (int)nblk);
        tame_grid_sync(F.bar, nblk, phase);
        // ---- ELBO / MSE partial sums
        tame_cellterms_impl<R>(P, F.logdetS0, F.logdetQ, part4, *reinterpret_cast<TameCellSmem<R>*>(smem_raw), bid, (int)nblk);
        tame_llmse_small<R, YT>(P, F.part, reinterpret_cast<double*>(smem_raw), bid, (int)nblk);
        tame_grid_sync(F.bar, nblk, phase);
        // ---- block 0: deterministic reduction, ELBO (k_finalize's formulas), the stop rule of base.py:183-203
        if (bid == 0) {
            double* red6 = reinterpret_cast<double*>(smem_raw);
            if (tid < 6) {
                double a = 0.0;
                for (unsigned int b = 0; b < nblk; ++b) a += (tid < 2) ? F.part[(size_t)b * 6 + tid] : part4[(size_t)b * 4 + (tid - 2)];
                red6[tid] = a;
            }
            __syncthreads();
            if (tid == 0) {
                const double LOG2PI = 1.8378770664093454835606594728112;
                const double n = (double)P.n, npairs = 0.5 * n * (n - 1.0);
                double ll = red6[1] + npairs * (double)P.T * (F.logdetR + 2.0 * LOG2PI);
                if (P.mode != 0) ll += 0.1 * (P.p0 + P.p1) / (double)D * (n - 1.0) * red6[5];
                ll *= -0.5;
                const double elbo = ((ll + red6[2]) + red6[3]) + red6[4];
                const double mse = red6[0] / (n * (n - 1.0) * (double)P.T);
                F.elbo_trace[it] = elbo;
                F.mse_trace[it] = mse;
                *F.n_done = it + 1;
                bool converged = false;
                if (it > 0) {
                    const double prev = F.ctl[0];
                    const double rel = fabs(elbo - prev) / (fabs(prev) + 1e-8);
                    const double pat = (rel < F.tolerance) ? F.ctl[1] + 1.0 : 0.0;
                    F.ctl[1] = pat;
                    converged = pat >= 3.0;
                }
                F.ctl[0] = elbo;
                if (converged || *((volatile int*)P.abort_flag)) F.ctl[2] = 1.0;
            }
        }
        tame_grid_sync(F.bar, nblk, phase);
        if (*((volatile double*)&F.ctl[2]) != 0.0) break;
    }
}

// launchers of the kernels that read Y, for one element type of Y (each queries its own instantiation: the shared-memory
// footprint depends on the type)
struct TameYOps {
    void (*contract)(const TameParams&, int k0, int k1, int j0, int j1, int tri, int accumulate, cudaStream_t);
    cudaError_t (*chain)(const TameParams&, int i0, int i1, cudaStream_t);
    cudaError_t (*sweep_fused)(const TameParams&, cudaStream_t);
    cudaError_t (*fit_device)(const TameParams&, const TameFitArgs&, int* grid_out, cudaStream_t);
    int (*fit_grid)(const TameParams&);
    int (*sweep_capacity)(int nh);
    void (*llmse)(const TameParams&, double* partial, int* nblocks, int symmetric, cudaStream_t);
};

// function table of one latent dimension
struct TameOps {
    int r;
    size_t chain_smem;
    int tot;
    void (*totals)(const TameParams&, double* partial, int NS, cudaStream_t);
    void (*covblend)(const TameParams&, cudaStream_t);
    int (*chain_max_T)();
    void (*cellterms)(const TameParams&, double logdetS0, double logdetQ, double* partial, int nblocks, cudaStream_t);
    int (*llmse_blocks)(const TameParams&);
    int (*cellterms_blocks)(const TameParams&);
    TameYOps f64, f32;         // Y stored as double / as float
};
const TameOps* tame_get_ops(int r);
void tame_count_launch(int n);
