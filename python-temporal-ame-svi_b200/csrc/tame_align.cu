// tame_align.cu -- the step after the fit in every driver of the reference: src/utils/alignment.py
// (align_temporal_states :224-313, compute_alignment_error :316-385, procrustes_alignment :31-103, align_signs :106-166).
// The reference runs O(n T) Python iterations (three per-row sign loops per time step); here the whole step is four
// small launches over the state arrays, which never leave HBM:
//   k_align_cross   M[t][b] = X_true[:,t,blk]' X_est[:,t,blk]      per time step and block (U, V), split over rows;
//                   FP64 tensor cores (DMMA m8n8k4), the node index is the inner dimension
//   k_align_reduce  fixed-order sum of the row splits
//   k_align_rot     R = U Vt of svd(M) (the orthogonal polar factor), last singular direction negated if det < 0,
//                   by one-sided Jacobi with parallel round-robin pair ordering -- one warp per k x k matrix, k <= 16
//   k_align_apply   rotate the U / V rows, per-row sign flips of the (a,b), U and V parts, squared error
//   k_align_sum     fixed-order reduction of the partial sums
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cmath>
#include <cstdint>

#include "../../include/tame_b200.h"

void tame_count_launch(int n);
int tame_set_error(int code, const char* fmt, ...);

#define ACK(call)                                                                                           \
    do {                                                                                                    \
        cudaError_t e_ = (call);                                                                            \
        if (e_ != cudaSuccess)                                                                              \
            return tame_set_error(TAME_ECUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
    } while (0)

namespace {
constexpr int KMAX = 16;     // largest rotation: the 2r-dimensional block of the global mode, r <= 8

// X is (n, T, d) row-major.  Block b of time step t covers the columns off + b*k .. off + (b+1)*k - 1.
// The cross-covariance X_true' X_est is a GEMM with the node index as the inner dimension, so it runs on the FP64
// tensor cores: mma.sync.m8n8k4 with A = X_true' (8 columns x 4 nodes), B = X_est (4 nodes x 8 columns), C an 8 x 8 tile
// of M.  grid (T, NS), 4 warps: a warp owns one (block, 8x8 tile) unit and every nsub-th group of four nodes of the
// block's row split, with four independent accumulator pairs; the warps' tiles are combined in fixed order.
// partial[((t*NS + s) * nblk + b) * k*k + a*k + c].
__device__ __forceinline__ void align_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(128) k_align_cross(const double* __restrict__ est, const double* __restrict__ tru, int n, int T,
                                                     int d, int off, int k, int nblk, double* __restrict__ partial) {
    __shared__ double ctile[4][64];
    const int t = blockIdx.x, s = blockIdx.y, NS = gridDim.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int TA = (k + 7) / 8, tiles = TA * TA, units = nblk * tiles, nsub = 4 / units;     // units in {1, 2, 4}
    const int unit = warp % units, sub = warp / units;
    const int b = unit / tiles, ta = (unit % tiles) / TA, tc = (unit % tiles) % TA;
    const int i0 = (int)((long)n * s / NS), i1 = (int)((long)n * (s + 1) / NS);
    const int kq = lane & 3, c8 = lane >> 2;
    const bool va = ta * 8 + c8 < k, vc = tc * 8 + c8 < k;
    const size_t stride = (size_t)T * d;
    const double* pt = tru + (size_t)t * d + off + b * k + ta * 8 + c8;
    const double* pe = est + (size_t)t * d + off + b * k + tc * 8 + c8;
    double acc[4][2];
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u][0] = acc[u][1] = 0.0;
    const int ngroups = (i1 - i0 + 3) / 4;
    for (int g = sub; g < ngroups; g += 4 * nsub) {
        double x[4], y[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + 4 * (g + u * nsub) + kq;
            const bool in = (g + u * nsub < ngroups) && i < i1;
            x[u] = (in && va) ? pt[(size_t)i * stride] : 0.0;
            y[u] = (in && vc) ? pe[(size_t)i * stride] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) align_dmma(acc[u][0], acc[u][1], x[u], y[u]);
    }
    const double c0 = (acc[0][0] + acc[1][0]) + (acc[2][0] + acc[3][0]);
    const double c1 = (acc[0][1] + acc[1][1]) + (acc[2][1] + acc[3][1]);
    ctile[warp][c8 * 8 + kq * 2] = c0;              // C fragment: row = lane >> 2, columns 2*(lane & 3), +1
    ctile[warp][c8 * 8 + kq * 2 + 1] = c1;
    __syncthreads();
    for (int e = threadIdx.x; e < units * 64; e += blockDim.x) {
        const int un = e / 64, el = e % 64;
        double v = 0.0;
        for (int sb = 0; sb < nsub; ++sb) v += ctile[un + units * sb][el];
        const int bb = un / tiles, a = ((un % tiles) / TA) * 8 + el / 8, c = ((un % tiles) % TA) * 8 + el % 8;
        if (a < k && c < k) partial[((size_t)(t * NS + s) * nblk + bb) * k * k + a * k + c] = v;
    }
}

// M[mat][el] = sum over the NS row splits, fixed order; mat = t*nblk + b
__global__ void k_align_reduce(const double* __restrict__ partial, int nmat, int nblk, int NS, int kk, double* __restrict__ M) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nmat * kk) return;
    const int mat = e / kk, el = e % kk, t = mat / nblk, b = mat % nblk;
    double v = 0.0;
    for (int s = 0; s < NS; ++s) v += partial[((size_t)(t * NS + s) * nblk + b) * kk + el];
    M[e] = v;
}

// One WARP per k x k matrix (k <= 16), four matrices per block.  One-sided Jacobi: column pairs of A (= M at the start)
// are rotated until mutually orthogonal, the rotations accumulated in V: A = U diag(sigma), M = U diag(sigma) V'.
// Disjoint pairs of one round-robin step are rotated at the same time: a group of RP lanes (one per matrix row) owns a
// pair, forms the three dot products by shuffles and updates its rows of A and V in shared memory.
// R = U V' is what alignment.py:82-85 forms from torch.linalg.svd; if det(R) < 0 the reference negates the last row of
// Vt, i.e. the direction of the SMALLEST singular value (alignment.py:88-90): R -= 2 u_min v_min'.
__global__ void __launch_bounds__(128) k_align_rot(const double* __restrict__ Mall, int nmat, int k, double* __restrict__ rot) {
    __shared__ double sA[4][KMAX * KMAX], sV[4][KMAX * KMAX], sR[4][KMAX * KMAX], sL[4][KMAX * KMAX];
    __shared__ double sSig[4][KMAX];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int m = blockIdx.x * 4 + warp;
    if (m >= nmat) return;
    double* A = sA[warp];
    double* V = sV[warp];
    double* Rm = sR[warp];
    double* L = sL[warp];
    double* sig = sSig[warp];
    const int kk = k * k;
    for (int e = lane; e < kk; e += 32) {
        A[e] = Mall[(size_t)m * kk + e];
        V[e] = (e / k == e % k) ? 1.0 : 0.0;
    }
    __syncwarp();
    const int RP = (k <= 8) ? 8 : 16, PP = 32 / RP;           // lanes per pair, pairs in flight
    const int players = k + (k & 1), npairs = players / 2, nsteps = players - 1;
    const int grp = lane / RP, a = lane % RP;
    for (int sweep = 0; sweep < 40 && k > 1; ++sweep) {
        bool any = false;
        for (int step = 0; step < nsteps; ++step) {
            for (int g0 = 0; g0 < npairs; g0 += PP) {
                const int pi = g0 + grp;
                int p = 0, q = 0;
                if (pi == 0) { p = players - 1; q = step; }
                else { p = (step + pi) % (players - 1); q = (step - pi + (players - 1)) % (players - 1); }
                if (p > q) { const int tmp = p; p = q; q = tmp; }
                const bool valid = pi < npairs && q < k;                 // q == k is the bye of an odd k
                const bool row = valid && a < k;
                const double ap = row ? A[a * k + p] : 0.0, aq = row ? A[a * k + q] : 0.0;
                const double vp = row ? V[a * k + p] : 0.0, vq = row ? V[a * k + q] : 0.0;
                double alpha = ap * ap, beta = aq * aq, gamma = ap * aq;
                for (int o = RP / 2; o > 0; o >>= 1) {
                    alpha += __shfl_xor_sync(0xffffffffu, alpha, o);
                    beta += __shfl_xor_sync(0xffffffffu, beta, o);
                    gamma += __shfl_xor_sync(0xffffffffu, gamma, o);
                }
                const bool rotate = valid && gamma != 0.0 && fabs(gamma) > 1e-15 * sqrt(alpha * beta);
                if (rotate && row) {
                    const double zeta = (beta - alpha) / (2.0 * gamma);
                    const double tt = copysign(1.0, zeta) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
                    const double cs = 1.0 / sqrt(1.0 + tt * tt), sn = cs * tt;
                    A[a * k + p] = cs * ap - sn * aq;
                    A[a * k + q] = sn * ap + cs * aq;
                    V[a * k + p] = cs * vp - sn * vq;
                    V[a * k + q] = sn * vp + cs * vq;
                }
                any |= __any_sync(0xffffffffu, rotate);
                __syncwarp();
            }
        }
        if (!any) break;
    }
    // singular values; left vectors = normalised columns
    double sj = 0.0;
    if (lane < k) {
        double s2 = 0.0;
        for (int r2 = 0; r2 < k; ++r2) s2 = fma(A[r2 * k + lane], A[r2 * k + lane], s2);
        sj = sqrt(s2);
    }
    double smax = sj;
    for (int o = 16; o > 0; o >>= 1) smax = fmax(smax, __shfl_xor_sync(0xffffffffu, smax, o));
    if (lane < k) {
        const bool ok = sj > 1e-14 * smax && sj > 0.0;
        const double inv = ok ? 1.0 / sj : 0.0;
        for (int r2 = 0; r2 < k; ++r2) A[r2 * k + lane] *= inv;           // rank-deficient columns become zero
        sig[lane] = ok ? sj : -1.0;
    }
    __syncwarp();
    if (lane == 0) {
        // rank-deficient cross-covariance (e.g. an all-zero estimate): complete U to an orthonormal basis.  The
        // reference's result is LAPACK-specific there; this keeps R orthogonal and finite.
        for (int j = 0; j < k; ++j) {
            if (sig[j] >= 0.0) continue;
            for (int cand = 0; cand < k; ++cand) {
                double w[KMAX];
                for (int r2 = 0; r2 < k; ++r2) w[r2] = (r2 == cand) ? 1.0 : 0.0;
                for (int pass = 0; pass < 2; ++pass)
                    for (int j2 = 0; j2 < k; ++j2) {
                        if (j2 == j || (sig[j2] < 0.0 && j2 > j)) continue;
                        double dot = 0.0;
                        for (int r2 = 0; r2 < k; ++r2) dot = fma(w[r2], A[r2 * k + j2], dot);
                        for (int r2 = 0; r2 < k; ++r2) w[r2] = fma(-dot, A[r2 * k + j2], w[r2]);
                    }
                double nw = 0.0;
                for (int r2 = 0; r2 < k; ++r2) nw = fma(w[r2], w[r2], nw);
                if (nw > 0.5 / k) {
                    const double inv = 1.0 / sqrt(nw);
                    for (int r2 = 0; r2 < k; ++r2) A[r2 * k + j] = w[r2] * inv;
                    sig[j] = 0.0;
                    break;
                }
            }
        }
    }
    __syncwarp();
    // R0 = U V'
    for (int e = lane; e < kk; e += 32) {
        const int r2 = e / k, c = e % k;
        double v = 0.0;
        for (int j = 0; j < k; ++j) v = fma(A[r2 * k + j], V[c * k + j], v);
        Rm[e] = v;
        L[e] = v;
    }
    __syncwarp();
    // sign of det(R0) by elimination with partial pivoting (one lane; k <= 16), smallest singular direction
    int flip = 0, jmin = 0;
    if (lane == 0) {
        double det = 1.0;
        for (int p = 0; p < k; ++p) {
            int piv = p;
            for (int r2 = p + 1; r2 < k; ++r2)
                if (fabs(L[r2 * k + p]) > fabs(L[piv * k + p])) piv = r2;
            if (piv != p) {
                for (int c = 0; c < k; ++c) { const double tmp = L[p * k + c]; L[p * k + c] = L[piv * k + c]; L[piv * k + c] = tmp; }
                det = -det;
            }
            det *= L[p * k + p];
            if (L[p * k + p] == 0.0) break;
            const double inv = 1.0 / L[p * k + p];
            for (int r2 = p + 1; r2 < k; ++r2) {
                const double f = L[r2 * k + p] * inv;
                for (int c = p + 1; c < k; ++c) L[r2 * k + c] = fma(-f, L[p * k + c], L[r2 * k + c]);
            }
        }
        flip = det < 0.0 ? 1 : 0;
        for (int j = 1; j < k; ++j)
            if (sig[j] < sig[jmin]) jmin = j;
    }
    flip = __shfl_sync(0xffffffffu, flip, 0);
    jmin = __shfl_sync(0xffffffffu, jmin, 0);
    double* out = rot + (size_t)m * kk;
    for (int e = lane; e < kk; e += 32) {
        const int r2 = e / k, c = e % k;
        out[e] = flip ? fma(-2.0 * A[r2 * k + jmin], V[c * k + jmin], Rm[e]) : Rm[e];
    }
}

// temporal mean of every (node, component): alignment.py:287-288
__global__ void k_align_tmean(const double* __restrict__ X, int n, int T, int d, double* __restrict__ out) {
    const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long)n * d) return;
    const int i = (int)(e / d), c = (int)(e % d);
    double s = 0.0;
    for (int t = 0; t < T; ++t) s += X[((size_t)i * T + t) * d + c];
    out[e] = s / T;
}

// Rotation + signs + squared error.  grid (ceil(T/32), NI), 128 threads: lane = time step inside the 32-step slice,
// every warp walks over nodes.  The 32 rows (i, t0..t0+31) of a warp are one contiguous 32*D-double chunk: it is copied
// to shared memory with coalesced loads (row pitch D+1, conflict-free per lane), processed one row per lane, and the
// aligned rows go back the same way.
// EACH: rot is (T, 2, R, R): U rows times rot[t][0], V rows times rot[t][1], one sign per part (alignment.py:204-214);
//       staged as Rs[element][lane] so that lanes (different t) read different banks.
// !EACH (global mode): rot is (2R, 2R), the whole multiplicative row is rotated and gets one sign (alignment.py:296-311).
// partial[blockIdx.y * gridDim.x + blockIdx.x] = the block's sum of ||aligned - true||^2.
// dynamic shared memory: AlignSmem<R, EACH>::BYTES
template <int R, bool EACH>
struct AlignSmem {
    static constexpr int D = 2 + 2 * R, DP = D + 1, K = EACH ? R : 2 * R, NE = (EACH ? 2 : 1) * K * K;
    static constexpr int ROT = EACH ? NE * 32 : NE;                 // doubles
    static constexpr size_t BYTES = sizeof(double) * (ROT + 4 * 2 * 32 * DP);
};

template <int R, bool EACH>
__global__ void __launch_bounds__(128) k_align_apply(const double* __restrict__ est, const double* __restrict__ tru, int n, int T,
                                                     const double* __restrict__ rot, double* __restrict__ out,
                                                     double* __restrict__ partial) {
    using SM = AlignSmem<R, EACH>;
    constexpr int D = SM::D, DP = SM::DP, K = SM::K, NB = EACH ? 2 : 1, NE = SM::NE;
    extern __shared__ double align_smem[];
    __shared__ double red[4];
    double* Rs = align_smem;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* se = align_smem + SM::ROT + warp * 2 * 32 * DP;          // this warp's 32 estimate rows (aligned in place)
    double* sy = se + 32 * DP;                                      // ... and the 32 target rows
    const int t0 = blockIdx.x * 32, nt = min(32, T - t0);
    if (EACH) {
        for (int e = threadIdx.x; e < NE * 32; e += blockDim.x) {
            const int tl = e / NE, el = e % NE;                      // coalesced read of rot[t0 + tl][el]
            Rs[el * 32 + tl] = (tl < nt) ? rot[(size_t)(t0 + tl) * NE + el] : 0.0;
        }
    } else {
        for (int e = threadIdx.x; e < NE; e += blockDim.x) Rs[e] = rot[e];
    }
    __syncthreads();
    const int per = (n + gridDim.y - 1) / gridDim.y;
    const int ibeg = blockIdx.y * per, iend = min(n, ibeg + per);
    double sse = 0.0;
    double* x = se + lane * DP;
    const double* y = sy + lane * DP;
    for (int i = ibeg + warp; i < iend; i += 4) {
        const size_t base = ((size_t)i * T + t0) * D;
        {   // all 2*D loads of the lane are issued before the first shared-memory store (one DRAM round trip, not D)
            double ve[D], vy[D];
#pragma unroll
            for (int it = 0; it < D; ++it) {
                const int e = lane + 32 * it;
                const bool in = e < nt * D;
                ve[it] = in ? est[base + e] : 0.0;
                vy[it] = in ? tru[base + e] : 0.0;
            }
#pragma unroll
            for (int it = 0; it < D; ++it) {
                const int e = lane + 32 * it;
                if (e < nt * D) {
                    const int row = e / D, c = e - row * D;
                    se[row * DP + c] = ve[it];
                    sy[row * DP + c] = vy[it];
                }
            }
        }
        __syncwarp();
        if (lane < nt) {
            {   // additive pair: sign only (alignment.py:266-268)
                const double x0 = x[0], x1 = x[1], y0 = y[0], y1 = y[1];
                const double p0 = x0 - y0, p1 = x1 - y1, n0 = -x0 - y0, n1 = -x1 - y1;
                const double sg = (sqrt(fma(n1, n1, n0 * n0)) < sqrt(fma(p1, p1, p0 * p0))) ? -1.0 : 1.0;
                const double v0 = sg * x0, v1 = sg * x1;
                x[0] = v0;
                x[1] = v1;
                sse = fma(v0 - y0, v0 - y0, sse);
                sse = fma(v1 - y1, v1 - y1, sse);
            }
#pragma unroll 1
            for (int b = 0; b < NB; ++b) {
                double xv[K];
#pragma unroll
                for (int c = 0; c < K; ++c) xv[c] = x[2 + b * K + c];
                const double* Rb = Rs + (EACH ? (size_t)b * K * K * 32 + lane : 0);
                const double* yb = y + 2 + b * K;
                // two rolled passes over the output columns (decide the sign, then write); the rotated value is recomputed
                // by the same instruction sequence instead of kept -- K more registers would not fit for K = 16
                double pos = 0.0, neg = 0.0;
#pragma unroll 1
                for (int c = 0; c < K; ++c) {
                    double v = 0.0;
#pragma unroll
                    for (int a = 0; a < K; ++a) v = fma(xv[a], EACH ? Rb[(a * K + c) * 32] : Rb[a * K + c], v);   // X_est @ R  (alignment.py:92)
                    const double dp = v - yb[c], dn = -v - yb[c];
                    pos = fma(dp, dp, pos);
                    neg = fma(dn, dn, neg);
                }
                const double sg = (sqrt(neg) < sqrt(pos)) ? -1.0 : 1.0;       // alignment.py:141-146
#pragma unroll 1
                for (int c = 0; c < K; ++c) {
                    double v = 0.0;
#pragma unroll
                    for (int a = 0; a < K; ++a) v = fma(xv[a], EACH ? Rb[(a * K + c) * 32] : Rb[a * K + c], v);
                    v *= sg;
                    x[2 + b * K + c] = v;
                    sse = fma(v - yb[c], v - yb[c], sse);
                }
            }
        }
        __syncwarp();
#pragma unroll
        for (int it = 0; it < D; ++it) {
            const int e = lane + 32 * it;
            if (e < nt * D) {
                const int row = e / D, c = e - row * D;
                out[base + e] = se[row * DP + c];
            }
        }
        __syncwarp();
    }
    for (int o = 16; o > 0; o >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, o);
    if (lane == 0) red[warp] = sse;
    __syncthreads();
    if (threadIdx.x == 0) partial[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = (red[0] + red[1]) + (red[2] + red[3]);
}

template <int R, bool EACH>
cudaError_t launch_apply_t(dim3 grid, cudaStream_t st, const double* est, const double* tru, int n, int T, const double* rot,
                           double* out, double* partial) {
    constexpr size_t smem = AlignSmem<R, EACH>::BYTES;
    {   // per-device attribute, set on every call (cheap next to the launch; no per-process flag to go stale on a second GPU)
        cudaError_t e = cudaFuncSetAttribute(k_align_apply<R, EACH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    k_align_apply<R, EACH><<<grid, 128, smem, st>>>(est, tru, n, T, rot, out, partial);
    return cudaSuccess;
}

template <int R>
cudaError_t launch_apply(int each, dim3 grid, cudaStream_t st, const double* est, const double* tru, int n, int T,
                         const double* rot, double* out, double* partial) {
    return each ? launch_apply_t<R, true>(grid, st, est, tru, n, T, rot, out, partial)
                : launch_apply_t<R, false>(grid, st, est, tru, n, T, rot, out, partial);
}

__global__ void k_align_sum(const double* __restrict__ partial, long nb, int nq, double scale, double* __restrict__ out) {
    // nq interleaved quantities; one block of 256 threads, fixed order
    __shared__ double red[256];
    for (int q = 0; q < nq; ++q) {
        double s = 0.0;
        for (long b = threadIdx.x; b < nb; b += 256) s += partial[b * nq + q];
        red[threadIdx.x] = s;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
            __syncthreads();
        }
        if (threadIdx.x == 0) out[q] = red[0] * scale;
        __syncthreads();
    }
}

// rows x width: flip a row when the flipped row is strictly closer (alignment.py:138-146); optional squared error
__global__ void k_align_signs(const double* __restrict__ est, const double* __restrict__ tru, long rows, int width,
                              double* __restrict__ out, double* __restrict__ partial) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    double sse = 0.0;
    if (i < rows) {
        const double* x = est + (size_t)i * width;
        const double* y = tru + (size_t)i * width;
        double pos = 0.0, neg = 0.0;
        for (int a = 0; a < width; ++a) {
            const double dp = x[a] - y[a], dn = -x[a] - y[a];
            pos = fma(dp, dp, pos);
            neg = fma(dn, dn, neg);
        }
        const double sg = (sqrt(neg) < sqrt(pos)) ? -1.0 : 1.0;
        for (int a = 0; a < width; ++a) {
            const double v = sg * x[a];
            out[(size_t)i * width + a] = v;
            sse = fma(v - y[a], v - y[a], sse);
        }
    }
    if (partial) {
        __shared__ double red[8];
        for (int o = 16; o > 0; o >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sse;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
            partial[blockIdx.x] = s;
        }
    }
}

// X_est @ R for an (n, k) matrix, with the two traces of the optional scaling (alignment.py:95-101):
// partial[2*block] = sum X_true . Xa, partial[2*block+1] = sum Xa . Xa
__global__ void __launch_bounds__(128) k_align_rotate(const double* __restrict__ est, const double* __restrict__ tru, int n, int k,
                                                      const double* __restrict__ rot, double* __restrict__ out,
                                                      double* __restrict__ partial) {
    __shared__ double Rs[KMAX * KMAX];
    __shared__ double red[2][4];
    for (int e = threadIdx.x; e < k * k; e += blockDim.x) Rs[e] = rot[e];
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double num = 0.0, den = 0.0;
    if (i < n) {
        double x[KMAX];
        for (int a = 0; a < k; ++a) x[a] = est[(size_t)i * k + a];
        for (int c = 0; c < k; ++c) {
            double v = 0.0;
            for (int a = 0; a < k; ++a) v = fma(x[a], Rs[a * k + c], v);
            out[(size_t)i * k + c] = v;
            num = fma(tru[(size_t)i * k + c], v, num);
            den = fma(v, v, den);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        num += __shfl_xor_sync(0xffffffffu, num, o);
        den += __shfl_xor_sync(0xffffffffu, den, o);
    }
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = num; red[1][threadIdx.x >> 5] = den; }
    __syncthreads();
    if (threadIdx.x == 0) {
        partial[2 * blockIdx.x] = (red[0][0] + red[0][1]) + (red[0][2] + red[0][3]);
        partial[2 * blockIdx.x + 1] = (red[1][0] + red[1][1]) + (red[1][2] + red[1][3]);
    }
}

__global__ void k_align_scale(double* __restrict__ X, long count, const double* __restrict__ numden) {
    const double den = numden[1];
    if (!(den > 1e-10)) return;                        // alignment.py:99
    const double s = numden[0] / den;
    const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < count) X[e] *= s;
}

// ---- contribution / U'V-product diagnostics (src/utils/diagnostics.py:82-217,528-561) -----------------------------------
// The reference forms the n x n matrices a_i + b_j and U_i.V_j per time step.  Their sums of squares and products follow
// from r x r Gram matrices (the same DMMA kernel as the alignment) and a few per-time-step row sums:
//   sum_ij (a_i + b_j)^2   = n sum a^2 + n sum b^2 + 2 (sum a)(sum b)          diagonal: sum_i (a_i + b_i)^2
//   sum_ij (U_i.V_j)^2     = <U'U, V'V>                                        diagonal: sum_i (U_i.V_i)^2
//   sum_ij (U_i.V_j)       = (sum_i U_i).(sum_j V_j)
//   sum_ij (Ut_i.Vt_j)(Ue_i.Ve_j) = <Ut'Ue, Vt'Ve>
constexpr int DQ = 6;      // scalar row sums: sum a, sum b, sum a^2, sum b^2, sum (a+b)^2, sum (U.V)^2; then sum U (r), sum V (r)

// grid (ceil(T/32), NI), 128 threads: lane = time step, the four warps walk over nodes; every lane keeps the sums of its
// own time step, so there is no cross-lane reduction.  partial[((blockIdx.y*4 + warp) * T + t) * (DQ + 2R) + q]
template <int R>
__global__ void __launch_bounds__(128) k_diag_rows(const double* __restrict__ X, int n, int T, double* __restrict__ partial) {
    constexpr int D = 2 + 2 * R, NQ = DQ + 2 * R;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = blockIdx.x * 32 + lane;
    if (t >= T) return;
    const int per = (n + gridDim.y - 1) / gridDim.y;
    const int ibeg = blockIdx.y * per, iend = min(n, ibeg + per);
    double q[NQ];
#pragma unroll
    for (int k = 0; k < NQ; ++k) q[k] = 0.0;
    for (int i = ibeg + warp; i < iend; i += 4) {
        const double* x = X + ((size_t)i * T + t) * D;
        const double a = x[0], b = x[1];
        q[0] += a;
        q[1] += b;
        q[2] = fma(a, a, q[2]);
        q[3] = fma(b, b, q[3]);
        q[4] = fma(a + b, a + b, q[4]);
        double uv = 0.0;
#pragma unroll
        for (int k = 0; k < R; ++k) {
            const double u = x[2 + k], v = x[2 + R + k];
            uv = fma(u, v, uv);
            q[DQ + k] += u;
            q[DQ + R + k] += v;
        }
        q[5] = fma(uv, uv, q[5]);
    }
    double* out = partial + ((size_t)(blockIdx.y * 4 + warp) * T + t) * NQ;
#pragma unroll
    for (int k = 0; k < NQ; ++k) out[k] = q[k];
}

// sums[t][q] = sum over the (block, warp) slots: one warp per output element, lanes stride over the slots and combine by
// shuffles -- a fixed order, so the result is reproducible
__global__ void __launch_bounds__(128) k_diag_rows_reduce(const double* __restrict__ partial, int nslots, int T, int NQ,
                                                          double* __restrict__ sums) {
    const int e = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (e >= T * NQ) return;
    double v = 0.0;
    for (int s = lane; s < nslots; s += 32) v += partial[(size_t)s * T * NQ + e];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) sums[e] = v;
}

// one thread per time step.  gram: (T, 2, r, r) = U'U, V'V of X.
__global__ void k_diag_contrib(const double* __restrict__ sums, const double* __restrict__ gram, int n, int T, int r,
                               int exclude_diagonal, double* __restrict__ additive, double* __restrict__ multiplicative) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const double* q = sums + (size_t)t * (DQ + 2 * r);
    const double nn = (double)n;
    double add = nn * q[2] + nn * q[3] + 2.0 * q[0] * q[1];
    double mul = 0.0;
    const double* gu = gram + (size_t)t * 2 * r * r;
    const double* gv = gu + r * r;
    for (int e = 0; e < r * r; ++e) mul = fma(gu[e], gv[e], mul);
    double cnt = nn * nn;
    if (exclude_diagonal) {
        add -= q[4];
        mul -= q[5];
        cnt = nn * (nn - 1.0);
    }
    // n = 1 without the diagonal has no pair: the mean over none is NaN (add and mul are rounding residues there)
    additive[t] = cnt > 0.0 ? add / cnt : CUDART_NAN;
    multiplicative[t] = cnt > 0.0 ? mul / cnt : CUDART_NAN;
}

// Pearson correlation of the flattened n x n products U V' (diagonal included), one thread per time step.
// When either side's products are all zero (its U or V block is zero) the variance is exactly 0 and the correlation is
// undefined: NaN, as torch.corrcoef returns.  A variance <= 0 from rounding is treated the same, and the clamp to [-1, 1]
// passes NaN through (fmax(-1, NaN) would return -1).
__global__ void k_diag_corr(const double* __restrict__ sums_e, const double* __restrict__ sums_t, const double* __restrict__ gram_e,
                            const double* __restrict__ gram_t, const double* __restrict__ cross, int n, int T, int r,
                            double* __restrict__ corr) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int NQ = DQ + 2 * r, rr = r * r;
    const double* qe = sums_e + (size_t)t * NQ;
    const double* qt = sums_t + (size_t)t * NQ;
    double se = 0.0, st = 0.0;
    for (int k = 0; k < r; ++k) {
        se = fma(qe[DQ + k], qe[DQ + r + k], se);
        st = fma(qt[DQ + k], qt[DQ + r + k], st);
    }
    double see = 0.0, stt = 0.0, ste = 0.0;
    const double* ge = gram_e + (size_t)t * 2 * rr;
    const double* gt = gram_t + (size_t)t * 2 * rr;
    const double* gx = cross + (size_t)t * 2 * rr;
    for (int e = 0; e < rr; ++e) {
        see = fma(ge[e], ge[rr + e], see);
        stt = fma(gt[e], gt[rr + e], stt);
        ste = fma(gx[e], gx[rr + e], ste);
    }
    const double N = (double)n * (double)n;
    double c = 0.0;
    if (N > 1.0) {                                   // multiplicative_strength_comparison.py:82-86
        const double cov = ste - st * se / N, ve = see - se * se / N, vt = stt - st * st / N;
        if (ve > 0.0 && vt > 0.0) {
            c = cov / sqrt(ve * vt);
            c = c > 1.0 ? 1.0 : (c < -1.0 ? -1.0 : c);     // torch.corrcoef clips to [-1, 1]; NaN stays NaN
        } else {
            c = CUDART_NAN;
        }
    }
    corr[t] = c;
}

__global__ void k_diag_sqdiff(const double* __restrict__ A, const double* __restrict__ B, long count, double* __restrict__ partial) {
    __shared__ double red[8];
    double s = 0.0;
    for (long e = (long)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (long)gridDim.x * blockDim.x) {
        const double df = A[e] - B[e];
        s = fma(df, df, s);
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double v = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += red[w];
        partial[blockIdx.x] = v;
    }
}

template <int R>
void launch_diag_rows(dim3 grid, cudaStream_t st, const double* X, int n, int T, double* partial) {
    k_diag_rows<R><<<grid, 128, 0, st>>>(X, n, T, partial);
}

// row sums + Gram matrices of one state array: sums (T, DQ+2r), gram (T, 2, r, r); scratch is freed stream-ordered
int diag_moments(int n, int T, int r, const double* X, double* sums, double* gram, cudaStream_t st);

int split_rows(int n, int T) {
    // enough (time step, row split) blocks to keep every SM busy with the latency-bound accumulation, >= 64 rows each
    int ns = (4736 + T - 1) / T;            // ~32 blocks per SM
    if (ns > 64) ns = 64;
    if (ns > (n + 63) / 64) ns = (n + 63) / 64;
    return ns < 1 ? 1 : ns;
}
}  // namespace

extern "C" int tame_align_states(int32_t n, int32_t T, int32_t r, const double* X_est_dev, const double* X_true_dev,
                                 int32_t align_each_time, double* X_aligned_dev, double* rot_dev, double* mse_host,
                                 void* cuda_stream) {
    if (n < 1 || T < 1) return tame_set_error(TAME_EINVAL, "tame_align_states: n and T must be positive");
    if (r < 1 || r > TAME_MAX_R) return tame_set_error(TAME_EINVAL, "tame_align_states: latent_dim must be 1..%d", TAME_MAX_R);
    if (!X_est_dev || !X_true_dev || !X_aligned_dev) return tame_set_error(TAME_EINVAL, "tame_align_states: null argument");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int d = 2 + 2 * r, each = align_each_time ? 1 : 0;
    const int k = each ? r : 2 * r, nblk = each ? 2 : 1, Tm = each ? T : 1;
    const int NS = split_rows(n, Tm);
    const size_t rot_count = (size_t)Tm * nblk * k * k;
    const int nbx = (T + 31) / 32;
    int nby = (148 * 8 + nbx - 1) / nbx;           // ~8 blocks per SM, every warp walks >= 1 node
    if (nby > (n + 3) / 4) nby = (n + 3) / 4;
    if (nby < 1) nby = 1;
    const int nmat = Tm * nblk, kk = k * k;
    double *partial = nullptr, *rot = rot_dev, *means = nullptr, *sse = nullptr, *mse = nullptr, *M = nullptr;
    ACK(cudaMallocAsync((void**)&partial, sizeof(double) * (size_t)Tm * NS * nblk * kk, st));
    ACK(cudaMallocAsync((void**)&M, sizeof(double) * (size_t)nmat * kk, st));
    if (!rot) ACK(cudaMallocAsync((void**)&rot, sizeof(double) * rot_count, st));
    ACK(cudaMallocAsync((void**)&sse, sizeof(double) * (size_t)nby * nbx, st));
    ACK(cudaMallocAsync((void**)&mse, sizeof(double), st));
    if (each) {
        k_align_cross<<<dim3(T, NS), 128, 0, st>>>(X_est_dev, X_true_dev, n, T, d, 2, k, nblk, partial);
        tame_count_launch(1);
    } else {
        ACK(cudaMallocAsync((void**)&means, sizeof(double) * 2 * (size_t)n * d, st));
        const int nb = (int)(((long)n * d + 255) / 256);
        k_align_tmean<<<nb, 256, 0, st>>>(X_est_dev, n, T, d, means);
        k_align_tmean<<<nb, 256, 0, st>>>(X_true_dev, n, T, d, means + (size_t)n * d);
        k_align_cross<<<dim3(1, NS), 128, 0, st>>>(means, means + (size_t)n * d, n, 1, d, 2, k, 1, partial);
        tame_count_launch(3);
    }
    k_align_reduce<<<(nmat * kk + 255) / 256, 256, 0, st>>>(partial, nmat, nblk, NS, kk, M);
    k_align_rot<<<(nmat + 3) / 4, 128, 0, st>>>(M, nmat, k, rot);
    {
        const dim3 grid(nbx, nby);
        cudaError_t ae = cudaSuccess;
        switch (r) {
            case 1: ae = launch_apply<1>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
            case 2: ae = launch_apply<2>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
            case 3: ae = launch_apply<3>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
            case 4: ae = launch_apply<4>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
            case 5: ae = launch_apply<5>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
            case 6: ae = launch_apply<6>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
            case 7: ae = launch_apply<7>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
            default: ae = launch_apply<8>(each, grid, st, X_est_dev, X_true_dev, n, T, rot, X_aligned_dev, sse); break;
        }
        ACK(ae);
    }
    k_align_sum<<<1, 256, 0, st>>>(sse, (long)nby * nbx, 1, 1.0 / ((double)n * T * d), mse);
    tame_count_launch(4);
    ACK(cudaGetLastError());
    double host = 0.0;
    if (mse_host) ACK(cudaMemcpyAsync(&host, mse, sizeof(double), cudaMemcpyDeviceToHost, st));
    ACK(cudaFreeAsync(partial, st));
    ACK(cudaFreeAsync(M, st));
    if (!rot_dev) ACK(cudaFreeAsync(rot, st));
    if (means) ACK(cudaFreeAsync(means, st));
    ACK(cudaFreeAsync(sse, st));
    ACK(cudaFreeAsync(mse, st));
    if (mse_host) {
        ACK(cudaStreamSynchronize(st));
        *mse_host = host;
    }
    return TAME_OK;
}

extern "C" int tame_align_signs(int64_t rows, int32_t width, const double* X_est_dev, const double* X_true_dev,
                                double* X_aligned_dev, double* mse_host, void* cuda_stream) {
    if (rows < 1 || width < 1) return tame_set_error(TAME_EINVAL, "tame_align_signs: empty input");
    if (!X_est_dev || !X_true_dev || !X_aligned_dev) return tame_set_error(TAME_EINVAL, "tame_align_signs: null argument");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const long nb = (rows + 255) / 256;
    double *sse = nullptr, *mse = nullptr;
    if (mse_host) {
        ACK(cudaMallocAsync((void**)&sse, sizeof(double) * (size_t)nb, st));
        ACK(cudaMallocAsync((void**)&mse, sizeof(double), st));
    }
    k_align_signs<<<(unsigned)nb, 256, 0, st>>>(X_est_dev, X_true_dev, rows, width, X_aligned_dev, sse);
    tame_count_launch(1);
    if (mse_host) {
        k_align_sum<<<1, 256, 0, st>>>(sse, nb, 1, 1.0 / ((double)rows * width), mse);
        tame_count_launch(1);
        double host = 0.0;
        ACK(cudaMemcpyAsync(&host, mse, sizeof(double), cudaMemcpyDeviceToHost, st));
        ACK(cudaFreeAsync(sse, st));
        ACK(cudaFreeAsync(mse, st));
        ACK(cudaStreamSynchronize(st));
        *mse_host = host;
    }
    ACK(cudaGetLastError());
    return TAME_OK;
}

extern "C" int tame_procrustes(int32_t n, int32_t k, const double* X_est_dev, const double* X_true_dev, int32_t scaling,
                               double* X_aligned_dev, double* rot_dev, void* cuda_stream) {
    if (n < 1) return tame_set_error(TAME_EINVAL, "tame_procrustes: empty input");
    if (k < 1 || k > KMAX) return tame_set_error(TAME_EINVAL, "tame_procrustes: width must be 1..%d", KMAX);
    if (!X_est_dev || !X_true_dev || !X_aligned_dev) return tame_set_error(TAME_EINVAL, "tame_procrustes: null argument");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int NS = split_rows(n, 1);
    const int nb = (n + 127) / 128;
    double *partial = nullptr, *rot = rot_dev, *nd = nullptr, *numden = nullptr, *M = nullptr;
    ACK(cudaMallocAsync((void**)&partial, sizeof(double) * (size_t)NS * k * k, st));
    ACK(cudaMallocAsync((void**)&M, sizeof(double) * k * k, st));
    if (!rot) ACK(cudaMallocAsync((void**)&rot, sizeof(double) * k * k, st));
    ACK(cudaMallocAsync((void**)&nd, sizeof(double) * 2 * (size_t)nb, st));
    ACK(cudaMallocAsync((void**)&numden, sizeof(double) * 2, st));
    k_align_cross<<<dim3(1, NS), 128, 0, st>>>(X_est_dev, X_true_dev, n, 1, k, 0, k, 1, partial);
    k_align_reduce<<<(k * k + 255) / 256, 256, 0, st>>>(partial, 1, 1, NS, k * k, M);
    k_align_rot<<<1, 128, 0, st>>>(M, 1, k, rot);
    k_align_rotate<<<nb, 128, 0, st>>>(X_est_dev, X_true_dev, n, k, rot, X_aligned_dev, nd);
    tame_count_launch(4);
    if (scaling) {
        k_align_sum<<<1, 256, 0, st>>>(nd, nb, 2, 1.0, numden);
        const long count = (long)n * k;
        k_align_scale<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(X_aligned_dev, count, numden);
        tame_count_launch(2);
    }
    ACK(cudaGetLastError());
    ACK(cudaFreeAsync(partial, st));
    ACK(cudaFreeAsync(M, st));
    if (!rot_dev) ACK(cudaFreeAsync(rot, st));
    ACK(cudaFreeAsync(nd, st));
    ACK(cudaFreeAsync(numden, st));
    return TAME_OK;
}

namespace {
int diag_cross(int n, int T, int r, const double* est, const double* tru, double* out, cudaStream_t st) {
    // out (T, 2, r, r) = [X_true_U' X_est_U, X_true_V' X_est_V] per time step
    const int d = 2 + 2 * r, NS = split_rows(n, T), kk = r * r;
    double* partial = nullptr;
    ACK(cudaMallocAsync((void**)&partial, sizeof(double) * (size_t)T * NS * 2 * kk, st));
    k_align_cross<<<dim3(T, NS), 128, 0, st>>>(est, tru, n, T, d, 2, r, 2, partial);
    k_align_reduce<<<(T * 2 * kk + 255) / 256, 256, 0, st>>>(partial, T * 2, 2, NS, kk, out);
    tame_count_launch(2);
    ACK(cudaFreeAsync(partial, st));
    return TAME_OK;
}

int diag_moments(int n, int T, int r, const double* X, double* sums, double* gram, cudaStream_t st) {
    const int NQ = DQ + 2 * r, nbx = (T + 31) / 32;
    int nby = (148 * 8 + nbx - 1) / nbx;
    if (nby > (n + 3) / 4) nby = (n + 3) / 4;
    if (nby < 1) nby = 1;
    double* partial = nullptr;
    const size_t pbytes = sizeof(double) * (size_t)nby * 4 * T * NQ;
    ACK(cudaMallocAsync((void**)&partial, pbytes, st));
    ACK(cudaMemsetAsync(partial, 0, pbytes, st));        // slots of warps without rows stay zero
    const dim3 grid(nbx, nby);
    switch (r) {
        case 1: launch_diag_rows<1>(grid, st, X, n, T, partial); break;
        case 2: launch_diag_rows<2>(grid, st, X, n, T, partial); break;
        case 3: launch_diag_rows<3>(grid, st, X, n, T, partial); break;
        case 4: launch_diag_rows<4>(grid, st, X, n, T, partial); break;
        case 5: launch_diag_rows<5>(grid, st, X, n, T, partial); break;
        case 6: launch_diag_rows<6>(grid, st, X, n, T, partial); break;
        case 7: launch_diag_rows<7>(grid, st, X, n, T, partial); break;
        default: launch_diag_rows<8>(grid, st, X, n, T, partial); break;
    }
    k_diag_rows_reduce<<<(T * NQ + 3) / 4, 128, 0, st>>>(partial, nby * 4, T, NQ, sums);
    tame_count_launch(2);
    ACK(cudaFreeAsync(partial, st));
    if (gram) return diag_cross(n, T, r, X, X, gram, st);
    return TAME_OK;
}
}  // namespace

extern "C" int tame_contributions(int32_t n, int32_t T, int32_t r, const double* X_dev, int32_t exclude_diagonal,
                                  double* additive_dev, double* multiplicative_dev, void* cuda_stream) {
    if (n < 1 || T < 1) return tame_set_error(TAME_EINVAL, "tame_contributions: n and T must be positive");
    if (r < 1 || r > TAME_MAX_R) return tame_set_error(TAME_EINVAL, "tame_contributions: latent_dim must be 1..%d", TAME_MAX_R);
    if (!X_dev || !additive_dev || !multiplicative_dev) return tame_set_error(TAME_EINVAL, "tame_contributions: null argument");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    double *sums = nullptr, *gram = nullptr;
    ACK(cudaMallocAsync((void**)&sums, sizeof(double) * (size_t)T * (DQ + 2 * r), st));
    ACK(cudaMallocAsync((void**)&gram, sizeof(double) * (size_t)T * 2 * r * r, st));
    int rc = diag_moments(n, T, r, X_dev, sums, gram, st);
    if (rc != TAME_OK) return rc;
    k_diag_contrib<<<(T + 127) / 128, 128, 0, st>>>(sums, gram, n, T, r, exclude_diagonal ? 1 : 0, additive_dev, multiplicative_dev);
    tame_count_launch(1);
    ACK(cudaGetLastError());
    ACK(cudaFreeAsync(sums, st));
    ACK(cudaFreeAsync(gram, st));
    return TAME_OK;
}

extern "C" int tame_uv_correlation(int32_t n, int32_t T, int32_t r, const double* X_est_dev, const double* X_true_dev,
                                   double* corr_dev, void* cuda_stream) {
    if (n < 1 || T < 1) return tame_set_error(TAME_EINVAL, "tame_uv_correlation: n and T must be positive");
    if (r < 1 || r > TAME_MAX_R) return tame_set_error(TAME_EINVAL, "tame_uv_correlation: latent_dim must be 1..%d", TAME_MAX_R);
    if (!X_est_dev || !X_true_dev || !corr_dev) return tame_set_error(TAME_EINVAL, "tame_uv_correlation: null argument");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t ns = (size_t)T * (DQ + 2 * r), ng = (size_t)T * 2 * r * r;
    double* buf = nullptr;
    ACK(cudaMallocAsync((void**)&buf, sizeof(double) * (2 * ns + 3 * ng), st));
    double *sums_e = buf, *sums_t = buf + ns, *gram_e = buf + 2 * ns, *gram_t = gram_e + ng, *cross = gram_t + ng;
    int rc = diag_moments(n, T, r, X_est_dev, sums_e, gram_e, st);
    if (rc == TAME_OK) rc = diag_moments(n, T, r, X_true_dev, sums_t, gram_t, st);
    if (rc == TAME_OK) rc = diag_cross(n, T, r, X_est_dev, X_true_dev, cross, st);
    if (rc != TAME_OK) return rc;
    k_diag_corr<<<(T + 127) / 128, 128, 0, st>>>(sums_e, sums_t, gram_e, gram_t, cross, n, T, r, corr_dev);
    tame_count_launch(1);
    ACK(cudaGetLastError());
    ACK(cudaFreeAsync(buf, st));
    return TAME_OK;
}

extern "C" int tame_state_mse(int64_t count, const double* A_dev, const double* B_dev, double* mse_host, void* cuda_stream) {
    if (count < 1 || !A_dev || !B_dev || !mse_host) return tame_set_error(TAME_EINVAL, "tame_state_mse: bad argument");
    cudaStream_t st = (cudaStream_t)cuda_stream;
    long nb = (count + 2047) / 2048;
    if (nb > 148 * 8) nb = 148 * 8;
    double *partial = nullptr, *mse = nullptr;
    ACK(cudaMallocAsync((void**)&partial, sizeof(double) * (size_t)nb, st));
    ACK(cudaMallocAsync((void**)&mse, sizeof(double), st));
    k_diag_sqdiff<<<(unsigned)nb, 256, 0, st>>>(A_dev, B_dev, count, partial);
    k_align_sum<<<1, 256, 0, st>>>(partial, nb, 1, 1.0 / (double)count, mse);
    tame_count_launch(2);
    double host = 0.0;
    ACK(cudaMemcpyAsync(&host, mse, sizeof(double), cudaMemcpyDeviceToHost, st));
    ACK(cudaFreeAsync(partial, st));
    ACK(cudaFreeAsync(mse, st));
    ACK(cudaStreamSynchronize(st));
    *mse_host = host;
    return TAME_OK;
}

