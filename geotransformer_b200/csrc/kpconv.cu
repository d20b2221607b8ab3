// KPConv-FPN backbone kernels: kernel-point convolution, Linear, GroupNorm(+LeakyReLU/+residual), max-pool,
// nearest-upsample+concat.
//
// Reference semantics (all under /root/reference/geotransformer/modules/kpconv):
//   kpconv.py:79-122        KPConv.forward
//   modules.py:33-50        GroupNorm over the whole stacked (1,C,N) tensor
//   modules.py:53-104       UnaryBlock / LastUnaryBlock
//   functional.py:6-22,54-67 nearest_upsample / maxpool
// The reference runs these as ~20 eager ATen launches per block with (M,H,K,3)/(M,H,C) intermediates in HBM;
// here one kernel gathers each neighbour row once, keeps the K=15 kernel-point accumulators in registers,
// stages the (queries x K*C) tile in shared memory and contracts it with the weights without leaving the SM.
// Feature tables are L2-resident; the compulsory HBM traffic is the index table + the output.
#include "common.cuh"
#include "geob200.h"

namespace geob200 {

constexpr int KP = 15;        // kernel points of every shipped model (config.py: backbone.kernel_size)
constexpr int KP_PAD = 16;
constexpr int TQ = 32;        // queries per CTA
constexpr int CC = 32;        // input-channel chunk staged in shared memory (one float per lane per neighbour row)

__device__ __forceinline__ void influence15(const float* __restrict__ kp_s, float rx, float ry, float rz, float inv_dummy,
                                            float sigma, float* w) {
#pragma unroll
    for (int k = 0; k < KP; ++k) {
        const float dx = rx - kp_s[3 * k], dy = ry - kp_s[3 * k + 1], dz = rz - kp_s[3 * k + 2];
        const float sq = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
        w[k] = fmaxf(1.0f - sqrtf(sq) / sigma, 0.0f);      // kpconv.py:96-99
    }
    (void)inv_dummy;
}

// First layer of every backbone: Cin == 1 (features are all-ones columns, model input_dim = 1).
// out[m][c'] = (sum_k (sum_h w[h][k] f[h]) W[k][0][c']) / max(#{h: f[h] > 0}, 1) + bias
// Half a warp per query point (16 queries per CTA): with H = 27..38 neighbours a full warp spends its second pass over the
// neighbour list almost idle; 16 lanes take 2-3 passes at 80-100 % occupancy and the 15 reductions need 4 shuffle steps.
__global__ void __launch_bounds__(256) kpconv_c1_kernel(const float* __restrict__ feats, const float* __restrict__ q_pts,
                                                        const float* __restrict__ s_pts, const long long* __restrict__ nbr,
                                                        int H, const float* __restrict__ kp, const float* __restrict__ W,
                                                        const float* __restrict__ bias, float sigma, int Ns, int M, int Cout,
                                                        float* __restrict__ out) {
    __shared__ float kp_s[KP * 3];
    __shared__ float wk_s[16][KP_PAD];
    __shared__ float np_s[16];
    if (threadIdx.x < KP * 3) kp_s[threadIdx.x] = kp[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int sub = lane >> 4, sl = lane & 15;
    const int slot = warp * 2 + sub;
    const int m = blockIdx.x * 16 + slot;
    const bool live = m < M;
    float acc[KP];
#pragma unroll
    for (int k = 0; k < KP; ++k) acc[k] = 0.f;
    int npos = 0;
    if (live) {
        const float qx = q_pts[3ll * m], qy = q_pts[3ll * m + 1], qz = q_pts[3ll * m + 2];
        for (int h = sl; h < H; h += 16) {
            const long long idx = nbr[(long long)m * H + h];
            if (idx < Ns) {
                float w[KP];
                influence15(kp_s, s_pts[3 * idx] - qx, s_pts[3 * idx + 1] - qy, s_pts[3 * idx + 2] - qz, 0.f, sigma, w);
                const float f = feats[idx];
                npos += (f > 0.f);
#pragma unroll
                for (int k = 0; k < KP; ++k) acc[k] = fmaf(w[k], f, acc[k]);
            }
        }
    }
    // reductions over the 16 lanes of the half warp (xor offsets < 16 stay inside it); every lane of the warp takes part
#pragma unroll
    for (int k = 0; k < KP; ++k) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    }
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) npos += __shfl_xor_sync(0xffffffffu, npos, o);
    if (sl == 0) {
#pragma unroll
        for (int k = 0; k < KP; ++k) wk_s[slot][k] = acc[k];
        np_s[slot] = (float)max(npos, 1);
    }
    __syncwarp();
    if (!live) return;
    for (int c = sl; c < Cout; c += 16) {
        float o = 0.f;
#pragma unroll
        for (int k = 0; k < KP; ++k) o = fmaf(wk_s[slot][k], W[k * Cout + c], o);
        o = o / np_s[slot];
        if (bias != nullptr) o += bias[c];
        out[(long long)m * Cout + c] = o;
    }
}

// pos[n] = 1 iff the sum of support row n is > 0: KPConv normalises by the number of such neighbours (kpconv.py:113-116)
__global__ void __launch_bounds__(256) row_positive_kernel(const float* __restrict__ x, int N, int C, unsigned char* __restrict__ pos) {
    const int lane = threadIdx.x & 31;
    const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (n >= N) return;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s += x[(long long)n * C + c];
    s = warp_sum(s);
    if (lane == 0) pos[n] = (s > 0.f) ? 1 : 0;
}

// KPConv, stage 1 of 2 (tensor-core path): wf[m][k*Cin + c] = sum_h influence[m][h][k] * f[nbr[m][h]][c]   (kpconv.py:91-105)
// One warp per query point, small shared-memory footprint (many resident warps hide the gather latency); the neighbour
// rows are fetched eight at a time.  Also emits inv_count[m] = 1 / max(#neighbours with a positive feature sum, 1)
// (kpconv.py:113-116).  Stage 2 is the 3xTF32 tcgen05 GEMM wf (M x 15 Cin) . W (15 Cin x Cout) with the per-row scale and the
// bias applied in its epilogue (linear_tc.cu).
// CPL = channels per lane: 2 when Cin is a multiple of 64 (every broadcast read of an influence row then feeds 30 FMAs instead
// of 15; with 15 the kernel is bound by the shared-memory pipe, 4 LDS.128 per 15 FMAs)
template <int CPL>
__global__ void __launch_bounds__(256, 4) kpconv_gather_kernel(const float* __restrict__ feats, const unsigned char* __restrict__ pos,
                                                            const float* __restrict__ q_pts, const float* __restrict__ s_pts,
                                                            const long long* __restrict__ nbr, int H, const float* __restrict__ kp,
                                                            float sigma, int Ns, int M, int Cin, float* __restrict__ wf,
                                                            float* __restrict__ inv_count) {
    __shared__ float infl[8][32][KP_PAD];
    __shared__ int sidx[8][32];
    __shared__ float kp_s[KP * 3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < KP * 3) kp_s[threadIdx.x] = kp[threadIdx.x];
    __syncthreads();
    const int m = blockIdx.x * 8 + warp;
    if (m >= M) return;
    const float qx = q_pts[3ll * m], qy = q_pts[3ll * m + 1], qz = q_pts[3ll * m + 2];
    int npos = 0;
    for (int c0 = 0; c0 < Cin; c0 += 32 * CPL) {
        float acc[CPL][KP];
#pragma unroll
        for (int p = 0; p < CPL; ++p)
#pragma unroll
            for (int k = 0; k < KP; ++k) acc[p][k] = 0.f;
        for (int h0 = 0; h0 < H; h0 += 32) {
            const int h = h0 + lane;
            const long long idx = (h < H) ? nbr[(long long)m * H + h] : (long long)Ns;
            float w[KP];
            int id = 0;
            if (idx < Ns) {
                id = (int)idx;
                influence15(kp_s, s_pts[3 * idx] - qx, s_pts[3 * idx + 1] - qy, s_pts[3 * idx + 2] - qz, 0.f, sigma, w);
                if (c0 == 0) npos += pos[idx];
            } else {
#pragma unroll
                for (int k = 0; k < KP; ++k) w[k] = 0.f;
            }
            __syncwarp();
#pragma unroll
            for (int k = 0; k < KP; ++k) infl[warp][lane][k] = w[k];
            infl[warp][lane][KP] = 0.f;
            sidx[warp][lane] = id;
            __syncwarp();
            const int hn = min(32, H - h0);
            for (int hb = 0; hb < hn; hb += 8) {
                float f[8][CPL];
#pragma unroll
                for (int u = 0; u < 8; ++u)
#pragma unroll
                    for (int p = 0; p < CPL; ++p)
                        f[u][p] = __ldg(feats + (long long)sidx[warp][(hb + u) & 31] * Cin + c0 + 32 * p + lane);
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    if (hb + u < hn) {
                        const float4* iv = reinterpret_cast<const float4*>(&infl[warp][hb + u][0]);
                        const float4 a0 = iv[0], a1 = iv[1], a2 = iv[2], a3 = iv[3];
                        const float wv[16] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y, a2.z, a2.w, a3.x, a3.y, a3.z, a3.w};
#pragma unroll
                        for (int p = 0; p < CPL; ++p)
#pragma unroll
                            for (int k = 0; k < KP; ++k) acc[p][k] = fmaf(wv[k], f[u][p], acc[p][k]);
                    }
                }
            }
        }
#pragma unroll
        for (int p = 0; p < CPL; ++p) {
            float* wrow = wf + (long long)m * (KP * Cin) + c0 + 32 * p + lane;
#pragma unroll
            for (int k = 0; k < KP; ++k) wrow[(long long)k * Cin] = acc[p][k];
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) npos += __shfl_xor_sync(0xffffffffu, npos, o);
    if (lane == 0) inv_count[m] = 1.0f / (float)max(npos, 1);
}

static void launch_kpconv_gather(const float* s_feats, const unsigned char* pos, const float* q_points, const float* s_points,
                                 const long long* neighbors, int n_neighbors, const float* kernel_points, float sigma, int n_support,
                                 int n_query, int c_in, float* wf, float* inv_count, cudaStream_t st) {
    const unsigned grid = (unsigned)((n_query + 7) / 8);
    if (c_in % 64 == 0)
        kpconv_gather_kernel<2><<<grid, 256, 0, st>>>(s_feats, pos, q_points, s_points, neighbors, n_neighbors, kernel_points, sigma,
                                                     n_support, n_query, c_in, wf, inv_count);
    else
        kpconv_gather_kernel<1><<<grid, 256, 0, st>>>(s_feats, pos, q_points, s_points, neighbors, n_neighbors, kernel_points, sigma,
                                                     n_support, n_query, c_in, wf, inv_count);
}

// General KPConv, Cin % 32 == 0 and Cout % 32 == 0 (mid channels 32..512 of the bottleneck blocks).
// RC = output columns per lane handled by this CTA (the CTA owns columns [col0, col0 + 32*RC)).
// Input channels are processed in chunks of CC = 32 (one float per lane per neighbour row): the tile
// wf[TQ][15*32] lives in 61 KB of shared memory so that 2-3 CTAs share an SM, and the neighbour rows of a query are
// fetched eight at a time so that the gather is throughput- rather than latency-bound.
template <int RC>
__global__ void __launch_bounds__(256) kpconv_kernel(const float* __restrict__ feats, const unsigned char* __restrict__ pos,
                                                     const float* __restrict__ q_pts, const float* __restrict__ s_pts,
                                                     const long long* __restrict__ nbr, int H, const float* __restrict__ kp,
                                                     const float* __restrict__ W, const float* __restrict__ bias, float sigma,
                                                     int Ns, int M, int Cin, int Cout, float* __restrict__ out) {
    const int col0 = blockIdx.y * (RC * 32);
    extern __shared__ float smem[];
    float* wf = smem;                                  // [TQ][KP*CC]
    float* infl = wf + TQ * KP * CC;                   // [8 warps][32][KP_PAD]
    int* sidx = (int*)(infl + 8 * 32 * KP_PAD);        // [8][32]
    float* npos_s = (float*)(sidx + 8 * 32);           // [TQ]
    float* kp_s = npos_s + TQ;                         // [KP*3]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < KP * 3) kp_s[threadIdx.x] = kp[threadIdx.x];
    __syncthreads();
    const int m0 = blockIdx.x * TQ;

    float acc_out[4][RC];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int j = 0; j < RC; ++j) acc_out[r][j] = 0.f;

    for (int c0 = 0; c0 < Cin; c0 += CC) {
        // ---- phase A: one warp per query; acc[k] = sum_h infl[h][k] * f[nbr_h][c0 + lane]
        for (int q = warp; q < TQ; q += 8) {
            const int m = m0 + q;
            float acc[KP];
#pragma unroll
            for (int k = 0; k < KP; ++k) acc[k] = 0.f;
            int npos = 0;
            if (m < M) {
                const float qx = q_pts[3ll * m], qy = q_pts[3ll * m + 1], qz = q_pts[3ll * m + 2];
                for (int h0 = 0; h0 < H; h0 += 32) {
                    const int h = h0 + lane;
                    long long idx = (h < H) ? nbr[(long long)m * H + h] : (long long)Ns;
                    float w[KP];
                    int id = 0;                         // shadow neighbours: zero influence, row 0 is read but unused
                    if (idx < Ns) {
                        id = (int)idx;
                        influence15(kp_s, s_pts[3 * idx] - qx, s_pts[3 * idx + 1] - qy, s_pts[3 * idx + 2] - qz, 0.f, sigma, w);
                        if (c0 == 0) npos += pos[idx];
                    } else {
#pragma unroll
                        for (int k = 0; k < KP; ++k) w[k] = 0.f;
                    }
                    float* irow = infl + (warp * 32 + lane) * KP_PAD;
#pragma unroll
                    for (int k = 0; k < KP; ++k) irow[k] = w[k];
                    irow[KP] = 0.f;
                    sidx[warp * 32 + lane] = id;
                    __syncwarp();
                    const int hn = min(32, H - h0);
                    for (int hb = 0; hb < hn; hb += 8) {
                        float f[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) {   // 8 independent row fetches in flight (rows past hn have zero weights)
                            const int id2 = sidx[warp * 32 + ((hb + u) & 31)];
                            f[u] = __ldg(feats + (long long)id2 * Cin + c0 + lane);
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            if (hb + u < hn) {
                                const float4* iv = reinterpret_cast<const float4*>(infl + (warp * 32 + hb + u) * KP_PAD);
                                const float4 a0 = iv[0], a1 = iv[1], a2 = iv[2], a3 = iv[3];
                                const float wv[16] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w,
                                                      a2.x, a2.y, a2.z, a2.w, a3.x, a3.y, a3.z, a3.w};
#pragma unroll
                                for (int k = 0; k < KP; ++k) acc[k] = fmaf(wv[k], f[u], acc[k]);
                            }
                        }
                    }
                    __syncwarp();
                }
            }
            float* wrow = wf + q * (KP * CC);
#pragma unroll
            for (int k = 0; k < KP; ++k) wrow[k * CC + lane] = acc[k];
            if (c0 == 0) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) npos += __shfl_xor_sync(0xffffffffu, npos, o);
                if (lane == 0) npos_s[q] = (float)max(npos, 1);
            }
        }
        __syncthreads();
        // ---- phase B: out[TQ x 32*RC] += wf[TQ x (KP*CC)] . W[k][c0:c0+CC][col0 : col0+32*RC]
        // warp `warp` owns query rows 4*warp .. 4*warp+3 ; lane owns columns col0 + lane + 32 j
        {
            const float* a0p = wf + (4 * warp + 0) * (KP * CC);
            const float* a1p = wf + (4 * warp + 1) * (KP * CC);
            const float* a2p = wf + (4 * warp + 2) * (KP * CC);
            const float* a3p = wf + (4 * warp + 3) * (KP * CC);
            for (int k = 0; k < KP; ++k) {
                const float* wbase = W + ((long long)k * Cin + c0) * Cout + col0 + lane;
#pragma unroll 2
                for (int c = 0; c < CC; c += 4) {
                    const float4 x0 = *reinterpret_cast<const float4*>(a0p + k * CC + c);
                    const float4 x1 = *reinterpret_cast<const float4*>(a1p + k * CC + c);
                    const float4 x2 = *reinterpret_cast<const float4*>(a2p + k * CC + c);
                    const float4 x3 = *reinterpret_cast<const float4*>(a3p + k * CC + c);
                    float b[4][RC];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
#pragma unroll
                        for (int j = 0; j < RC; ++j) b[u][j] = __ldg(wbase + (long long)(c + u) * Cout + 32 * j);
#pragma unroll
                    for (int j = 0; j < RC; ++j) {
                        acc_out[0][j] = fmaf(x0.x, b[0][j], acc_out[0][j]); acc_out[0][j] = fmaf(x0.y, b[1][j], acc_out[0][j]);
                        acc_out[0][j] = fmaf(x0.z, b[2][j], acc_out[0][j]); acc_out[0][j] = fmaf(x0.w, b[3][j], acc_out[0][j]);
                        acc_out[1][j] = fmaf(x1.x, b[0][j], acc_out[1][j]); acc_out[1][j] = fmaf(x1.y, b[1][j], acc_out[1][j]);
                        acc_out[1][j] = fmaf(x1.z, b[2][j], acc_out[1][j]); acc_out[1][j] = fmaf(x1.w, b[3][j], acc_out[1][j]);
                        acc_out[2][j] = fmaf(x2.x, b[0][j], acc_out[2][j]); acc_out[2][j] = fmaf(x2.y, b[1][j], acc_out[2][j]);
                        acc_out[2][j] = fmaf(x2.z, b[2][j], acc_out[2][j]); acc_out[2][j] = fmaf(x2.w, b[3][j], acc_out[2][j]);
                        acc_out[3][j] = fmaf(x3.x, b[0][j], acc_out[3][j]); acc_out[3][j] = fmaf(x3.y, b[1][j], acc_out[3][j]);
                        acc_out[3][j] = fmaf(x3.z, b[2][j], acc_out[3][j]); acc_out[3][j] = fmaf(x3.w, b[3][j], acc_out[3][j]);
                    }
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int q = 4 * warp + r;
        const int m = m0 + q;
        if (m >= M) continue;
        const float nn = npos_s[q];
#pragma unroll
        for (int j = 0; j < RC; ++j) {
            const int c = col0 + lane + 32 * j;
            float o = acc_out[r][j] / nn;                          // kpconv.py:116
            if (bias != nullptr) o += bias[c];
            out[(long long)m * Cout + c] = o;
        }
    }
}

// ----------------------------------------------------------------------------------------------------------
// Linear: Y[M,N] = X[M,K] . W[N,K]^T + b  (torch.nn.Linear layout), optional ReLU.  Classic 64x64x16 smem-tiled
// fp32 SGEMM (the reference's Linears are true fp32: torch default allow_tf32=False).
// ----------------------------------------------------------------------------------------------------------
template <int BM, int BN>
__global__ void __launch_bounds__(256) linear_kernel(const float* __restrict__ X, int ldx, const float* __restrict__ W, int ldw,
                                                     const float* __restrict__ bias, float* __restrict__ Y, int ldy, int M,
                                                     int N, int K, int relu, long long sx, long long sw, long long sb,
                                                     long long sy) {
    X += sx * blockIdx.z; W += sw * blockIdx.z; Y += sy * blockIdx.z;
    if (bias != nullptr) bias += sb * blockIdx.z;
    constexpr int BK = 16;
    constexpr int TM = BM / 16, TN = BN / 16;
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
    const bool vec_ok = ((K & 3) == 0) && ((ldx & 3) == 0) && ((ldw & 3) == 0) &&
                        ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
    for (int k0 = 0; k0 < K; k0 += BK) {
        // load tiles: BM x BK of X and BN x BK of W, both K-contiguous; 4 floats per thread-load
        for (int e = threadIdx.x; e < BM * BK / 4; e += 256) {
            const int r = e / (BK / 4), kq = (e % (BK / 4)) * 4;
            const int gm = m0 + r, gk = k0 + kq;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (gm < M) {
                if (vec_ok && gk + 3 < K) v = *reinterpret_cast<const float4*>(X + (long long)gm * ldx + gk);
                else {
                    if (gk < K) v.x = X[(long long)gm * ldx + gk];
                    if (gk + 1 < K) v.y = X[(long long)gm * ldx + gk + 1];
                    if (gk + 2 < K) v.z = X[(long long)gm * ldx + gk + 2];
                    if (gk + 3 < K) v.w = X[(long long)gm * ldx + gk + 3];
                }
            }
            As[kq][r] = v.x; As[kq + 1][r] = v.y; As[kq + 2][r] = v.z; As[kq + 3][r] = v.w;
        }
        for (int e = threadIdx.x; e < BN * BK / 4; e += 256) {
            const int r = e / (BK / 4), kq = (e % (BK / 4)) * 4;
            const int gn = n0 + r, gk = k0 + kq;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (gn < N) {
                if (vec_ok && gk + 3 < K) v = *reinterpret_cast<const float4*>(W + (long long)gn * ldw + gk);
                else {
                    if (gk < K) v.x = W[(long long)gn * ldw + gk];
                    if (gk + 1 < K) v.y = W[(long long)gn * ldw + gk + 1];
                    if (gk + 2 < K) v.z = W[(long long)gn * ldw + gk + 2];
                    if (gk + 3 < K) v.w = W[(long long)gn * ldw + gk + 3];
                }
            }
            Bs[kq][r] = v.x; Bs[kq + 1][r] = v.y; Bs[kq + 2][r] = v.z; Bs[kq + 3][r] = v.w;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) a[i] = As[kk][ty + 16 * i];
#pragma unroll
            for (int j = 0; j < TN; ++j) b[j] = Bs[kk][tx + 16 * j];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int gm = m0 + ty + 16 * i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int gn = n0 + tx + 16 * j;
            if (gn >= N) continue;
            float v = acc[i][j] + (bias != nullptr ? bias[gn] : 0.f);
            if (relu) v = fmaxf(v, 0.f);
            Y[(long long)gm * ldy + gn] = v;
        }
    }
}

// ---- GroupNorm: statistics per pair (GnSeg; a single pair is one segment), then affine + residual + LeakyReLU ---------------
// Same per-128-row-tile partial layout as the GEMM epilogue produces ([tile][slot][2] doubles, slot = gn_slot_width channels),
// for activations whose producer has no fused statistics (fp32 fallbacks, split-K GEMMs, the c_in = 1 first KPConv).
__global__ void __launch_bounds__(256) gn_tile_stats_kernel(const float* __restrict__ x, int N, int C, int slot_width,
                                                            double* __restrict__ partial) {
    extern __shared__ double sh[];           // [C / slot_width][2]
    const int slots = C / slot_width;
    for (int i = threadIdx.x; i < 2 * slots; i += blockDim.x) sh[i] = 0.0;
    __syncthreads();
    const int r0 = blockIdx.x * 128, r1 = min(N, r0 + 128);
    const int cw = C < 256 ? C : 256;        // channels walked concurrently
    const int rpb = 256 / cw;                // row lanes
    const int rr = threadIdx.x / cw;
    if (rr < rpb)
        for (int c = threadIdx.x % cw; c < C; c += cw) {
            double s = 0.0, s2 = 0.0;
            for (int r = r0 + rr; r < r1; r += rpb) {
                const double v = (double)x[(long long)r * C + c];
                s += v;
                s2 += v * v;
            }
            atomicAdd(&sh[2 * (c / slot_width)], s);
            atomicAdd(&sh[2 * (c / slot_width) + 1], s2);
        }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * slots; i += blockDim.x) partial[(long long)blockIdx.x * 2 * slots + i] = sh[i];
}

// One 128-thread CTA per (group, pair): folds the tile partials of the tiles lying completely inside one of the pair's clouds
// and adds the rows of the (at most two per cloud) tiles that straddle a cloud boundary directly from the activations; the
// threads stride over the (tile, slot) entries and the edge elements (short dependent chains: the kernel is pure latency).
// mean_rstd [pair][G][2].
__global__ void __launch_bounds__(128) gn_seg_finalize_kernel(const double* __restrict__ partial, const float* __restrict__ x, int C,
                                                              int slots_total, int spg, int G, double eps, GnSeg seg,
                                                              float* __restrict__ mean_rstd) {
    __shared__ double red[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = blockIdx.x, p = blockIdx.y;
    const int cpg = C / G;
    const double2* part = reinterpret_cast<const double2*>(partial);
    double sa = 0.0, sb = 0.0;
    long long rows = 0;
    for (int c = p; c < seg.n_clouds; c += seg.n_pairs) {
        const int r0 = seg.start[c], r1 = seg.start[c + 1];
        rows += r1 - r0;
        int t0 = (r0 + 127) / 128, t1 = r1 / 128;          // full tiles [t0, t1)
        if (t1 < t0) t1 = t0;                              // the cloud lies inside one tile: all rows direct
        const int n_full = (t1 - t0) * spg;                // (tile, slot-of-group) entries
        for (int i = threadIdx.x; i < n_full; i += 128) {
            const int t = t0 + i / spg, sl = i % spg;
            const double2 v = part[(long long)t * slots_total + (long long)g * spg + sl];
            sa += v.x;
            sb += v.y;
        }
        const int e0 = min(r1, t0 * 128);                  // rows [r0, e0) and [b1, r1) are in straddling tiles
        const int b1 = min(r1, max(e0, t1 * 128));
        const int n_edge = (e0 - r0) + (r1 - b1);
        for (int i = threadIdx.x; i < n_edge * cpg; i += 128) {
            const int ri = i / cpg, j = i % cpg;
            const int r = ri < e0 - r0 ? r0 + ri : b1 + (ri - (e0 - r0));
            const double v = (double)x[(long long)r * C + g * cpg + j];
            sa += v;
            sb += v * v;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sa += __shfl_xor_sync(0xffffffffu, sa, o);
        sb += __shfl_xor_sync(0xffffffffu, sb, o);
    }
    if (lane == 0) { red[2 * warp] = sa; red[2 * warp + 1] = sb; }
    __syncthreads();
    if (threadIdx.x == 0) {
        sa = (red[0] + red[2]) + (red[4] + red[6]);
        sb = (red[1] + red[3]) + (red[5] + red[7]);
        const double count = (double)cpg * (double)rows;
        const double mean = sa / count;
        double var = sb / count - mean * mean;
        if (var < 0.0) var = 0.0;
        mean_rstd[((long long)p * G + g) * 2] = (float)mean;
        mean_rstd[((long long)p * G + g) * 2 + 1] = (float)(1.0 / sqrt(var + eps));
    }
}

// y = leaky((x - mean) * rstd * gamma + beta + residual) with the statistics of the row's pair.  One CTA normalises GN_RPB
// consecutive rows: they lie in at most two clouds unless a cloud is shorter than GN_RPB rows, so the per-channel scale / shift
// of the first two clouds of the block are tabulated once in shared memory (mean and rstd expanded per channel: no group
// arithmetic and no statistics loads per element, same expression as the per-element path); rows of a third cloud (tiny
// clouds only) take the per-element path.
constexpr int GN_RPB = 32;
__global__ void __launch_bounds__(256) gn_seg_apply_kernel(const float* __restrict__ x, const float* __restrict__ mean_rstd,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           const float* __restrict__ residual, float* __restrict__ y, int n_rows,
                                                           int C, int cpg, int G, int leaky, float slope, GnSeg seg) {
    extern __shared__ float gn_tab[];             // [2 clouds][mean | rstd][C]
    __shared__ int starts[GEOB_MAX_CLOUDS + 1];
    for (int i = threadIdx.x; i <= seg.n_clouds; i += blockDim.x) starts[i] = seg.start[i];
    __syncthreads();
    const int r0 = blockIdx.x * GN_RPB, r1 = min(n_rows, r0 + GN_RPB);
    int c0 = 0, hi = seg.n_clouds;                // cloud of the block's first row
    while (hi - c0 > 1) {
        const int mid = (c0 + hi) >> 1;
        if (starts[mid] <= r0) c0 = mid; else hi = mid;
    }
    for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
        const int t = i / C, c = i % C;
        const int cl = min(c0 + t, seg.n_clouds - 1);
        const float* mr = mean_rstd + (long long)(cl % seg.n_pairs) * 2 * G + 2 * (c / cpg);
        gn_tab[(2 * t) * C + c] = mr[0];
        gn_tab[(2 * t + 1) * C + c] = mr[1];
    }
    __syncthreads();
    const int b0 = starts[c0 + 1];                                        // rows < b0 use table 0
    const int b1 = (c0 + 2 <= seg.n_clouds) ? starts[c0 + 2] : n_rows;    // rows in [b0, b1) use table 1
    const int C4 = C >> 2;
    const long long base4 = (long long)r0 * C4;
    const int total4 = (r1 - r0) * C4;
    for (int i = threadIdx.x; i < total4; i += blockDim.x) {
        const int row = r0 + i / C4, c = (i % C4) * 4;
        const float4 v = reinterpret_cast<const float4*>(x)[base4 + i];
        float4 rv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (residual != nullptr) rv = reinterpret_cast<const float4*>(residual)[base4 + i];
        float in[4] = {v.x, v.y, v.z, v.w}, o[4];
        const float rs[4] = {rv.x, rv.y, rv.z, rv.w};
        if (row < b1) {
            const float* ta = gn_tab + (row < b0 ? 0 : 2 * C) + c;
            const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma + c)), bt = __ldg(reinterpret_cast<const float4*>(beta + c));
            const float ga[4] = {gm.x, gm.y, gm.z, gm.w}, ba[4] = {bt.x, bt.y, bt.z, bt.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) o[u] = (in[u] - ta[u]) * ta[C + u] * ga[u] + ba[u] + rs[u];
        } else {                                   // third cloud inside one block: clouds shorter than GN_RPB rows
            int lo = c0, hh = seg.n_clouds;
            while (hh - lo > 1) {
                const int mid = (lo + hh) >> 1;
                if (starts[mid] <= row) lo = mid; else hh = mid;
            }
            const float* mr = mean_rstd + (long long)(lo % seg.n_pairs) * 2 * G;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int g = (c + u) / cpg;
                o[u] = (in[u] - mr[2 * g]) * mr[2 * g + 1] * gamma[c + u] + beta[c + u] + rs[u];
            }
        }
        if (leaky) {
#pragma unroll
            for (int u = 0; u < 4; ++u) o[u] = o[u] > 0.f ? o[u] : o[u] * slope;
        }
        reinterpret_cast<float4*>(y)[base4 + i] = make_float4(o[0], o[1], o[2], o[3]);
    }
}

// One warp pools one output row: the row's neighbour indices are fetched once (lane h holds index h, broadcast by shuffle),
// channels are walked as float4 (coalesced 512-byte segments of a neighbour row), four neighbour rows in flight.
__device__ __forceinline__ void maxpool_row(const float* __restrict__ x, const long long* __restrict__ nb, int W, int Ns, int C,
                                            float* __restrict__ yrow, int lane) {
    constexpr int NI = 5;                           // rows of up to 160 neighbours keep their indices in registers
    if ((C & 3) == 0 && W <= 32 * NI) {
        int idx_l[NI];
#pragma unroll
        for (int i = 0; i < NI; ++i) idx_l[i] = (lane + 32 * i < W) ? (int)min(nb[lane + 32 * i], (long long)Ns) : Ns;
        const int C4 = C >> 2;
        for (int c0 = 0; c0 < C4; c0 += 32) {       // warp-uniform trip count: every lane takes part in the shuffles
            const int c4 = c0 + lane;
            const bool active = c4 < C4;
            float4 best = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
            for (int h0 = 0; h0 < W; h0 += 4) {
                float4 v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int h = h0 + u;
                    int id = Ns;
#pragma unroll
                    for (int i = 0; i < NI; ++i) {
                        const int t = __shfl_sync(0xffffffffu, idx_l[i], h & 31);
                        if ((h >> 5) == i) id = t;
                    }
                    v[u] = (active && h < W && id < Ns) ? __ldg(reinterpret_cast<const float4*>(x + (long long)id * C) + c4)
                                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                    if (h >= W) v[u] = best;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    best.x = fmaxf(best.x, v[u].x); best.y = fmaxf(best.y, v[u].y);
                    best.z = fmaxf(best.z, v[u].z); best.w = fmaxf(best.w, v[u].w);
                }
            }
            if (active) reinterpret_cast<float4*>(yrow)[c4] = best;
        }
        return;
    }
    for (int c = lane; c < C; c += 32) {
        float best = -INFINITY;
        for (int h = 0; h < W; ++h) {
            const long long idx = nb[h];
            const float v = (idx < Ns) ? x[idx * C + c] : 0.f;
            best = fmaxf(best, v);
        }
        yrow[c] = best;
    }
}

// Batched maxpool: the reference cuts a neighbour table to min(limit, max neighbour count OF THE PAIR) columns
// (radius_search.py:25-26 on the pair's own collate), and a row whose count equals that width has no shadow entry in its max.
// A batched table is as wide as the widest pair needs, so the columns past a pair's own width must not exist for its rows:
// cloud_max[c] = max neighbour count over the query rows of cloud c (geob200_cloud_max_count); pair width =
// min(H, max(cloud_max[p], cloud_max[B + p])).
__global__ void __launch_bounds__(256) maxpool_seg_kernel(const float* __restrict__ x, const long long* __restrict__ nbr, int H,
                                                          int Ns, int M, int C, float* __restrict__ y, GnSeg seg,
                                                          const int* __restrict__ cloud_max) {
    __shared__ int starts[GEOB_MAX_CLOUDS + 1];
    __shared__ int width[GEOB_MAX_CLOUDS];
    for (int i = threadIdx.x; i <= seg.n_clouds; i += blockDim.x) starts[i] = seg.start[i];
    for (int i = threadIdx.x; i < seg.n_clouds; i += blockDim.x) {
        const int p = i % seg.n_pairs;
        int w = 0;
        for (int c = p; c < seg.n_clouds; c += seg.n_pairs) w = max(w, cloud_max[c]);
        width[i] = min(H, w);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (m >= M) return;
    int lo = 0, hi = seg.n_clouds;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (starts[mid] <= m) lo = mid; else hi = mid;
    }
    const int W = width[lo];
    maxpool_row(x, nbr + (long long)m * H, W, Ns, C, y + (long long)m * C, lane);
}

// cloud_max[c] = max over the rows of cloud c of the number of real (non-sentinel) entries of a neighbour table row
__global__ void __launch_bounds__(256) cloud_max_count_kernel(const long long* __restrict__ nbr, int H, int Ns, GnSeg seg,
                                                              int* __restrict__ cloud_max) {
    __shared__ int red[8];
    const int c = blockIdx.x;
    const int r0 = seg.start[c], r1 = seg.start[c + 1];
    int best = 0;
    for (int m = r0 + (int)threadIdx.x; m < r1; m += blockDim.x) {
        // real indices come first: binary search for the first sentinel of the row
        int lo = 0, hi = H;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (nbr[(long long)m * H + mid] < Ns) lo = mid + 1; else hi = mid;
        }
        best = max(best, lo);
    }
    for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) best = max(best, red[w]);
        cloud_max[c] = best;
    }
}

// max over neighbour rows (shadow row = zeros), functional.py:54-67.  One warp per output row.
__global__ void __launch_bounds__(256) maxpool_kernel(const float* __restrict__ x, const long long* __restrict__ nbr, int H,
                                                      int Ns, int M, int C, float* __restrict__ y) {
    const int lane = threadIdx.x & 31;
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (m >= M) return;
    if ((C & 3) == 0 && H <= 160) {
        maxpool_row(x, nbr + (long long)m * H, H, Ns, C, y + (long long)m * C, lane);
        return;
    }
    for (int c = lane; c < C; c += 32) {
        float best = -INFINITY;
        for (int h = 0; h < H; ++h) {
            const long long idx = nbr[(long long)m * H + h];
            const float v = (idx < Ns) ? x[idx * C + c] : 0.f;
            best = fmaxf(best, v);
        }
        y[(long long)m * C + c] = best;
    }
}

// y[m] = [ x_pad[up[m][0]] | skip[m] ]   (functional.py:6-22 followed by torch.cat in backbone.py)
__global__ void __launch_bounds__(256) upsample_concat_kernel(const float* __restrict__ x, const long long* __restrict__ up,
                                                              int up_stride, int Ns, const float* __restrict__ skip, int M,
                                                              int C1, int C2, float* __restrict__ y) {
    const int lane = threadIdx.x & 31;
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (m >= M) return;
    const long long idx = up[(long long)m * up_stride];
    float* yr = y + (long long)m * (C1 + C2);
    for (int c = lane; c < C1; c += 32) yr[c] = (idx < Ns) ? x[idx * C1 + c] : 0.f;
    if (skip != nullptr)
        for (int c = lane; c < C2; c += 32) yr[C1 + c] = skip[(long long)m * C2 + c];
}

}  // namespace geob200

using namespace geob200;

namespace geob200 {
int linear_tc(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* bias, const float* row_scale, float* y, int64_t ldy,
              int64_t m, int64_t n, int64_t k, int relu, cudaStream_t st, const GnFuse* gn = nullptr);   // linear_tc.cu
static int g_linear_mode = 1;   // 1 = tcgen05 3xTF32 where the shape allows, 0 = fp32 CUDA cores only
}

extern "C" {

void geob200_set_linear_mode(int mode) { g_linear_mode = mode; }

size_t geob200_kpconv_workspace_bytes(int64_t n_support) { return (size_t)n_support + 256; }

// Tensor-core KPConv: gather stage + 3xTF32 GEMM.  weights_t = weights viewed as (15*c_in, c_out), transposed to (c_out, 15*c_in).
// workspace: n_support bytes (positivity flags) + n_query floats (row scales) + n_query*15*c_in floats (gathered features).
size_t geob200_kpconv_tc_workspace_bytes(int64_t n_query, int64_t n_support, int64_t c_in) {
    return align_up((size_t)n_support, 256) + align_up((size_t)n_query * 4, 256) + (size_t)n_query * KP * (size_t)c_in * 4 + 1024;
}

int geob200_kpconv_tc(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors, int64_t n_query,
                      int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel, const float* weights_t,
                      const float* bias, int64_t c_in, int64_t c_out, float sigma, float* out, void* workspace, size_t workspace_bytes,
                      void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GEOB_REQUIRE(n_kernel == KP, "kpconv_tc: kernel_size %lld unsupported", (long long)n_kernel);
    GEOB_REQUIRE(n_query > 0 && n_support > 0 && n_neighbors > 0, "kpconv_tc: empty input");
    GEOB_REQUIRE(c_in % 32 == 0 && c_out % 16 == 0 && c_out >= 32 && (c_out <= 128 || c_out % 128 == 0) && n_query >= 64,
                 "kpconv_tc: unsupported shape (%lld -> %lld, %lld queries)", (long long)c_in, (long long)c_out, (long long)n_query);
    GEOB_REQUIRE(workspace_bytes >= geob200_kpconv_tc_workspace_bytes(n_query, n_support, c_in), "kpconv_tc: workspace too small");
    Arena ar(workspace, workspace_bytes);
    unsigned char* pos = ar.take<unsigned char>(n_support);
    float* inv_count = ar.take<float>(n_query);
    float* wf = ar.take<float>((size_t)n_query * KP * c_in);
    row_positive_kernel<<<(unsigned)((n_support + 7) / 8), 256, 0, st>>>(s_feats, (int)n_support, (int)c_in, pos);
    launch_kpconv_gather(s_feats, pos, q_points, s_points, (const long long*)neighbors, (int)n_neighbors, kernel_points, sigma,
                         (int)n_support, (int)n_query, (int)c_in, wf, inv_count, st);
    GEOB_CHECK_LAUNCH();
    count_launches(2);
    const int rc = linear_tc(wf, KP * c_in, weights_t, KP * c_in, bias, inv_count, out, c_out, n_query, c_out, KP * c_in, 0, st);
    GEOB_REQUIRE(rc == 0, "kpconv_tc: tensor-core GEMM rejected the shape");
    return 0;
}

int geob200_kpconv(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors,
                   int64_t n_query, int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel,
                   const float* weights, const float* bias, int64_t c_in, int64_t c_out, float sigma, float* out,
                   void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GEOB_REQUIRE(n_kernel == KP, "kpconv: kernel_size %lld unsupported (all shipped models use 15)", (long long)n_kernel);
    GEOB_REQUIRE(n_query > 0 && n_support > 0 && n_neighbors > 0, "kpconv: empty input");
    if (c_in == 1) {
        kpconv_c1_kernel<<<(unsigned)((n_query + 15) / 16), 256, 0, st>>>(s_feats, q_points, s_points, (const long long*)neighbors,
                                                                       (int)n_neighbors, kernel_points, weights, bias, sigma,
                                                                       (int)n_support, (int)n_query, (int)c_out, out);
        GEOB_CHECK_LAUNCH();
        count_launches(1);
        return 0;
    }
    GEOB_REQUIRE(c_in % 32 == 0 && c_out % 32 == 0 && c_out <= 512,
                 "kpconv: channel counts (%lld -> %lld) must be multiples of 32, c_out <= 512", (long long)c_in, (long long)c_out);
    GEOB_REQUIRE(workspace != nullptr && workspace_bytes >= geob200_kpconv_workspace_bytes(n_support), "kpconv: workspace too small");
    unsigned char* pos = (unsigned char*)workspace;
    row_positive_kernel<<<(unsigned)((n_support + 7) / 8), 256, 0, st>>>(s_feats, (int)n_support, (int)c_in, pos);
    const size_t smem = sizeof(float) * (TQ * KP * CC + 8 * 32 * KP_PAD + TQ + KP * 3 + 3) + sizeof(int) * 8 * 32;
    const unsigned qtiles = (unsigned)((n_query + TQ - 1) / TQ);
    // columns per CTA: full width unless the level has too few query tiles to fill the GPU; then split the columns over at
    // most 4 CTAs (each of them repeats the gather phase)
    int rc = (int)(c_out / 32);
    int split = 1;
    while (rc > 1 && split < 4 && (long long)qtiles * split < 2ll * num_sms()) { rc >>= 1; split <<= 1; }
    const dim3 grid(qtiles, (unsigned)split);
#define LAUNCH_KP(RCV)                                                                                              \
    {                                                                                                               \
        if (ensure_max_smem((const void*)kpconv_kernel<RCV>)) return -1;                                            \
        kpconv_kernel<RCV><<<grid, 256, smem, st>>>(s_feats, pos, q_points, s_points, (const long long*)neighbors,  \
                                                    (int)n_neighbors, kernel_points, weights, bias, sigma,         \
                                                    (int)n_support, (int)n_query, (int)c_in, (int)c_out, out);     \
    }
    switch (rc) {
        case 1: LAUNCH_KP(1) break;
        case 2: LAUNCH_KP(2) break;
        case 4: LAUNCH_KP(4) break;
        case 8: LAUNCH_KP(8) break;
        case 16: LAUNCH_KP(16) break;
        default: GEOB_REQUIRE(false, "kpconv: c_out %lld unsupported (32,64,128,256,512)", (long long)c_out);
    }
#undef LAUNCH_KP
    GEOB_CHECK_LAUNCH();
    count_launches(2);
    return 0;
}

int geob200_linear_batched(const float* x, int64_t ldx, int64_t stride_x, const float* weight, int64_t ldw, int64_t stride_w,
                           const float* bias, int64_t stride_b, float* y, int64_t ldy, int64_t stride_y, int64_t m, int64_t n,
                           int64_t k, int64_t batch, int relu, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    GEOB_REQUIRE(m > 0 && n > 0 && k > 0 && batch > 0, "linear: empty problem");
    if (batch == 1 && g_linear_mode == 1) {
        const int rc = linear_tc(x, ldx, weight, ldw, bias, nullptr, y, ldy, m, n, k, relu, st);
        if (rc <= 0) return rc;       // done (0) or hard error (<0); 1 = shape not handled -> fp32 kernel below
    }
    const unsigned z = (unsigned)batch;
    const long long c64 = ((n + 63) / 64) * ((m + 63) / 64) * batch, c6432 = ((n + 31) / 32) * ((m + 63) / 64) * batch;
    if (c64 >= 148) {
        dim3 grid((unsigned)((n + 63) / 64), (unsigned)((m + 63) / 64), z);
        linear_kernel<64, 64><<<grid, 256, 0, st>>>(x, (int)ldx, weight, (int)ldw, bias, y, (int)ldy, (int)m, (int)n, (int)k, relu,
                                                    stride_x, stride_w, stride_b, stride_y);
    } else if (c6432 >= 148) {
        dim3 grid((unsigned)((n + 31) / 32), (unsigned)((m + 63) / 64), z);
        linear_kernel<64, 32><<<grid, 256, 0, st>>>(x, (int)ldx, weight, (int)ldw, bias, y, (int)ldy, (int)m, (int)n, (int)k, relu,
                                                    stride_x, stride_w, stride_b, stride_y);
    } else {
        dim3 grid((unsigned)((n + 31) / 32), (unsigned)((m + 31) / 32), z);
        linear_kernel<32, 32><<<grid, 256, 0, st>>>(x, (int)ldx, weight, (int)ldw, bias, y, (int)ldy, (int)m, (int)n, (int)k, relu,
                                                    stride_x, stride_w, stride_b, stride_y);
    }
    GEOB_CHECK_LAUNCH();
    count_launches(1);
    return 0;
}

int geob200_linear(const float* x, int64_t ldx, const float* weight, const float* bias, float* y, int64_t ldy, int64_t m,
                   int64_t n, int64_t k, int relu, void* stream) {
    return geob200_linear_batched(x, ldx, 0, weight, k, 0, bias, 0, y, ldy, 0, m, n, k, 1, relu, stream);
}

}  // extern "C"

namespace geob200 {
// Channels per statistics slot: the widest divisor of the group width up to 32.  For the group widths the GEMM epilogue fuses
// (divisors and multiples of 32) this is the epilogue's min(cpg, 32), so both producers write the same [tile][slot][2] layout.
static int gn_slot_width(int64_t cpg) {
    int w = cpg < 32 ? (int)cpg : 32;
    while (cpg % w != 0) --w;
    return w;
}
constexpr int GN_MAX_CHANNELS = 8192;   // gn_seg_apply_kernel tabulates 16 B per channel in shared memory (128 KB here)
struct GnWs { float* mean_rstd; double* partial; };
static GnWs gn_carve(void* workspace, size_t bytes, int64_t groups, int64_t n_pairs) {
    Arena ar(workspace, bytes);
    GnWs w;
    w.mean_rstd = ar.take<float>(2 * groups * n_pairs);
    w.partial = ar.take<double>(1);
    return w;
}
// Checked before the producer of the activations runs, so that a GroupNorm never fails at launch: workspace size, and the
// shared memory of the apply kernel (16 B per channel) and of the stand-alone statistics kernel (16 B per slot).
static int gn_prepare(int64_t n_rows, int64_t channels, int64_t groups, const GnSeg& seg, size_t workspace_bytes, const char* what) {
    GEOB_REQUIRE(channels <= GN_MAX_CHANNELS, "%s: at most %d channels", what, GN_MAX_CHANNELS);
    GEOB_REQUIRE(workspace_bytes >= geob200_group_norm_workspace_bytes(n_rows, channels, groups, seg.n_pairs),
                 "%s: workspace smaller than geob200_group_norm_workspace_bytes", what);
    if (16 * channels > 48 * 1024 &&
        (ensure_max_smem((const void*)gn_seg_apply_kernel) || ensure_max_smem((const void*)gn_tile_stats_kernel))) return -1;
    return 0;
}
// fold the tile partials per pair, then normalise every row with its pair's statistics
static void launch_gn_seg_apply(const float* x, const GnWs& w, const float* gamma, const float* beta, const float* residual, float* y,
                                int64_t n_rows, int64_t channels, int64_t groups, float eps, int leaky, float slope, const GnSeg& seg,
                                cudaStream_t st) {
    const int cpg = (int)(channels / groups);
    const int slot_width = gn_slot_width(cpg);
    gn_seg_finalize_kernel<<<dim3((unsigned)groups, (unsigned)seg.n_pairs), 128, 0, st>>>(
        w.partial, x, (int)channels, (int)(channels / slot_width), cpg / slot_width, (int)groups, (double)eps, seg, w.mean_rstd);
    gn_seg_apply_kernel<<<(unsigned)((n_rows + GN_RPB - 1) / GN_RPB), 256, sizeof(float) * 4 * channels, st>>>(
        x, w.mean_rstd, gamma, beta, residual, y, (int)n_rows, (int)channels, cpg, (int)groups, leaky, slope, seg);
    count_launches(2);
}
static void launch_gn_tile_stats(const float* x, const GnWs& w, int64_t n_rows, int64_t channels, int64_t groups, cudaStream_t st) {
    const int slot_width = gn_slot_width(channels / groups);
    gn_tile_stats_kernel<<<(unsigned)((n_rows + 127) / 128), 256, sizeof(double) * 2 * (channels / slot_width), st>>>(
        x, (int)n_rows, (int)channels, slot_width, w.partial);
    count_launches(1);
}
}  // namespace geob200

extern "C" {

// mean / rstd per (pair, group), then the per-128-row-tile statistics partials
size_t geob200_group_norm_workspace_bytes(int64_t n_rows, int64_t channels, int64_t groups, int64_t n_pairs) {
    if (n_rows <= 0 || channels <= 0 || groups <= 0 || channels % groups != 0 || n_pairs < 1) return 0;
    const size_t tiles = (size_t)((n_rows + 127) / 128), slots = (size_t)(channels / geob200::gn_slot_width(channels / groups));
    return align_up((size_t)(2 * groups * n_pairs) * sizeof(float), 256) + tiles * slots * 2 * sizeof(double);
}

int geob200_group_norm(const float* x, int64_t n_rows, int64_t channels, int64_t groups, const float* gamma,
                       const float* beta, float eps, const float* residual, int leaky, float slope, float* y,
                       void* workspace, size_t workspace_bytes, void* stream) {
    return geob200::group_norm_impl(x, n_rows, channels, groups, gamma, beta, eps, residual, leaky, slope, y, workspace, workspace_bytes,
                                    stream, geob200::gn_one_segment(n_rows));
}
}  // extern "C"

namespace geob200 {
int group_norm_impl(const float* x, int64_t n_rows, int64_t channels, int64_t groups, const float* gamma, const float* beta, float eps,
                    const float* residual, int leaky, float slope, float* y, void* workspace, size_t workspace_bytes, void* stream,
                    const GnSeg& seg) {
    cudaStream_t st = (cudaStream_t)stream;
    GEOB_REQUIRE(n_rows > 0 && channels > 0 && groups > 0 && channels % groups == 0, "group_norm: bad shape");
    GEOB_REQUIRE(channels % 4 == 0, "group_norm: channels must be a multiple of 4");
    if (int rc = gn_prepare(n_rows, channels, groups, seg, workspace_bytes, "group_norm")) return rc;
    const GnWs w = gn_carve(workspace, workspace_bytes, groups, seg.n_pairs);
    launch_gn_tile_stats(x, w, n_rows, channels, groups, st);
    launch_gn_seg_apply(x, w, gamma, beta, residual, y, n_rows, channels, groups, eps, leaky, slope, seg, st);
    GEOB_CHECK_LAUNCH();
    return 0;
}
}  // namespace geob200

extern "C" {

int geob200_maxpool(const float* x, const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors,
                    int64_t channels, float* y, void* stream) {
    maxpool_kernel<<<(unsigned)((n_query + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, (const long long*)neighbors, (int)n_neighbors,
                                                                                  (int)n_support, (int)n_query, (int)channels, y);
    GEOB_CHECK_LAUNCH();
    count_launches(1);
    return 0;
}

int geob200_upsample_concat(const float* x, const int64_t* up_indices, int64_t up_stride, int64_t n_support,
                            const float* skip, int64_t n_query, int64_t c1, int64_t c2, float* y, void* stream) {
    upsample_concat_kernel<<<(unsigned)((n_query + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
        x, (const long long*)up_indices, (int)up_stride, (int)n_support, skip, (int)n_query, (int)c1, (int)c2, y);
    GEOB_CHECK_LAUNCH();
    count_launches(1);
    return 0;
}

// Linear -> GroupNorm (+ residual) (+ LeakyReLU): UnaryBlock / the unary parts of ResidualBlock (modules.py:33-104,150-225).
// On the tensor-core path the GroupNorm statistics come out of the GEMM epilogue (no pass over the activations for them).
// pre_norm (m, n) receives the Linear output, y (m, n) the normalised result.
int geob200_linear_group_norm(const float* x, int64_t ldx, const float* weight, const float* bias, int64_t m, int64_t n, int64_t k,
                              int64_t groups, const float* gamma, const float* beta, float eps, const float* residual, int leaky,
                              float slope, float* pre_norm, float* y, void* workspace, size_t workspace_bytes, void* stream) {
    return geob200::linear_group_norm_impl(x, ldx, weight, bias, m, n, k, groups, gamma, beta, eps, residual, leaky, slope, pre_norm, y,
                                           workspace, workspace_bytes, stream, geob200::gn_one_segment(m));
}
}  // extern "C"

namespace geob200 {
int linear_group_norm_impl(const float* x, int64_t ldx, const float* weight, const float* bias, int64_t m, int64_t n, int64_t k,
                           int64_t groups, const float* gamma, const float* beta, float eps, const float* residual, int leaky,
                           float slope, float* pre_norm, float* y, void* workspace, size_t workspace_bytes, void* stream,
                           const GnSeg& seg) {
    cudaStream_t st = (cudaStream_t)stream;
    GEOB_REQUIRE(m > 0 && n > 0 && k > 0 && groups > 0 && n % groups == 0 && n % 4 == 0, "linear_group_norm: bad shape");
    if (int rc = gn_prepare(m, n, groups, seg, workspace_bytes, "linear_group_norm")) return rc;
    if (g_linear_mode == 1) {
        const GnWs w = gn_carve(workspace, workspace_bytes, groups, seg.n_pairs);
        GnFuse gn{(int)groups, 0, w.partial};
        const int rc = linear_tc(x, ldx, weight, k, bias, nullptr, pre_norm, n, m, n, k, 0, st, &gn);
        if (rc < 0) return rc;
        if (rc == 0) {
            launch_gn_seg_apply(pre_norm, w, gamma, beta, residual, y, m, n, groups, eps, leaky, slope, seg, st);
            GEOB_CHECK_LAUNCH();
            return 0;
        }
    }
    int rc = geob200_linear(x, ldx, weight, bias, pre_norm, n, m, n, k, 0, stream);
    if (rc != 0) return rc;
    return group_norm_impl(pre_norm, m, n, groups, gamma, beta, eps, residual, leaky, slope, y, workspace, workspace_bytes, stream, seg);
}
}  // namespace geob200

extern "C" {

// KPConv (gather + tcgen05 GEMM) -> GroupNorm (+ LeakyReLU): ConvBlock / the conv part of ResidualBlock (modules.py:107-147,205-207)
int geob200_kpconv_group_norm(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors,
                              int64_t n_query, int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel,
                              const float* weights_t, const float* bias, int64_t c_in, int64_t c_out, float sigma, int64_t groups,
                              const float* gamma, const float* beta, float eps, int leaky, float slope, float* pre_norm, float* y,
                              void* gn_workspace, size_t gn_workspace_bytes, void* workspace, size_t workspace_bytes, void* stream) {
    return geob200::kpconv_group_norm_impl(s_feats, q_points, s_points, neighbors, n_query, n_support, n_neighbors, kernel_points, n_kernel,
                                           weights_t, bias, c_in, c_out, sigma, groups, gamma, beta, eps, leaky, slope, pre_norm, y,
                                           gn_workspace, gn_workspace_bytes, workspace, workspace_bytes, stream,
                                           geob200::gn_one_segment(n_query));
}
}  // extern "C"

namespace geob200 {
int kpconv_group_norm_impl(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors,
                           int64_t n_query, int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel,
                           const float* weights_t, const float* bias, int64_t c_in, int64_t c_out, float sigma, int64_t groups,
                           const float* gamma, const float* beta, float eps, int leaky, float slope, float* pre_norm, float* y,
                           void* gn_workspace, size_t gn_workspace_bytes, void* workspace, size_t workspace_bytes, void* stream,
                           const GnSeg& seg) {
    cudaStream_t st = (cudaStream_t)stream;
    GEOB_REQUIRE(n_kernel == KP, "kpconv_group_norm: kernel_size %lld unsupported", (long long)n_kernel);
    GEOB_REQUIRE(n_query > 0 && n_support > 0 && n_neighbors > 0, "kpconv_group_norm: empty input");
    GEOB_REQUIRE(c_in % 32 == 0 && c_out % 16 == 0 && c_out >= 32 && (c_out <= 128 || c_out % 128 == 0) && n_query >= 64,
                 "kpconv_group_norm: unsupported shape (%lld -> %lld, %lld queries)", (long long)c_in, (long long)c_out,
                 (long long)n_query);
    GEOB_REQUIRE(groups > 0 && c_out % groups == 0, "kpconv_group_norm: bad group count");
    if (int rc = gn_prepare(n_query, c_out, groups, seg, gn_workspace_bytes, "kpconv_group_norm")) return rc;
    GEOB_REQUIRE(workspace_bytes >= geob200_kpconv_tc_workspace_bytes(n_query, n_support, c_in), "kpconv_group_norm: workspace too small");
    Arena ar(workspace, workspace_bytes);
    unsigned char* pos = ar.take<unsigned char>(n_support);
    float* inv_count = ar.take<float>(n_query);
    float* wf = ar.take<float>((size_t)n_query * KP * c_in);
    row_positive_kernel<<<(unsigned)((n_support + 7) / 8), 256, 0, st>>>(s_feats, (int)n_support, (int)c_in, pos);
    launch_kpconv_gather(s_feats, pos, q_points, s_points, (const long long*)neighbors, (int)n_neighbors, kernel_points, sigma,
                         (int)n_support, (int)n_query, (int)c_in, wf, inv_count, st);
    GEOB_CHECK_LAUNCH();
    count_launches(2);
    const GnWs w = gn_carve(gn_workspace, gn_workspace_bytes, groups, seg.n_pairs);
    GnFuse gn{(int)groups, 0, w.partial};
    int rc = linear_tc(wf, KP * c_in, weights_t, KP * c_in, bias, inv_count, pre_norm, c_out, n_query, c_out, KP * c_in, 0, st, &gn);
    if (rc < 0) return rc;
    if (rc == 0) {
        launch_gn_seg_apply(pre_norm, w, gamma, beta, nullptr, y, n_query, c_out, groups, eps, leaky, slope, seg, st);
        GEOB_CHECK_LAUNCH();
        return 0;
    }
    // group layout not expressible in the epilogue: plain GEMM, then the stand-alone statistics kernel
    rc = linear_tc(wf, KP * c_in, weights_t, KP * c_in, bias, inv_count, pre_norm, c_out, n_query, c_out, KP * c_in, 0, st);
    GEOB_REQUIRE(rc == 0, "kpconv_group_norm: tensor-core GEMM rejected the shape");
    return group_norm_impl(pre_norm, n_query, c_out, groups, gamma, beta, eps, nullptr, leaky, slope, y, gn_workspace, gn_workspace_bytes,
                           stream, seg);
}
}  // namespace geob200

namespace geob200 {
static int make_seg(GnSeg* g, int64_t n_pairs, const int64_t* cloud_rows_h, int64_t n_rows) {
    GEOB_REQUIRE(n_pairs >= 1 && 2 * n_pairs <= GEOB_MAX_CLOUDS && cloud_rows_h != nullptr, "group_norm: 1 <= pairs per batch <= %d", GEOB_MAX_CLOUDS / 2);
    g->n_pairs = (int)n_pairs; g->n_clouds = (int)(2 * n_pairs); g->start[0] = 0;
    for (int c = 0; c < g->n_clouds; ++c) g->start[c + 1] = g->start[c] + (int)cloud_rows_h[c];
    GEOB_REQUIRE(g->start[g->n_clouds] == n_rows, "group_norm: cloud rows do not add up to n_rows");
    return 0;
}
// GroupNorm statistics of a batch: a single pair is one segment, so its result does not depend on the entry point
static int make_gn_seg(GnSeg* g, int64_t n_pairs, const int64_t* cloud_rows_h, int64_t n_rows) {
    if (make_seg(g, n_pairs, cloud_rows_h, n_rows)) return -2;
    if (n_pairs == 1) *g = gn_one_segment(n_rows);
    return 0;
}
}  // namespace geob200

extern "C" {

int geob200_group_norm_batched(const float* x, int64_t n_rows, int64_t channels, int64_t groups, const float* gamma, const float* beta,
                               float eps, const float* residual, int leaky, float slope, float* y, void* workspace, size_t workspace_bytes,
                               void* stream, int64_t n_pairs, const int64_t* cloud_rows_h) {
    geob200::GnSeg seg;
    if (geob200::make_gn_seg(&seg, n_pairs, cloud_rows_h, n_rows)) return -2;
    return geob200::group_norm_impl(x, n_rows, channels, groups, gamma, beta, eps, residual, leaky, slope, y, workspace, workspace_bytes,
                                    stream, seg);
}

int geob200_linear_group_norm_batched(const float* x, int64_t ldx, const float* weight, const float* bias, int64_t m, int64_t n, int64_t k,
                                      int64_t groups, const float* gamma, const float* beta, float eps, const float* residual, int leaky,
                                      float slope, float* pre_norm, float* y, void* workspace, size_t workspace_bytes, void* stream,
                                      int64_t n_pairs, const int64_t* cloud_rows_h) {
    geob200::GnSeg seg;
    if (geob200::make_gn_seg(&seg, n_pairs, cloud_rows_h, m)) return -2;
    return geob200::linear_group_norm_impl(x, ldx, weight, bias, m, n, k, groups, gamma, beta, eps, residual, leaky, slope, pre_norm, y,
                                           workspace, workspace_bytes, stream, seg);
}

/* cloud_max[c] (device int32[2 * n_pairs]) = widest row (number of real neighbours) among the query rows of cloud c */
int geob200_cloud_max_count(const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors, int64_t n_pairs,
                            const int64_t* cloud_rows_h, int32_t* cloud_max, void* stream) {
    geob200::GnSeg seg;
    if (geob200::make_seg(&seg, n_pairs, cloud_rows_h, n_query)) return -2;
    geob200::cloud_max_count_kernel<<<seg.n_clouds, 256, 0, (cudaStream_t)stream>>>((const long long*)neighbors, (int)n_neighbors,
                                                                                   (int)n_support, seg, cloud_max);
    GEOB_CHECK_LAUNCH();
    geob200::count_launches(1);
    return 0;
}

int geob200_maxpool_batched(const float* x, const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors,
                            int64_t channels, float* y, int64_t n_pairs, const int64_t* cloud_rows_h, const int32_t* cloud_max,
                            void* stream) {
    geob200::GnSeg seg;
    if (geob200::make_seg(&seg, n_pairs, cloud_rows_h, n_query)) return -2;
    return geob200::maxpool_seg(x, neighbors, n_query, n_support, n_neighbors, channels, y, &seg, cloud_max, stream);
}

}  // extern "C"

namespace geob200 {
int maxpool_seg(const float* x, const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors, int64_t channels,
                float* y, const GnSeg* seg, const int* cloud_max, void* stream) {
    maxpool_seg_kernel<<<(unsigned)((n_query + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, (const long long*)neighbors, (int)n_neighbors,
                                                                                      (int)n_support, (int)n_query, (int)channels, y, *seg,
                                                                                      cloud_max);
    GEOB_CHECK_LAUNCH();
    count_launches(1);
    return 0;
}
}  // namespace geob200
