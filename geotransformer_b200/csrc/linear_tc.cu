// nn.Linear on the 5th-gen tensor cores: Y[M,N] = X[M,K] . W[N,K]^T + b (optional ReLU), fp32 in / fp32 out.
//
// The reference's Linears are true fp32 (torch default allow_tf32=False), so the product is computed with the
// error-compensated 3xTF32 scheme: x = x_hi + x_lo, w = w_hi + w_lo (hi = top 19 bits), D += x_hi w_hi + x_hi w_lo +
// x_lo w_hi with fp32 accumulation in TMEM (~1e-6 relative, same as an fp32 FMA chain).
//
// One CTA per 128 x BN output tile (BN = min(N,128)), K in chunks of 32 floats (one 128-byte swizzle row):
//   warp 0      TMA producer : cp.async.bulk.tensor.2d (UTMALDG) of the raw X tile (128 x 32) and W tile (BN x 32) through
//                              SWIZZLE_128B tensor maps; out-of-bounds rows/columns are zero-filled by the TMA unit
//   warps 1-8   splitters    : in-place hi = tf32_rn(x), lo = x - hi into a second buffer (generic proxy ->
//                              fence.proxy.async), so the MMA sees exact tf32 operands
//   warp 9      MMA issuer   : tcgen05.mma.cta_group::1.kind::tf32 M128 N{BN} K8, 3 per K-step; tcgen05.commit frees the stage
//   warps 10-13 epilogue     : tcgen05.ld 32x32b, + bias, ReLU, direct row-segment stores (each thread owns one output row);
//                              optionally the GroupNorm statistics of the output (per-tile column sums through a transposing
//                              warp butterfly, written as per-tile partials in double)
#include <cuda.h>

#include <cstdlib>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "geob200.h"

namespace geob200 {
namespace ltc {

constexpr int BM = 128;
constexpr int KC = 32;
constexpr int TILE_A = BM * 128;       // 16 KB
constexpr int TILE_B = 128 * 128;      // 16 KB (BN <= 128 rows)
constexpr int STAGE = 2 * TILE_A + 2 * TILE_B;   // raw/hi + lo for both operands = 64 KB
constexpr int NSTAGE = 3;
constexpr int NSPLIT_WARPS = 8;                       // warps 1..8
constexpr int MMA_WARP = 1 + NSPLIT_WARPS;            // warp 9
constexpr int EPI_WARP0 = MMA_WARP + 1;               // warps 10..13 (warp & 3 covers the four TMEM lane quarters)
constexpr int NTHREADS = (EPI_WARP0 + 4) * 32;        // 448
// 193.25 KB + the 1 KB the system reserves per CTA fits the 196 KB shared-memory carve-out; anything larger forces the 228 KB
// configuration and costs ~8 us per launch in carve-out switches against the neighbouring kernels (measured)
constexpr int SMEM = NSTAGE * STAGE + 1024 + 256;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(addr), "r"(parity)
                     : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(dst)),
                 "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {   // K-major SWIZZLE_128B, SBO = 1024 B (see gse_tc.cu)
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- pieces shared by the one-CTA-per-tile kernel and the persistent kernel ---------------------------------------------------
// splitter: in-place hi = tf32_rn(x), lo = x - hi into the second buffer of each operand (element-wise, so the swizzled
// positions are irrelevant: same offset in the hi and lo buffers).  Two 16-byte vectors per thread and iteration: their
// shared-memory round trips overlap.  t = thread index among the NSPLIT_WARPS * 32 splitter threads.
__device__ __forceinline__ void split_stage(unsigned char* st, int BN, int t) {
    constexpr int NT = NSPLIT_WARPS * 32;
    const int nvec_a = TILE_A / 16, nvec_b = BN * 128 / 16;
    const int nvec = nvec_a + nvec_b;            // multiple of NT (BN is a multiple of 16)
    for (int v0 = t; v0 < nvec; v0 += 2 * NT) {
        const int v1 = v0 + NT;
        unsigned char* p0 = (v0 < nvec_a) ? (st + v0 * 16) : (st + 2 * TILE_A + (v0 - nvec_a) * 16);
        unsigned char* l0 = p0 + ((v0 < nvec_a) ? TILE_A : TILE_B);
        const bool two = v1 < nvec;
        unsigned char* p1 = !two ? p0 : (v1 < nvec_a) ? (st + v1 * 16) : (st + 2 * TILE_A + (v1 - nvec_a) * 16);
        unsigned char* l1 = p1 + ((v1 < nvec_a) ? TILE_A : TILE_B);
        const float4 x0 = *reinterpret_cast<float4*>(p0);
        const float4 x1 = *reinterpret_cast<float4*>(p1);
        float4 h0, q0, h1, q1;
        h0.x = tf32_rn(x0.x); q0.x = x0.x - h0.x;     // round-to-nearest split: |lo| <= 2^-12 |x|, unbiased
        h0.y = tf32_rn(x0.y); q0.y = x0.y - h0.y;
        h0.z = tf32_rn(x0.z); q0.z = x0.z - h0.z;
        h0.w = tf32_rn(x0.w); q0.w = x0.w - h0.w;
        h1.x = tf32_rn(x1.x); q1.x = x1.x - h1.x;
        h1.y = tf32_rn(x1.y); q1.y = x1.y - h1.y;
        h1.z = tf32_rn(x1.z); q1.z = x1.z - h1.z;
        h1.w = tf32_rn(x1.w); q1.w = x1.w - h1.w;
        *reinterpret_cast<float4*>(p0) = h0;
        *reinterpret_cast<float4*>(l0) = q0;
        if (two) {
            *reinterpret_cast<float4*>(p1) = h1;
            *reinterpret_cast<float4*>(l1) = q1;
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// the 12 MMAs of one 32-float K chunk: main products and the (2^-11 smaller) correction products go to separate accumulators
// (columns [acc, acc+128) and [acc+128, acc+256)): the fp32 accumulation in the tensor core truncates, so keeping the number of
// additions into the main accumulator at K/8 instead of 3K/8 cuts the systematic error by 3x
__device__ __forceinline__ void issue_chunk_mmas(uint32_t st, uint32_t acc, uint32_t idesc, bool first_chunk) {
    const uint64_t a_hi = make_desc(st), a_lo = make_desc(st + TILE_A);
    const uint64_t b_hi = make_desc(st + 2 * TILE_A), b_lo = make_desc(st + 2 * TILE_A + TILE_B);
#pragma unroll
    for (int kk = 0; kk < KC / 8; ++kk) {
        const uint64_t adv = (uint64_t)(kk * 2);
        const uint32_t first = (first_chunk && kk == 0) ? 0u : 1u;
        umma_tf32(acc, a_hi + adv, b_hi + adv, idesc, first);
        umma_tf32(acc + 128, a_hi + adv, b_lo + adv, idesc, first);
        umma_tf32(acc + 128, a_lo + adv, b_hi + adv, idesc, 1u);
    }
}

// 32 columns of both accumulators (main, corrections) of this thread's row
__device__ __forceinline__ void tmem_ld_pair(uint32_t taddr, uint32_t (&v)[32], uint32_t (&w2)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(w2[0]), "=r"(w2[1]), "=r"(w2[2]), "=r"(w2[3]), "=r"(w2[4]), "=r"(w2[5]), "=r"(w2[6]), "=r"(w2[7]), "=r"(w2[8]),
          "=r"(w2[9]), "=r"(w2[10]), "=r"(w2[11]), "=r"(w2[12]), "=r"(w2[13]), "=r"(w2[14]), "=r"(w2[15]), "=r"(w2[16]),
          "=r"(w2[17]), "=r"(w2[18]), "=r"(w2[19]), "=r"(w2[20]), "=r"(w2[21]), "=r"(w2[22]), "=r"(w2[23]), "=r"(w2[24]),
          "=r"(w2[25]), "=r"(w2[26]), "=r"(w2[27]), "=r"(w2[28]), "=r"(w2[29]), "=r"(w2[30]), "=r"(w2[31])
        : "r"(taddr + 128));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// epilogue of one 32-column chunk of this thread's row: (main + corrections) * row scale + bias (+ ReLU), direct row-segment
// store, and the GroupNorm column sums over the warp's 32 rows (rows past M and columns past N contribute nothing) through the
// transposing butterfly into gn_sm[q][slot]
__device__ __forceinline__ void finish_chunk(const uint32_t (&v)[32], const uint32_t (&w2)[32], float rs, const float* bias_s, int cc,
                                             int relu, bool row_ok, float* yr, int nvalid, const GnFuse& gn, float2* gn_sm, int q,
                                             int lane) {
    float o[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) {
        float t = (__uint_as_float(v[c]) + __uint_as_float(w2[c])) * rs + bias_s[cc + c];
        if (relu) t = fmaxf(t, 0.f);
        o[c] = t;
    }
    if (row_ok) {
        if (nvalid == 32 && ((reinterpret_cast<uintptr_t>(yr) & 15) == 0)) {
#pragma unroll
            for (int c = 0; c < 32; c += 4) *reinterpret_cast<float4*>(yr + c) = make_float4(o[c], o[c + 1], o[c + 2], o[c + 3]);
        } else {
#pragma unroll
            for (int c = 0; c < 32; ++c)
                if (c < nvalid) yr[c] = o[c];
        }
    }
    if (gn.groups > 0) {
        float s1[32], s2[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const float t = (row_ok && c < nvalid) ? o[c] : 0.f;
            s1[c] = t;
            s2[c] = t * t;
        }
        float a = warp_butterfly(s1, lane), b2 = warp_butterfly(s2, lane);
        for (int off = 1; off < gn.slot_width; off <<= 1) {
            a += __shfl_xor_sync(0xffffffffu, a, off);
            b2 += __shfl_xor_sync(0xffffffffu, b2, off);
        }
        if ((lane & (gn.slot_width - 1)) == 0) gn_sm[q * 128 + (cc + lane) / gn.slot_width] = make_float2(a, b2);
    }
}

// 4 epilogue warps -> per-tile partial in a fixed order; gn_seg_finalize (kpconv.cu) folds the tiles afterwards
// (no fence / last-CTA fold here: the CTA must not wait for its output stores to drain).  et = thread index among the 128 epilogue threads.
__device__ __forceinline__ void write_gn_partials(const GnFuse& gn, const float2* gn_sm, int et, int BN, int N, int n0, int tile_row) {
    const int slots_tile = BN / gn.slot_width, slots_total = N / gn.slot_width;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (et < slots_tile) {
        const float2 p0 = gn_sm[et], p1 = gn_sm[128 + et], p2 = gn_sm[256 + et], p3 = gn_sm[384 + et];
        double* dst = gn.partial + ((long long)tile_row * slots_total + n0 / gn.slot_width + et) * 2;
        dst[0] = ((double)p0.x + (double)p1.x) + ((double)p2.x + (double)p3.x);
        dst[1] = ((double)p0.y + (double)p1.y) + ((double)p2.y + (double)p3.y);
    }
}

__global__ void __launch_bounds__(NTHREADS, 1) linear_tc_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                const __grid_constant__ CUtensorMap map_w,
                                                                const float* __restrict__ bias, const float* __restrict__ row_scale,
                                                                float* __restrict__ Y, int ldy, int M, int N, int K, int BN, int relu,
                                                                GnFuse gn, float* __restrict__ splitk_out, int chunks_per_split) {
    extern __shared__ unsigned char smem_raw[];
    __shared__ float bias_s[128];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + NSTAGE * STAGE);
    uint64_t* raw_full = bars;                  // TMA landed
    uint64_t* split_full = bars + NSTAGE;       // hi/lo ready
    uint64_t* empty = bars + 2 * NSTAGE;        // MMAs done with the stage
    uint64_t* acc_full = bars + 3 * NSTAGE;
    uint32_t* tmem_slot = (uint32_t*)(acc_full + 1);
    float2* gn_sm = (float2*)smem;      // GroupNorm column sums [4 warps][128 slots]: stage 0 is idle once acc_full has fired
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int nk = (K + KC - 1) / KC;
    // split-K: CTA z accumulates K-chunks [kc0, kc1) and stores its raw partial tile; splitk_reduce_kernel finishes the job
    const int kc0 = blockIdx.z * chunks_per_split, kc1 = min(nk, kc0 + chunks_per_split);

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&split_full[s], NSPLIT_WARPS); mbar_init(&empty[s], 1); }
        mbar_init(acc_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int kc = kc0; kc < kc1; ++kc) {
                mbar_wait(&empty[s], ph ^ 1u);
                unsigned char* st = smem + s * STAGE;
                mbar_arrive_expect_tx(&raw_full[s], (uint32_t)(TILE_A + BN * 128));
                tma_load_2d(st, &map_x, kc * KC, m0, &raw_full[s]);
                tma_load_2d(st + 2 * TILE_A, &map_w, kc * KC, n0, &raw_full[s]);
                if (++s == NSTAGE) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp <= NSPLIT_WARPS) {
        const int t = threadIdx.x - 32;              // 0..NSPLIT_WARPS*32-1
        int s = 0;
        uint32_t ph = 0;
        for (int kc = kc0; kc < kc1; ++kc) {
            mbar_wait(&raw_full[s], ph);
            split_stage(smem + s * STAGE, BN, t);
            __syncwarp();
            if (lane == 0) mbar_arrive(&split_full[s]);
            if (++s == NSTAGE) { s = 0; ph ^= 1u; }
        }
    } else if (warp == MMA_WARP) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            int s = 0;
            uint32_t ph = 0;
            for (int kc = kc0; kc < kc1; ++kc) {
                mbar_wait(&split_full[s], ph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                issue_chunk_mmas(smem_u32(smem + s * STAGE), tmem_base, idesc, kc == kc0);
                umma_commit(&empty[s]);
                if (++s == NSTAGE) { s = 0; ph ^= 1u; }
            }
            umma_commit(acc_full);
        }
    } else {
        const int q = warp & 3;
        // the tile's bias row goes through shared memory once (loaded while the main loop runs): per-element global loads in
        // the epilogue are a chain of 32 dependent L2 round trips per chunk (~8 us per tile, measured)
        {
            const int et = threadIdx.x - EPI_WARP0 * 32;
            bias_s[et] = (bias != nullptr && n0 + et < N) ? __ldg(bias + n0 + et) : 0.f;
            asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        mbar_wait(acc_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int m = m0 + q * 32 + lane;
        const float rs = (row_scale != nullptr && m < M) ? row_scale[m] : 1.0f;   // KPConv: 1 / neighbour count
        for (int cc = 0; cc < BN; cc += 32) {
            uint32_t v[32], w2[32];
            tmem_ld_pair(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)cc, v, w2);
            const int nvalid = min(32, N - (n0 + cc));
            if (splitk_out != nullptr) {              // raw partial sums of this K-slice (N is a multiple of 16: float4-aligned)
                if (m < M) {
                    float* pr = splitk_out + ((long long)blockIdx.z * M + m) * N + n0 + cc;
#pragma unroll
                    for (int c = 0; c < 32; c += 4)
                        if (c < nvalid)
                            *reinterpret_cast<float4*>(pr + c) =
                                make_float4(__uint_as_float(v[c]) + __uint_as_float(w2[c]), __uint_as_float(v[c + 1]) + __uint_as_float(w2[c + 1]),
                                            __uint_as_float(v[c + 2]) + __uint_as_float(w2[c + 2]), __uint_as_float(v[c + 3]) + __uint_as_float(w2[c + 3]));
                }
                continue;
            }
            finish_chunk(v, w2, rs, bias_s, cc, relu, m < M, Y + (long long)m * ldy + n0 + cc, nvalid, gn, gn_sm, q, lane);
        }
        if (gn.groups > 0 && splitk_out == nullptr) write_gn_partials(gn, gn_sm, threadIdx.x - EPI_WARP0 * 32, BN, N, n0, blockIdx.y);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem_base) : "memory");
    }
}

// ---- persistent variant (multi-wave GEMMs) ----------------------------------------------------------------------------------
// One CTA per SM walks the output tiles t = blockIdx.x, blockIdx.x + gridDim.x, ...  The operand ring keeps running across
// tile boundaries and there are TWO accumulator sets in TMEM (2 x (main 128 + corrections 128) = 512 columns): while the four
// epilogue warps drain, normalise and store tile i, the producer / splitters / MMA issuer are already deep in the K loop of
// tile i + 1, so the per-tile fixed cost (first TMA round trip, TMEM drain, stores) is hidden instead of paid per CTA.
// 202.5 KB: 6 KB over the 196 KB carve-out the per-tile kernel stays under, i.e. this kernel runs in the 228 KB shared-memory
// configuration.  Accepted: it is only chosen for GEMMs of more than one wave of tiles (>= 0.1 ms each in batch mode), where a
// carve-out switch against a neighbouring kernel (~8 us, measured in round 1) is noise, and the GroupNorm / bias staging must
// survive across the tile loop next to the three operand stages.
constexpr int SMEM_PERSIST = SMEM + 4 * 128 * 8 + 512;      // + GroupNorm column sums [4][128] float2 + the bias row

__global__ void __launch_bounds__(NTHREADS, 1) linear_tc_persistent_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                           const __grid_constant__ CUtensorMap map_w,
                                                                           const float* __restrict__ bias,
                                                                           const float* __restrict__ row_scale, float* __restrict__ Y,
                                                                           int ldy, int M, int N, int K, int BN, int relu, GnFuse gn,
                                                                           int col_tiles, int num_tiles) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = (unsigned char*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(smem + NSTAGE * STAGE);
    uint64_t* raw_full = bars;                  // TMA landed
    uint64_t* split_full = bars + NSTAGE;       // hi/lo ready
    uint64_t* empty = bars + 2 * NSTAGE;        // MMAs done with the stage
    uint64_t* acc_full = bars + 3 * NSTAGE;     // [2] accumulator set complete
    uint64_t* acc_empty = acc_full + 2;         // [2] accumulator set drained by the epilogue
    uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);
    float2* gn_sm = (float2*)(smem + NSTAGE * STAGE + 256);
    float* bias_s = (float*)(smem + NSTAGE * STAGE + 256 + 4 * 128 * 8);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nk = (K + KC - 1) / KC;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&raw_full[s], 1); mbar_init(&split_full[s], NSPLIT_WARPS); mbar_init(&empty[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&acc_full[a], 1); mbar_init(&acc_empty[a], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_w) : "memory");
    }
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int s = 0;
            uint32_t ph = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
                const int m0 = (t / col_tiles) * BM, n0 = (t % col_tiles) * BN;
                for (int kc = 0; kc < nk; ++kc) {
                    mbar_wait(&empty[s], ph ^ 1u);
                    unsigned char* st = smem + s * STAGE;
                    mbar_arrive_expect_tx(&raw_full[s], (uint32_t)(TILE_A + BN * 128));
                    tma_load_2d(st, &map_x, kc * KC, m0, &raw_full[s]);
                    tma_load_2d(st + 2 * TILE_A, &map_w, kc * KC, n0, &raw_full[s]);
                    if (++s == NSTAGE) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp <= NSPLIT_WARPS) {
        const int tt = threadIdx.x - 32;
        int s = 0;
        uint32_t ph = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
            for (int kc = 0; kc < nk; ++kc) {
                mbar_wait(&raw_full[s], ph);
                split_stage(smem + s * STAGE, BN, tt);
                __syncwarp();
                if (lane == 0) mbar_arrive(&split_full[s]);
                if (++s == NSTAGE) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == MMA_WARP) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
            int s = 0;
            uint32_t ph = 0;
            int it = 0;
            for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
                const int set = it & 1;
                mbar_wait(&acc_empty[set], (((uint32_t)it >> 1) & 1u) ^ 1u);      // the epilogue has drained the previous use of this set
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t acc = tmem_base + (uint32_t)(set * 256);
                for (int kc = 0; kc < nk; ++kc) {
                    mbar_wait(&split_full[s], ph);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    issue_chunk_mmas(smem_u32(smem + s * STAGE), acc, idesc, kc == 0);
                    umma_commit(&empty[s]);
                    if (++s == NSTAGE) { s = 0; ph ^= 1u; }
                }
                umma_commit(&acc_full[set]);
            }
        }
    } else {
        const int q = warp & 3;
        const int et = threadIdx.x - EPI_WARP0 * 32;
        int it = 0;
        for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
            const int set = it & 1;
            const int ty = t / col_tiles;
            const int m0 = ty * BM, n0 = (t % col_tiles) * BN;
            asm volatile("bar.sync 1, 128;" ::: "memory");                          // previous tile's readers of bias_s / gn_sm are done
            bias_s[et] = (bias != nullptr && n0 + et < N) ? __ldg(bias + n0 + et) : 0.f;
            asm volatile("bar.sync 1, 128;" ::: "memory");
            mbar_wait(&acc_full[set], ((uint32_t)it >> 1) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const int m = m0 + q * 32 + lane;
            const float rs = (row_scale != nullptr && m < M) ? row_scale[m] : 1.0f;
            for (int cc = 0; cc < BN; cc += 32) {
                uint32_t v[32], w2[32];
                tmem_ld_pair(tmem_base + (uint32_t)(set * 256) + ((uint32_t)(q * 32) << 16) + (uint32_t)cc, v, w2);
                if (cc + 32 >= BN) {        // last chunk read: hand the accumulator set back before the stores and statistics
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[set]);
                }
                finish_chunk(v, w2, rs, bias_s, cc, relu, m < M, Y + (long long)m * ldy + n0 + cc, min(32, N - (n0 + cc)), gn, gn_sm, q, lane);
            }
            if (gn.groups > 0) write_gn_partials(gn, gn_sm, et, BN, N, n0, ty);
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == MMA_WARP) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// y[m][n] = (sum_z P[z][m][n]) * row_scale[m] + bias[n] (+ ReLU): the splits are added in a fixed order
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ P, int splits, long long MN, int N,
                                                            const float* __restrict__ bias, const float* __restrict__ row_scale,
                                                            float* __restrict__ Y, int ldy, int relu) {
    const long long i4 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i4 >= MN) return;
    float4 a = *reinterpret_cast<const float4*>(P + i4);
    for (int z = 1; z < splits; ++z) {
        const float4 b = *reinterpret_cast<const float4*>(P + (long long)z * MN + i4);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    const long long m = i4 / N;
    const int n = (int)(i4 % N);
    const float rs = row_scale != nullptr ? row_scale[m] : 1.0f;
    float o[4] = {a.x * rs, a.y * rs, a.z * rs, a.w * rs};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        if (bias != nullptr) o[u] += bias[n + u];
        if (relu) o[u] = fmaxf(o[u], 0.f);
    }
    float* y = Y + m * ldy + n;
    if ((reinterpret_cast<uintptr_t>(y) & 15) == 0) *reinterpret_cast<float4*>(y) = make_float4(o[0], o[1], o[2], o[3]);
    else { y[0] = o[0]; y[1] = o[1]; y[2] = o[2]; y[3] = o[3]; }
}

// cuTensorMapEncodeTiled is fetched through the runtime (cudaGetDriverEntryPoint) so that libgeob200.so does not link
// libcuda directly and still loads on a machine without a driver (the no-GPU ABI tests).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

static int encode_map(CUtensorMap* map, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
    EncodeTiledFn fn = encode_fn();
    if (fn == nullptr) { set_error("cuTensorMapEncodeTiled entry point not available"); return -1; }
    cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t gstride[1] = {(cuuint64_t)ld * sizeof(float)};
    cuuint32_t box[2] = {(cuuint32_t)KC, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return -1; }
    return 0;
}

}  // namespace ltc

// ---- optional per-launch profile (bench.py roofline): CUDA events around every linear_tc launch + its shape ----------------
struct ProfRec { cudaEvent_t a, b; long long m, n, k; };
static std::vector<ProfRec> g_prof;
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static bool g_splitk_on = true;
static bool g_persistent_on = true;    // persistent tile loop for GEMMs of more than one wave of tiles (geob200_set_linear_persistent)

// ---- split-K scratch: one grow-only buffer per stream (like a BLAS workspace; freed with the process) ---------------------
struct SplitWs { void* ptr; size_t bytes; };
static std::vector<std::pair<cudaStream_t, SplitWs>> g_split_ws;
static std::mutex g_split_mu;
static float* splitk_scratch(cudaStream_t st, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_split_mu);
    for (auto& e : g_split_ws)
        if (e.first == st) {
            if (e.second.bytes >= bytes) return (float*)e.second.ptr;
            // stream-ordered free: earlier kernels on this stream may still read the old buffer
            cudaFreeAsync(e.second.ptr, st);
            e.second = {nullptr, 0};
            if (cudaMallocAsync(&e.second.ptr, bytes * 2, st) != cudaSuccess) return nullptr;
            e.second.bytes = bytes * 2;
            return (float*)e.second.ptr;
        }
    SplitWs w{nullptr, 0};
    const size_t cap = bytes * 2 > (16u << 20) ? bytes * 2 : (16u << 20);
    if (cudaMallocAsync(&w.ptr, cap, st) != cudaSuccess) return nullptr;
    w.bytes = cap;
    g_split_ws.push_back({st, w});
    return (float*)w.ptr;
}

// returns 1 when the shape/alignment is not handled by the tensor-core path (caller falls back to the fp32 kernel)
int linear_tc(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* bias, const float* row_scale, float* y, int64_t ldy,
              int64_t m, int64_t n, int64_t k, int relu, cudaStream_t st, const GnFuse* gn) {
    if (m < 64 || n < 32 || (n % 16) != 0 || (k % 4) != 0 || (ldx % 4) != 0 || (ldw % 4) != 0) return 1;
    if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(w) & 15)) return 1;
    if (n > 128 && (n % 128) != 0) return 1;
    const int BN = (int)(n >= 128 ? 128 : n);
    CUtensorMap mx, mw;
    if (ltc::encode_map(&mx, x, m, k, ldx, ltc::BM)) return -1;
    if (ltc::encode_map(&mw, w, n, k, ldw, BN)) return -1;
    if (ensure_max_smem((const void*)ltc::linear_tc_kernel)) return -1;
    dim3 grid((unsigned)(n / BN), (unsigned)((m + ltc::BM - 1) / ltc::BM));
    GnFuse g{};
    if (gn != nullptr) {
        g = *gn;
        const int64_t cpg = n / g.groups;
        // groups must tile the 32-column epilogue chunks: cpg in {1,2,4,...,32} or a multiple of 32 dividing the column tile
        if (g.groups <= 0 || n % g.groups != 0 || (cpg < 32 ? (32 % cpg) != 0 : (cpg % 32) != 0 || (BN % cpg) != 0) || relu) return 1;
        g.slot_width = (int)(cpg < 32 ? cpg : 32);
    }
    // split-K: a deep K loop on a handful of tiles leaves most SMs idle and is pure latency (1.4 us per 32-wide chunk): give
    // every K-slice of >= 8 chunks its own CTA when the grid would cover less than half of the GPU
    const int nk = (int)((k + ltc::KC - 1) / ltc::KC);
    const int tiles = (int)(grid.x * grid.y);
    int splits = 1;
    if (g_splitk_on && tiles * 2 <= num_sms() && nk >= 16) {
        splits = nk / 8;
        if (splits > num_sms() / tiles) splits = num_sms() / tiles;
        if (splits > 16) splits = 16;
        if (splits < 2) splits = 1;
    }
    // the epilogue statistics need the complete sums: with split-K the caller runs the stand-alone GroupNorm statistics instead
    if (gn != nullptr && splits > 1) return 1;
    int cps = nk;
    float* part = nullptr;
    if (splits > 1) {
        cps = (nk + splits - 1) / splits;
        splits = (nk + cps - 1) / cps;
        part = splitk_scratch(st, (size_t)splits * (size_t)m * (size_t)n * sizeof(float));
        if (part == nullptr) { splits = 1; cps = nk; }
    }
    grid.z = (unsigned)splits;
    ProfRec rec{};
    const bool prof = g_prof_on;
    if (prof) {
        cudaEventCreate(&rec.a);
        cudaEventCreate(&rec.b);
        rec.m = m; rec.n = n; rec.k = k;
        cudaEventRecord(rec.a, st);
    }
    const bool persistent = g_persistent_on && splits == 1 && tiles > num_sms();
    if (persistent) {
        if (ensure_max_smem((const void*)ltc::linear_tc_persistent_kernel)) return -1;
        ltc::linear_tc_persistent_kernel<<<num_sms(), ltc::NTHREADS, ltc::SMEM_PERSIST, st>>>(mx, mw, bias, row_scale, y, (int)ldy, (int)m, (int)n,
                                                                                            (int)k, BN, relu, g, (int)grid.x, tiles);
    } else {
        ltc::linear_tc_kernel<<<grid, ltc::NTHREADS, ltc::SMEM, st>>>(mx, mw, bias, row_scale, y, (int)ldy, (int)m, (int)n, (int)k, BN, relu, g,
                                                                      part, cps);
    }
    if (part != nullptr) {
        const long long mn = (long long)m * n;
        ltc::splitk_reduce_kernel<<<(unsigned)((mn / 4 + 255) / 256), 256, 0, st>>>(part, splits, mn, (int)n, bias, row_scale, y, (int)ldy, relu);
        count_launches(1);
    }
    if (prof) {
        cudaEventRecord(rec.b, st);
        std::lock_guard<std::mutex> lk(g_prof_mu);
        g_prof.push_back(rec);
    }
    GEOB_CHECK_LAUNCH();
    count_launches(1);
    return 0;
}

}  // namespace geob200

extern "C" {

int geob200_set_linear_persistent(int on) {
    geob200::g_persistent_on = on != 0;
    return 0;
}

int geob200_set_split_k(int on) {
    geob200::g_splitk_on = on != 0;
    return 0;
}

// Profiling aid for bench.py: while enabled every tensor-core GEMM launch is bracketed by CUDA events on its stream.
int geob200_linear_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(geob200::g_prof_mu);
    for (auto& r : geob200::g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    geob200::g_prof.clear();
    geob200::g_prof_on = on != 0;
    return 0;
}

// Synchronises the recorded launches and returns their number; shapes[3*i..] = (m, n, k), ms[i] = kernel time.
int64_t geob200_linear_profile_read(int64_t capacity, int64_t* shapes, float* ms) {
    std::lock_guard<std::mutex> lk(geob200::g_prof_mu);
    int64_t n = 0;
    for (auto& r : geob200::g_prof) {
        if (n >= capacity) break;
        if (cudaEventSynchronize(r.b) != cudaSuccess) break;
        float t = 0.f;
        cudaEventElapsedTime(&t, r.a, r.b);
        shapes[3 * n] = r.m; shapes[3 * n + 1] = r.n; shapes[3 * n + 2] = r.k;
        ms[n] = t;
        ++n;
    }
    return n;
}

}  // extern "C"
