// Shared helpers for the geob200 CUDA kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace geob200 {

// Error plumbing for the C ABI: every entry point returns 0 on success or a negative code and leaves a
// human-readable message retrievable with geob200_last_error().
void set_error(const char* fmt, ...);
// number of kernels launched by this library since load (bench.py reports it as gpu_launches)
void count_launches(int n);
// Opt a kernel in to the device's maximum dynamic shared memory, once per (kernel, device), thread-safe (the engine launches
// from several host threads and a process may drive several GPUs).  Returns 0, or -1 with the error message set.
int ensure_max_smem(const void* kernel);

#define GEOB_CHECK_CUDA(expr)                                                                   \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) {                                                                \
            geob200::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,            \
                               cudaGetErrorString(_e));                                         \
            return -1;                                                                          \
        }                                                                                       \
    } while (0)

#define GEOB_CHECK_LAUNCH()                                                                     \
    do {                                                                                        \
        cudaError_t _e = cudaGetLastError();                                                    \
        if (_e != cudaSuccess) {                                                                \
            geob200::set_error("%s:%d kernel launch failed: %s", __FILE__, __LINE__,            \
                               cudaGetErrorString(_e));                                         \
            return -1;                                                                          \
        }                                                                                       \
    } while (0)

#define GEOB_REQUIRE(cond, ...)                                                                 \
    do {                                                                                        \
        if (!(cond)) {                                                                          \
            geob200::set_error(__VA_ARGS__);                                                    \
            return -2;                                                                          \
        }                                                                                       \
    } while (0)

static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Transposing warp butterfly: every lane holds NV = 2^b partial values v[0..NV); afterwards v[0] of lane l is the sum over
// all 32 lanes of value index (l >> (5 - b)) (NV - 1 exchange shuffles + (5 - b) plain ones instead of 5 per value).
template <int CNT, int MASK>
struct Butterfly {
    template <int NV>
    static __device__ __forceinline__ void run(float (&v)[NV], int lane) {
        if constexpr (CNT > 1) {
            constexpr int HALF = CNT / 2;
            const bool upper = (lane & MASK) != 0;
#pragma unroll
            for (int i = 0; i < HALF; ++i) {
                const float send = upper ? v[i] : v[i + HALF];
                const float keep = upper ? v[i + HALF] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, MASK);
            }
            if constexpr (MASK > 1) Butterfly<HALF, MASK / 2>::run(v, lane);
        } else {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], MASK);
            if constexpr (MASK > 1) Butterfly<1, MASK / 2>::run(v, lane);
        }
    }
};
template <int NV>
__device__ __forceinline__ float warp_butterfly(float (&v)[NV], int lane) {
    Butterfly<NV, 16>::run(v, lane);
    return v[0];
}

// GroupNorm statistics fused into the tensor-core GEMM epilogue (linear_tc.cu): per row-tile partial (sum, sumsq) per column
// slot in double; gn_seg_finalize_kernel (kpconv.cu) folds them into mean / rstd.
struct GnFuse {
    int groups;          // 0 = off
    int slot_width;      // min(channels per group, 32); filled in by linear_tc
    double* partial;     // [ceil(M/128)][N / slot_width][2]
};

// Rows of the GroupNorm statistics.  The backbone's GroupNorm normalises over the stacked rows of ONE pair
// (modules/kpconv/modules.py:46-50); a batch of several pairs (stack order [ref_1..ref_B, src_1..src_B] like the reference's
// collate with batch_size B, utils/data.py:144) has 2B clouds and cloud c belongs to pair c % n_pairs.  A single pair is one
// segment [0, n_rows), whatever its cloud split.  Passed to kernels by value (kernel parameter space), no device allocation.
constexpr int GEOB_MAX_CLOUDS = 64;
struct GnSeg {
    int n_clouds;                          // 2 * n_pairs; 1 in the GroupNorm segmentation of a single pair
    int n_pairs;
    int start[GEOB_MAX_CLOUDS + 1];        // first row of every cloud in the stacked level, start[n_clouds] = rows
};
static inline GnSeg gn_one_segment(int64_t n_rows) {
    GnSeg g;
    g.n_clouds = 1; g.n_pairs = 1; g.start[0] = 0; g.start[1] = (int)n_rows;
    return g;
}
// Internal forms of the GroupNorm-bearing entry points of geob200.h with the segmentation explicit; mean / rstd need
// 2 * groups * seg.n_pairs floats: size the workspace with geob200_group_norm_workspace_bytes.
int group_norm_impl(const float* x, int64_t n_rows, int64_t channels, int64_t groups, const float* gamma, const float* beta, float eps,
                    const float* residual, int leaky, float slope, float* y, void* workspace, size_t workspace_bytes, void* stream,
                    const GnSeg& seg);
int linear_group_norm_impl(const float* x, int64_t ldx, const float* weight, const float* bias, int64_t m, int64_t n, int64_t k,
                           int64_t groups, const float* gamma, const float* beta, float eps, const float* residual, int leaky,
                           float slope, float* pre_norm, float* y, void* workspace, size_t workspace_bytes, void* stream,
                           const GnSeg& seg);
int kpconv_group_norm_impl(const float* s_feats, const float* q_points, const float* s_points, const int64_t* neighbors,
                           int64_t n_query, int64_t n_support, int64_t n_neighbors, const float* kernel_points, int64_t n_kernel,
                           const float* weights_t, const float* bias, int64_t c_in, int64_t c_out, float sigma, int64_t groups,
                           const float* gamma, const float* beta, float eps, int leaky, float slope, float* pre_norm, float* y,
                           void* gn_workspace, size_t gn_workspace_bytes, void* workspace, size_t workspace_bytes, void* stream,
                           const GnSeg& seg);

int maxpool_seg(const float* x, const int64_t* neighbors, int64_t n_query, int64_t n_support, int64_t n_neighbors, int64_t channels,
                float* y, const GnSeg* seg, const int* cloud_max, void* stream);

// Bump allocator over a caller-provided workspace.
struct Arena {
    char* base;
    size_t off;
    size_t cap;
    __host__ Arena(void* p, size_t bytes) : base(static_cast<char*>(p)), off(0), cap(bytes) {}
    template <typename T>
    __host__ T* take(size_t n) {
        off = align_up(off, 256);
        T* r = reinterpret_cast<T*>(base + off);
        off += n * sizeof(T);
        return r;
    }
    __host__ bool ok() const { return off <= cap; }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// fp32 -> tf32 (10-bit mantissa) with round-to-nearest, returned as an fp32 bit pattern (low 13 bits zero)
__device__ __forceinline__ float tf32_rn(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

static inline int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

}  // namespace geob200
