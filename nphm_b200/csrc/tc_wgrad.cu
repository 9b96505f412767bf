// Weight gradients of a dense layer over the rows of a batch:  dW[n][k] = scale * sum_r D[r][n] * A[r][k]
//
// D (the layer's pre-activation gradient) and A (its input activation) are read in the packed operand format the layer chain
// writes (tc_linear.cuh: per 128-row tile and k-step of 16 features, [128 x 16 fp16 hi | 128 x 16 fp16 lo] in core-matrix order).
// The reduction runs over rows, so rows are the MMA K dimension and both operands are MN-major: one 16-byte chunk of the packed
// format (one row, 8 consecutive features) is one row of an MN-major no-swizzle core matrix, and a whole core matrix (8 rows x 8
// features, 128 contiguous bytes) is contiguous there too.  Only the order of the core matrices is not the uniform feature stride a
// descriptor needs (16-feature slabs lie 8 KB apart), so the loaders restage whole core matrices with cp.async: no conversion, no
// transposition.  Rows at or past M are zero-filled (the forward GEMMs never cared what the pad rows of the last tile hold).
//
// Arithmetic: 3-pass fp16 (hi*hi + hi*lo + lo*hi) with fp32 accumulation in TMEM, as every other layer of the project.
// Work split: an output tile is 128 x Kt (Kt <= 256); a 512 x 512 layer is 8 tiles, so the rows are split into ranges as well.
// Each range writes an fp32 partial, and a second kernel sums the partials in a fixed order: bitwise identical from run to run.
//
// The skinny products (the input layer's [xyz | noise] columns, the 3-row output layer, bias sums) use a SIMT kernel with the
// same partial / fixed-order reduction scheme.
#include "tc_linear.cuh"
#include <cuda_fp16.h>

namespace nphm {
namespace wg {
using namespace tc;

constexpr int kRows = 64;                 // rows (MMA K) per pipeline stage: 4 MMA k-steps
constexpr int kThreads = 256;
constexpr int kMaxKt = 256;
constexpr int kPackedStep = 8192;
constexpr int kHeadBytes = 1024;          // barriers and the TMEM address in front of the two stages

struct TcParams {
    const uint8_t *D; int d_ksteps, N;    // MMA A operand: rows of dW
    const uint8_t *A; int a_ksteps;       // MMA B operand: columns of dW
    long long M;
    int Kt, chunks, splits;
    float *partial; int ldp;              // partial[split][N][ldp]
};

__host__ __device__ inline size_t stage_bytes(int Kt) { return (size_t)(128 + Kt) * kRows * 4; }

// F features starting at k-step j0 of a packed buffer, rows [row0, row0 + 64) -> shared memory in MN-major core-matrix order:
// hi half then lo half (F * 128 bytes each); core matrix (row group g, feature group f) at g * F * 16 + f * 128.
__device__ __forceinline__ void stage_operand(uint32_t dst, const uint8_t *__restrict__ buf, int ksteps, int j0, int F,
                                              long long row0, long long M)
{
    // row0 is a multiple of 64: rows 0..63 or 64..127 of a 128-row tile, 2 KB of every k-step half
    const uint8_t *tile = buf + (size_t)(row0 >> 7) * ksteps * kPackedStep + (size_t)(row0 & 127) * 32;
    const int pieces = F * 16;            // 16-byte chunks: (slab, hi/lo, 128 per 64 rows)
    for (int i = threadIdx.x; i < pieces; i += kThreads) {
        const int c = i & 127, hl = (i >> 7) & 1, j = i >> 8;
        const int g = c >> 4, h = (c >> 3) & 1, rr = c & 7;
        const bool ok = row0 + g * 8 + rr < M && j0 + j < ksteps;
        const uint8_t *src = ok ? tile + (size_t)(j0 + j) * kPackedStep + hl * 4096 + c * 16 : buf;
        const uint32_t d = dst + (uint32_t)hl * F * kRows * 2 + (uint32_t)g * F * 16 + (uint32_t)(2 * j + h) * 128 + rr * 16;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(ok ? 16 : 0) : "memory");
    }
}

__global__ void __launch_bounds__(kThreads, 1) wgrad_tc_kernel(const TcParams p)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t *empty = reinterpret_cast<uint64_t *>(smem);          // [2]: the MMAs of a stage completed
    uint64_t *done = empty + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(empty + 4);
    uint8_t *const st0 = smem + kHeadBytes;
    const uint32_t sb = (uint32_t)stage_bytes(p.Kt);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_tile = blockIdx.x, k_tile = blockIdx.y, split = blockIdx.z;
    const int c0 = (int)((long long)split * p.chunks / p.splits), c1 = (int)((long long)(split + 1) * p.chunks / p.splits);

    if (threadIdx.x == 0) {
        mbar_init(&empty[0], 1); mbar_init(&empty[1], 1); mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kMaxKt)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    // MN-major A and B (instruction-descriptor bits 15 / 16)
    const uint32_t idesc = make_idesc_m(128, p.Kt) | (1u << 15) | (1u << 16);

    auto load = [&](int chunk, int s) {
        const uint32_t base = smem_u32(st0) + (uint32_t)s * sb;
        const long long row0 = (long long)chunk * kRows;
        stage_operand(base, p.D, p.d_ksteps, n_tile * 8, 128, row0, p.M);
        stage_operand(base + 128 * kRows * 4, p.A, p.a_ksteps, k_tile * (p.Kt / 16), p.Kt, row0, p.M);
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    load(c0, 0);
    for (int c = c0; c < c1; ++c) {
        const int i = c - c0, s = i & 1;
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            tc_fence_after();
            const uint32_t a = smem_u32(st0) + (uint32_t)s * sb, b = a + 128 * kRows * 4;
            const uint32_t a_lo = 128 * kRows * 2, b_lo = (uint32_t)p.Kt * kRows * 2;
            // descriptors of MN-major no-swizzle operands: LBO = stride between 8-row groups (K), SBO = between 8-feature groups
            for (int ks = 0; ks < kRows / 16; ++ks) {
                const uint32_t ao = a + ks * 2 * 128 * 16, bo = b + ks * 2 * (uint32_t)p.Kt * 16;
                const uint64_t ah = make_desc(ao, 128 * 16, 128), al = make_desc(ao + a_lo, 128 * 16, 128);
                const uint64_t bh = make_desc(bo, (uint32_t)p.Kt * 16, 128), bl = make_desc(bo + b_lo, (uint32_t)p.Kt * 16, 128);
                tc_mma_ss(tmem, ah, bh, idesc, (i | ks) ? 1 : 0);
                tc_mma_ss(tmem, ah, bl, idesc, 1);
                tc_mma_ss(tmem, al, bh, idesc, 1);
            }
            tc_commit(&empty[s]);
            if (c == c1 - 1) tc_commit(done);
        }
        if (c + 1 < c1) {
            if (i >= 1) mbar_wait(&empty[s ^ 1], ((i - 1) >> 1) & 1);     // the MMAs of chunk c - 1 have read stage s ^ 1
            load(c + 1, s ^ 1);
        }
    }
    mbar_wait(done, 0);
    tc_fence_after();
    // epilogue: warp (q, half) reads accumulator lanes 32 q .. (rows n of dW), every other 16-column unit
    const int q = warp & 3, half = warp >> 2;
    const int n = n_tile * 128 + q * 32 + lane;
    const int kbase = k_tile * p.Kt;
    float *dst = p.partial + ((size_t)split * p.N + (n < p.N ? n : 0)) * p.ldp + kbase;
    for (int u = half; u < p.Kt / 16; u += 2) {
        uint32_t r0[8], r1[8];
        const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + u * 16;
        tc_ld8(ta, r0);
        tc_ld8(ta + 8, r1);
        tc_wait_ld();
        if (n < p.N) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (kbase + u * 16 + e < p.ldp) dst[u * 16 + e] = __uint_as_float(r0[e]);
                if (kbase + u * 16 + 8 + e < p.ldp) dst[u * 16 + 8 + e] = __uint_as_float(r1[e]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kMaxKt) : "memory");
}

// partial[split][p][w] = sum over the rows of the split of P[r][p] * X[r][w],  X = [R (Wr columns) | 1 (ones)]:
// P packed (k-steps p_ksteps, width Pw), R row-major fp32.  Block = (16-feature slab of P, row range), thread = (feature, row lane);
// the 16 row lanes are summed in a fixed order.
constexpr int kSimtMaxW = 40;
__global__ void __launch_bounds__(256) wgrad_simt_kernel(const uint8_t *__restrict__ P, int p_ksteps, int Pw, const float *__restrict__ R,
                                                         int ldr, int Wr, int ones, long long M, long long rows_per_split,
                                                         float *__restrict__ partial)
{
    __shared__ float red[16][16][kSimtMaxW + 1];
    const int c = threadIdx.x & 15, rl = threadIdx.x >> 4, j = blockIdx.x;
    const int W = Wr + ones;
    const long long r0 = (long long)blockIdx.y * rows_per_split, r1 = min(M, r0 + rows_per_split);
    float acc[kSimtMaxW];
#pragma unroll
    for (int w = 0; w < kSimtMaxW; ++w) acc[w] = 0.f;
    for (long long r = r0 + rl; r < r1; r += 16) {
        const size_t off = ((size_t)(r >> 7) * p_ksteps + j) * 8192 + (size_t)((r & 127) >> 3) * 256 + (c >> 3) * 128 + (r & 7) * 16 +
                           (c & 7) * 2;
        const float v = __half2float(*reinterpret_cast<const __half *>(P + off)) +
                        __half2float(*reinterpret_cast<const __half *>(P + off + 4096));
        const float *rr = R ? R + (size_t)r * ldr : nullptr;
#pragma unroll
        for (int w = 0; w < kSimtMaxW; ++w) {
            if (w < Wr) acc[w] = fmaf(v, __ldg(rr + w), acc[w]);
            else if (w == Wr && ones) acc[w] += v;
        }
    }
#pragma unroll
    for (int w = 0; w < kSimtMaxW; ++w) if (w < W) red[rl][c][w] = acc[w];
    __syncthreads();
    for (int i = threadIdx.x; i < 16 * W; i += blockDim.x) {
        const int cc = i / W, w = i % W;
        float s = 0.f;
        for (int l = 0; l < 16; ++l) s += red[l][cc][w];
        if (j * 16 + cc < Pw) partial[((size_t)blockIdx.y * Pw + j * 16 + cc) * W + w] = s;
    }
}

// dst[n][col0 + k] (transpose: dst[k][col0 + n]) = scale * sum_s partial[s][n][k0 + k], splits summed in order
__device__ __forceinline__ float flag_nonfinite(float v, unsigned int *bad)
{
    if (bad && !isfinite(v)) atomicOr(bad, 1u);
    return v;
}

__global__ void reduce_partials_kernel(const float *__restrict__ partial, int splits, int N, int ldp, int k0, int K, float scale,
                                       float *__restrict__ dst, int ld_dst, int col0, int transpose, unsigned int *bad)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * K) return;
    const int n = (int)(idx / K), k = (int)(idx % K);
    float s = 0.f;
    for (int sp = 0; sp < splits; ++sp) s += partial[((size_t)sp * N + n) * ldp + k0 + k];
    if (transpose) dst[(size_t)k * ld_dst + col0 + n] = flag_nonfinite(scale * s, bad);
    else dst[(size_t)n * ld_dst + col0 + k] = flag_nonfinite(scale * s, bad);
}

// max |x| over n values (non-negative floats order like their bit patterns); *out zeroed by the caller
__global__ void abs_max_kernel(const float *__restrict__ x, long long n, unsigned int *__restrict__ out)
{
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(x[i]));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));
}

__global__ void scale_kernel(const float *__restrict__ x, long long n, float s, float *__restrict__ y, unsigned int *bad)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = flag_nonfinite(x[i] * s, bad);
}

// out[w] = sum_r R[r][w]: one block per column, fixed-order tree
__global__ void __launch_bounds__(256) column_sums_rows_kernel(const float *__restrict__ R, int ldr, long long M, float *__restrict__ out)
{
    __shared__ float s[256];
    float a = 0.f;
    for (long long r = threadIdx.x; r < M; r += 256) a += R[(size_t)r * ldr + blockIdx.x];
    s[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = s[0];
}

// condition columns: dst[n][col0 + j] (+)= scale * sum_q S[q][n] * cond[q][j]; accumulated for j < n_add (columns that also carry a
// point-dependent part), written for the rest
__global__ void cond_columns_kernel(const float *__restrict__ S, int N, const float *__restrict__ cond, int cond_dim, int Q, float scale,
                                    int n_add, float *__restrict__ dst, int ld, int col0, unsigned int *bad)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)N * cond_dim) return;
    const int n = (int)(idx / cond_dim), j = (int)(idx % cond_dim);
    float s = 0.f;
    for (int q = 0; q < Q; ++q) s = fmaf(S[(size_t)q * N + n], cond[(size_t)q * cond_dim + j], s);
    float *d = dst + (size_t)n * ld + col0 + j;
    *d = flag_nonfinite(j < n_add ? *d + scale * s : scale * s, bad);
}

static int reduce(const float *partial, int splits, int N, int ldp, int k0, int K, float scale, float *dst, int ld_dst, int col0,
                  bool transpose, unsigned int *bad, cudaStream_t stream)
{
    const long long total = (long long)N * K;
    if (total == 0) return NPHM_OK;
    reduce_partials_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, stream>>>(partial, splits, N, ldp, k0, K, scale, dst, ld_dst, col0,
                                                                                transpose ? 1 : 0, bad);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

int packed_packed(const uint8_t *D, int d_ksteps, int N, const uint8_t *A, int a_ksteps, int K, long long M, float scale, float *dst,
                  int ld_dst, DeviceBuffer &scratch, unsigned int *bad, cudaStream_t stream)
{
    NPHM_REQUIRE(D && A && dst && N > 0 && K > 0 && M > 0 && K <= a_ksteps * 16 && N <= d_ksteps * 16,
                 "wgrad: bad operands (N %d, K %d)", N, K);
    const int kpad = a_ksteps * 16;
    const int k_tiles = (kpad + kMaxKt - 1) / kMaxKt;
    const int Kt = ((kpad + k_tiles - 1) / k_tiles + 15) / 16 * 16;
    const int n_tiles = (N + 127) / 128;
    const int chunks = (int)ceil_div(M, kRows);
    const int splits = std::max(1, std::min(chunks, sm_count() / (n_tiles * k_tiles)));
    int rc;
    if ((rc = scratch.reserve((size_t)splits * N * kpad * sizeof(float)))) return rc;
    TcParams p{D, d_ksteps, N, A, a_ksteps, M, Kt, chunks, splits, scratch.as<float>(), kpad};
    const int smem = kHeadBytes + 2 * (int)stage_bytes(Kt);
    NPHM_CUDA_CHECK(cudaFuncSetAttribute(wgrad_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         kHeadBytes + 2 * (int)stage_bytes(kMaxKt)));
    wgrad_tc_kernel<<<dim3(n_tiles, k_tiles, splits), kThreads, smem, stream>>>(p);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return reduce(scratch.as<float>(), splits, N, kpad, 0, K, scale, dst, ld_dst, 0, false, bad, stream);
}

int packed_rows(const uint8_t *P, int p_ksteps, int Pw, const float *R, int ldr, int Wr, long long M, float scale, float *dst_w, int ld_w,
                bool transpose, float *dst_ones, DeviceBuffer &scratch, unsigned int *bad, cudaStream_t stream)
{
    const int ones = dst_ones ? 1 : 0, W = Wr + ones;
    NPHM_REQUIRE(P && M > 0 && Pw > 0 && Pw <= p_ksteps * 16 && W >= 1 && W <= kSimtMaxW && (Wr == 0 || R),
                 "wgrad: bad skinny operands (width %d)", Wr);
    const int slabs = (Pw + 15) / 16;
    const long long want = std::max(1LL, (long long)(4 * sm_count()) / slabs);
    const long long rows_per_split = std::max(256LL, ceil_div(M, want));
    const int splits = (int)ceil_div(M, rows_per_split);
    int rc;
    if ((rc = scratch.reserve((size_t)splits * Pw * W * sizeof(float)))) return rc;
    wgrad_simt_kernel<<<dim3(slabs, splits), 256, 0, stream>>>(P, p_ksteps, Pw, R, ldr, Wr, ones, M, rows_per_split,
                                                               scratch.as<float>());
    NPHM_CUDA_CHECK(cudaGetLastError());
    if (dst_w && Wr > 0 && (rc = reduce(scratch.as<float>(), splits, Pw, W, 0, Wr, scale, dst_w, ld_w, 0, transpose, bad, stream))) return rc;
    if (ones && (rc = reduce(scratch.as<float>(), splits, Pw, W, Wr, 1, scale, dst_ones, 1, 0, false, bad, stream))) return rc;
    return NPHM_OK;
}

int range_sums(const uint8_t *P, int p_ksteps, int Pw, long long M, long long rows_per_range, float *out, cudaStream_t stream)
{
    NPHM_REQUIRE(P && out && M > 0 && rows_per_range > 0 && Pw > 0 && Pw <= p_ksteps * 16, "wgrad: bad range sums");
    wgrad_simt_kernel<<<dim3((Pw + 15) / 16, (unsigned)ceil_div(M, rows_per_range)), 256, 0, stream>>>(P, p_ksteps, Pw, nullptr, 0, 0, 1, M,
                                                                                                      rows_per_range, out);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

int rows_column_sums(const float *R, int ldr, int W, long long M, float *out, cudaStream_t stream)
{
    column_sums_rows_kernel<<<W, 256, 0, stream>>>(R, ldr, M, out);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

int abs_max(const float *x, long long n, unsigned int *out_dev, cudaStream_t stream)
{
    NPHM_CUDA_CHECK(cudaMemsetAsync(out_dev, 0, sizeof(unsigned int), stream));
    abs_max_kernel<<<(unsigned)std::min(ceil_div(n, 256), 1024LL), 256, 0, stream>>>(x, n, out_dev);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

int scale(const float *x, long long n, float s, float *y, unsigned int *bad, cudaStream_t stream)
{
    if (n == 0) return NPHM_OK;
    scale_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, stream>>>(x, n, s, y, bad);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

int cond_columns(const float *S, int N, const float *cond, int cond_dim, int Q, float scale, int n_add, float *dst, int ld, int col0,
                 unsigned int *bad, cudaStream_t stream)
{
    const long long total = (long long)N * cond_dim;
    if (total == 0) return NPHM_OK;
    cond_columns_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, stream>>>(S, N, cond, cond_dim, Q, scale, n_add, dst, ld, col0, bad);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

}  // namespace wg
}  // namespace nphm
