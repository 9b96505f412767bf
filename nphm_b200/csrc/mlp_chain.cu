// Layer-by-layer passes of a DeepSDF-style stack on the generic tcgen05 linear layer (tc_linear.cu):
//
//   value pass     h_l = softplus(W_l in_l + c_l), s_l = softplus'(.)          (any width: the NPM baseline 515 -> 1024 x 8 ...)
//   tangent pass   forward-mode derivative w.r.t. xyz:  t_l = s_l * (W_l t_{l-1}),  3 rows per point  ->  Jacobian d out / d xyz
//   adjoint pass   d_l-1 = s_l-1 * (W_l^T d_l)  ->  gradient w.r.t. the per-query condition (and, optionally, w.r.t. xyz)
//
// Reference semantics: DeepSDF.forward src/NPHM/models/deepSDF.py:64-89 (skip connection `cat([x, inp]) / sqrt(2)` at layer
// nlayers // 2, Softplus(beta = 100)); `jac` src/NPHM/models/diff_operators.py:26-54 (three autograd passes there, one
// forward-mode pass here); the adjoint pass is what `loss.backward()` (src/NPHM/models/fitting.py:167) does to the deformation
// network in the joint fitter.  The condition is constant over the points of a query, so its part of layers 0 and `skip` is
// folded into per-query constants (simt.cu: cvec) and its gradient only needs the per-query column sums of d_0 and d_skip.
#include "tc_linear.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cuda_fp16.h>

namespace nphm {
namespace chain {

constexpr float kInvSqrt2 = 0.70710678118654752440f;

__global__ void column_sums_kernel(const float *__restrict__ X, int ld, long long rows_per_query, int n_cols, float *__restrict__ out)
{
    // out[q][c] = sum over the rows of query q of X[row][c]; grid = (col blocks, queries, row chunks), atomics across chunks
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int q = blockIdx.y;
    if (c >= n_cols) return;
    const long long chunk = (rows_per_query + gridDim.z - 1) / gridDim.z;
    const long long r0 = (long long)blockIdx.z * chunk, r1 = min(rows_per_query, r0 + chunk);
    float s = 0.f;
    for (long long r = r0; r < r1; ++r) s += X[((size_t)q * rows_per_query + r) * ld + c];
    if (r1 > r0) atomicAdd(out + (size_t)q * n_cols + c, s);
}

// The same sums over a PACKED activation buffer (tc_linear.cuh: per 128-row tile and k-step [128 x 16 fp16 hi | 128 x 16 fp16 lo],
// core-matrix order; value = hi + lo).  grid (tiles, k-steps), 256 threads: thread = (row of the tile, 8 of the 16 columns).
__global__ void __launch_bounds__(256) column_sums_packed_kernel(const uint8_t *__restrict__ X, int ksteps, long long M,
                                                                 long long rows_per_query, int n_cols, float *__restrict__ out)
{
    __shared__ float s_sum[16];
    const int r = threadIdx.x >> 1, ch = threadIdx.x & 1, lane = threadIdx.x & 31;
    const int j = blockIdx.y;
    const long long row0 = (long long)blockIdx.x * 128, row = row0 + r;
    const bool ok = row < M;
    const long long q = (ok ? row : M - 1) / rows_per_query;
    const long long q_first = row0 / rows_per_query, q_last = (min(row0 + 127, M - 1)) / rows_per_query;
    const bool block_uniform = q_first == q_last;
    if (threadIdx.x < 16) s_sum[threadIdx.x] = 0.f;
    __syncthreads();
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    if (ok) {
        const uint8_t *src = X + ((size_t)blockIdx.x * ksteps + j) * 8192 + (size_t)(r >> 3) * 256 + (size_t)ch * 128 + (size_t)(r & 7) * 16;
        const uint4 h = *reinterpret_cast<const uint4 *>(src), l = *reinterpret_cast<const uint4 *>(src + 4096);
        const uint32_t hw[4] = {h.x, h.y, h.z, h.w}, lw[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 a = __half22float2(*reinterpret_cast<const __half2 *>(&hw[i]));
            const float2 b = __half22float2(*reinterpret_cast<const __half2 *>(&lw[i]));
            v[2 * i] = a.x + b.x; v[2 * i + 1] = a.y + b.y;
        }
    }
    const int c0 = j * 16 + ch * 8;
    if (block_uniform) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float x = v[i];
#pragma unroll
            for (int o = 2; o < 32; o <<= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if (lane < 2 && x != 0.f) atomicAdd(&s_sum[ch * 8 + i], x);
        }
        __syncthreads();
        if (threadIdx.x < 16 && j * 16 + threadIdx.x < n_cols && s_sum[threadIdx.x] != 0.f)
            atomicAdd(out + (size_t)q_first * n_cols + j * 16 + threadIdx.x, s_sum[threadIdx.x]);
    } else if (ok) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (c0 + i < n_cols && v[i] != 0.f) atomicAdd(out + (size_t)q * n_cols + c0 + i, v[i]);
    }
}

// grad_cond[q][j] = sum_n W0[n][3 + j] * S0[q][n]  +  sum_n Ws[n][Nh + 3 + j] * Ss[q][n] / sqrt(2)
__global__ void cond_grad_kernel(const float *__restrict__ W0, int ld0, int N0, const float *__restrict__ S0,
                                 const float *__restrict__ Ws, int lds, int Ns, int skip_col0, const float *__restrict__ Ss,
                                 int cond_dim, float *__restrict__ out)
{
    // grid (column blocks, queries, chunks of the n range): `out` is zeroed by the caller, the chunks add their partial sums
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int q = blockIdx.y;
    if (j >= cond_dim) return;
    const int c0 = (N0 + gridDim.z - 1) / gridDim.z, a0 = blockIdx.z * c0, b0 = min(N0, a0 + c0);
    float s = 0.f;
    for (int n = a0; n < b0; ++n) s = fmaf(W0[(size_t)n * ld0 + 3 + j], S0[(size_t)q * N0 + n], s);
    if (Ws) {
        const int c1 = (Ns + gridDim.z - 1) / gridDim.z, a1 = blockIdx.z * c1, b1 = min(Ns, a1 + c1);
        float t = 0.f;
        for (int n = a1; n < b1; ++n) t = fmaf(Ws[(size_t)n * lds + skip_col0 + j], Ss[(size_t)q * Ns + n], t);
        s = fmaf(t, kInvSqrt2, s);
    }
    atomicAdd(out + (size_t)q * cond_dim + j, s);
}

// out[(q, n)][i][j] = T[(q, n, j)][i]   (tangent rows -> Jacobian layout B x N x out x 3)
__global__ void jacobian_layout_kernel(const float *__restrict__ T, int ld, long long n_rows, int out_dim, float *__restrict__ J)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n_rows * out_dim * 3) return;
    const int j = (int)(idx % 3);
    const int i = (int)((idx / 3) % out_dim);
    const long long n = idx / (3 * out_dim);
    J[idx] = T[(size_t)(n * 3 + j) * ld + i];
}

// in place: J (3 x 3 per point, row i = gradient of output i) -> (I + J)^-1  (adjugate / determinant)
__global__ void inverse_plus_identity_kernel(float *__restrict__ J, long long n)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    float *m = J + p * 9;
    const float a = m[0] + 1.f, b = m[1], c = m[2], d = m[3], e = m[4] + 1.f, f = m[5], g = m[6], h = m[7], i = m[8] + 1.f;
    const float A = e * i - f * h, B = -(d * i - f * g), C = d * h - e * g;
    const float inv = 1.0f / (a * A + b * B + c * C);
    m[0] = A * inv; m[1] = -(b * i - c * h) * inv; m[2] = (b * f - c * e) * inv;
    m[3] = B * inv; m[4] = (a * i - c * g) * inv;  m[5] = -(a * f - c * d) * inv;
    m[6] = C * inv; m[7] = -(a * h - b * g) * inv; m[8] = (a * e - b * d) * inv;
}

__global__ void add3_kernel(const float *__restrict__ src, int ld, long long rows, float *__restrict__ dst)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < rows * 3) dst[idx] += src[(idx / 3) * ld + idx % 3];
}

}  // namespace chain

// ------------------------------------------------------------------------------------------------ packed stack
struct MlpChain {
    bool packed = false;
    int n_lin = 0;
    tcl::PackedLinear fwd[kMaxLayers];        // B = W_l restricted to its point-dependent columns (1/sqrt2 folded at the skip)
    tcl::PackedLinear adj[kMaxLayers];        // B = W_l^T (input-activation columns only)
    tcl::PackedLinear adj_x0, adj_xs;         // W_0[:, 0:3]^T and W_skip[:, Nh:Nh+3]^T / sqrt2  (gradient w.r.t. xyz)
    // activations between the layers live in the packed operand format (Hp: values, Tp: tangents, Dp: adjoints), the
    // activation derivatives S in the blocked fp32 layout ([128-row tile][feature][128]) - every access of the passes is coalesced
    DeviceBuffer Hp[kMaxLayers], S[kMaxLayers], Tp[2], Dp[2], Tlast, sums0, sumss, out_tmp, xtmp;
    int ld[kMaxLayers];
    long long value_rows = 0;                 // rows of the last value pass that kept the activation derivatives
    bool have_deriv = false;
    // training forward with per-point condition noise: layers 0, skip - 1 and skip re-packed with the noise columns riding with
    // xyz (train_pack); valid for noise width `train_noise` of weight generation `train_gen`
    tcl::PackedLinear train_fwd[kMaxLayers];
    int train_noise = 0;
    unsigned long long train_gen = 0;
    DeviceBuffer wg_scratch;                  // partial sums of the weight-gradient GEMMs
    DeviceBuffer wg_sums0, wg_sumss, wg_grad;            // fixed-order per-query sums, scaled grad_out
    DeviceBuffer wg_flags;                    // [0] max |grad_out| (bits), [1] non-zero: a gradient output is not finite
};

static int pad4(int n) { return (n + 3) / 4 * 4; }
constexpr int kChainNt = 128;

int chain_pack(nphm_mlp *h, cudaStream_t stream)
{
    if (!h->chain) h->chain = new MlpChain();
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    c.n_lin = s.n_lin;
    int rc;
    for (int l = 0; l < s.n_lin; ++l) {
        const float *W = h->weights.W[l].as<float>();
        const int ldw = s.in_total[l];
        const float scale = l == s.skip ? chain::kInvSqrt2 : 1.0f;
        // forward: point-dependent leading columns (xyz | h_{l-1} | [h_{skip-1}, xyz])
        // (the layer in front of the skip layer reserves 3 output columns: its epilogue appends xyz / the tangent seeds)
        // tiles of <= 128 output columns: the passes run on a few thousand rows (fitting), where CTAs count more than tile width
        if ((rc = c.fwd[l].pack(W, ldw, s.N[l], s.K[l], 0, 0, false, scale, stream, 1, 0, nullptr, 0, l + 1 == s.skip ? 3 : 0,
                                kChainNt)))
            return rc;
        // adjoint w.r.t. the input activations of layer l (l >= 1): columns [0, N_{l-1})
        if (l >= 1 && (rc = c.adj[l].pack(W, ldw, s.N[l - 1], s.N[l], 0, 0, true, scale, stream, 1, 0, nullptr, 0, 0, kChainNt)))
            return rc;
        c.ld[l] = pad4(s.N[l]);
    }
    if ((rc = c.adj_x0.pack(h->weights.W[0].as<float>(), s.in_total[0], 3, s.N[0], 0, 0, true, 1.0f, stream))) return rc;
    if (s.skip > 0 && s.skip < s.n_lin &&
        (rc = c.adj_xs.pack(h->weights.W[s.skip].as<float>(), s.in_total[s.skip], 3, s.N[s.skip], s.N[s.skip - 1], 0, true,
                            chain::kInvSqrt2, stream))) return rc;
    c.packed = true;
    return NPHM_OK;
}

void chain_destroy(nphm_mlp *h)
{
    delete h->chain;
    h->chain = nullptr;
}

static size_t packed_bytes(long long rows, int ksteps) { return (size_t)ceil_div(rows, 128) * ksteps * 8192; }

// Where a value pass reads its point inputs and leaves its activations.  x: [M][xw] point-dependent input columns (xyz, or
// [xyz | noise] in a training forward): layer 0's input and the columns appended in front of the skip layer.
struct ChainIO {
    const float *x = nullptr; int xw = 3;
    const tcl::PackedLinear *fwd[kMaxLayers] = {};
    uint8_t *Hp[kMaxLayers] = {};
    float *S[kMaxLayers] = {};                // activation derivatives, blocked (NULL: not kept)
};

static int value_pass_io(nphm_mlp *h, const ChainIO &io, int n_queries, long long n_points, float *out, cudaStream_t stream)
{
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    const long long M = (long long)n_queries * n_points;
    int rc;
    for (int l = 0; l < s.n_lin; ++l) {
        const bool last = l == s.n_lin - 1;
        const tcl::PackedLinear &w = *io.fwd[l];
        tcl::LinearParams p;
        p.M = M;
        if (l == 0) { p.A1 = io.x; p.lda1 = io.xw; p.K1 = io.xw; }
        else { p.Ap = io.Hp[l - 1]; p.a_ksteps = w.ksteps; }     // at the skip layer: [h | x], appended below
        p.bias = h->cvec.as<float>() + s.coff[l]; p.ldb = s.cvec_stride; p.rows_per_bias = n_points;
        if (last) {
            p.mode = tcl::kModeLinear;
            p.C = out; p.ldc = s.N[l];
        } else {
            p.mode = tcl::kModeSoftplus;
            p.Cp = io.Hp[l]; p.c_ksteps = w.packed_ksteps_out();
            if (l + 1 == s.skip) { p.app = io.x; p.app_ld = io.xw; p.app_w = io.xw; }
            if (io.S[l]) { p.Dv = io.S[l]; p.lddv = c.ld[l]; p.dv_blocked = 1; }
        }
        if ((rc = tcl::launch_linear(w, p, stream))) return rc;
    }
    return NPHM_OK;
}

static size_t deriv_bytes(const MlpChain &c, long long rows, int l) { return (size_t)ceil_div(rows, 128) * 128 * c.ld[l] * sizeof(float); }

// value pass over M = n_queries * n_points rows into the handle's buffers; keeps h_l (packed) and (want_deriv) s_l (blocked) of
// every hidden layer; `out` = last layer, row-major
static int value_pass(nphm_mlp *h, const float *xyz, int n_queries, long long n_points, bool want_deriv, float *out,
                      cudaStream_t stream)
{
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    const long long M = (long long)n_queries * n_points;
    ChainIO io;
    io.x = xyz;
    int rc;
    for (int l = 0; l < s.n_lin; ++l) {
        io.fwd[l] = &c.fwd[l];
        if (l == s.n_lin - 1) break;
        if ((rc = c.Hp[l].reserve(packed_bytes(M, c.fwd[l].packed_ksteps_out())))) return rc;
        io.Hp[l] = c.Hp[l].as<uint8_t>();
        if (want_deriv) {
            if ((rc = c.S[l].reserve(deriv_bytes(c, M, l)))) return rc;
            io.S[l] = c.S[l].as<float>();
        }
    }
    if ((rc = value_pass_io(h, io, n_queries, n_points, out, stream))) return rc;
    c.value_rows = M;
    c.have_deriv = want_deriv;
    return NPHM_OK;
}

// the adjoint of a layer's pre-activations: row-major fp32 for the output layer (the caller's grad_out), packed below it
struct Adjoint { const float *rows; int ld; const uint8_t *packed; int ksteps; int width; };

// adjoint pass from the output layer down to d_0, d_{l-1} = s_{l-1} * (d_l W_l), over the activation derivatives S of a value pass:
// per-query column sums of d_0 / d_skip (c.sums0 / c.sumss), grad_cond [q][cond_dim] and grad_xyz [q][n][3] (each optional).
// on_layer(l, d_l) runs for l = L .. 0 while d_l is alive (d_l lives in Dp[l & 1], overwritten two layers further down).
template <class OnLayer>
static int adjoint_pass(nphm_mlp *h, long long M, long long n_points, const float *grad_out_dev, float *const *S, float *grad_cond_dev,
                        float *grad_xyz_dev, OnLayer &&on_layer, cudaStream_t stream)
{
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    const int L = s.n_lin - 1, out_dim = s.N[L];
    const int n_queries = (int)(M / n_points);
    int rc;
    int max_ks = 1;
    for (int l = 1; l <= L; ++l) max_ks = std::max(max_ks, (s.N[l - 1] + 15) / 16);
    for (int i = 0; i < 2; ++i)
        if ((rc = c.Dp[i].reserve(packed_bytes(M, max_ks)))) return rc;
    if ((rc = c.sums0.reserve((size_t)n_queries * s.N[0] * sizeof(float)))) return rc;
    if ((rc = c.sumss.reserve((size_t)n_queries * s.N[s.skip] * sizeof(float)))) return rc;
    NPHM_CUDA_CHECK(cudaMemsetAsync(c.sums0.ptr, 0, (size_t)n_queries * s.N[0] * sizeof(float), stream));
    NPHM_CUDA_CHECK(cudaMemsetAsync(c.sumss.ptr, 0, (size_t)n_queries * s.N[s.skip] * sizeof(float), stream));
    auto as_input = [&](tcl::LinearParams &p, const Adjoint &d) {
        if (d.packed) { p.Ap = d.packed; p.a_ksteps = d.ksteps; }
        else { p.A1 = d.rows; p.lda1 = d.ld; p.K1 = d.width; }
    };
    auto col_sums = [&](const Adjoint &d, float *out) {
        dim3 grid((unsigned)ceil_div(M, 128), (unsigned)d.ksteps);
        chain::column_sums_packed_kernel<<<grid, 256, 0, stream>>>(d.packed, d.ksteps, M, n_points, d.width, out);
    };
    // d_{l-1} = s_{l-1} * (d_l W_l), from the output layer down to d_0;  d_l lives in Dp[l & 1]
    Adjoint d_cur{grad_out_dev, out_dim, nullptr, 0, out_dim};
    for (int l = L; l >= 1; --l) {
        if ((rc = on_layer(l, d_cur))) return rc;
        tcl::LinearParams p;
        p.M = M;
        as_input(p, d_cur);
        p.mode = tcl::kModeMult; p.Mul = S[l - 1]; p.ldmul = c.ld[l - 1]; p.mul_div = 1; p.mul_blocked = 1;
        const int ks = (s.N[l - 1] + 15) / 16;
        p.Cp = c.Dp[(l - 1) & 1].as<uint8_t>(); p.c_ksteps = ks;
        if ((rc = tcl::launch_linear(c.adj[l], p, stream))) return rc;
        if (l == s.skip) {
            // d_skip (the layer's pre-activation gradient) is d_cur here: its column sums feed the condition gradient
            NPHM_REQUIRE(d_cur.packed, "adjoint pass: skip layer directly below the output is not supported");
            col_sums(d_cur, c.sumss.as<float>());
            NPHM_CUDA_CHECK(cudaGetLastError());
            if (grad_xyz_dev) {
                tcl::LinearParams px;
                px.M = M;
                as_input(px, d_cur);
                px.mode = tcl::kModeLinear; px.C = grad_xyz_dev; px.ldc = 3;
                if ((rc = tcl::launch_linear(c.adj_xs, px, stream))) return rc;
            }
        }
        d_cur = Adjoint{nullptr, 0, c.Dp[(l - 1) & 1].as<uint8_t>(), ks, s.N[l - 1]};
    }
    col_sums(d_cur, c.sums0.as<float>());
    NPHM_CUDA_CHECK(cudaGetLastError());
    if ((rc = on_layer(0, d_cur))) return rc;
    if (grad_cond_dev) {
        NPHM_CUDA_CHECK(cudaMemsetAsync(grad_cond_dev, 0, (size_t)n_queries * s.cond_dim * sizeof(float), stream));
        dim3 grid((unsigned)ceil_div(s.cond_dim, 128), (unsigned)n_queries, 16);
        chain::cond_grad_kernel<<<grid, 128, 0, stream>>>(h->weights.W[0].as<float>(), s.in_total[0], s.N[0], c.sums0.as<float>(),
                                                          h->weights.W[s.skip].as<float>(), s.in_total[s.skip], s.N[s.skip],
                                                          s.N[s.skip - 1] + 3, c.sumss.as<float>(), s.cond_dim, grad_cond_dev);
        NPHM_CUDA_CHECK(cudaGetLastError());
    }
    if (grad_xyz_dev) {
        // + d_0 W_0[:, 0:3]  (the skip-layer part was written above): through a temporary, then accumulate
        tcl::LinearParams px;
        px.M = M;
        as_input(px, d_cur);
        px.mode = tcl::kModeLinear;
        if ((rc = c.xtmp.reserve((size_t)M * 4 * sizeof(float)))) return rc;
        px.C = c.xtmp.as<float>(); px.ldc = 4;
        if ((rc = tcl::launch_linear(c.adj_x0, px, stream))) return rc;
        chain::add3_kernel<<<(unsigned)ceil_div(M * 3, 256), 256, 0, stream>>>(c.xtmp.as<float>(), 4, M, grad_xyz_dev);
        NPHM_CUDA_CHECK(cudaGetLastError());
    }
    return NPHM_OK;
}

}  // namespace nphm

using namespace nphm;

static int chain_ready(nphm_mlp *h, const char *who)
{
    NPHM_REQUIRE(h && h->loaded, "%s: weights not loaded", who);
    NPHM_REQUIRE(h->chain && h->chain->packed, "%s: layer chain not packed", who);
    NPHM_REQUIRE(h->dims.skip >= 1 && h->dims.skip < h->dims.n_lin - 1, "%s: unsupported skip position", who);
    return NPHM_OK;
}

// forward of an arbitrary-width stack, layer by layer (used when no fused kernel takes the shape)
extern "C" int nphm_mlp_query_layers(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                                     float *out_dev, void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int rc = chain_ready(h, "nphm_mlp_query_layers");
    if (rc) return rc;
    NPHM_REQUIRE(n_queries >= 1 && n_points >= 0 && cond_dev, "nphm_mlp_query_layers: bad arguments");
    if (n_points == 0) return NPHM_OK;
    NPHM_REQUIRE(xyz_dev && out_dev, "nphm_mlp_query_layers: NULL pointer");
    if ((rc = mlp_prepare(h, cond_dev, n_queries, stream))) return rc;
    return value_pass(h, xyz_dev, n_queries, n_points, false, out_dev, stream);
}

// value + forward-mode tangents: out [q][n][out_dim] (optional), jac [q][n][out_dim][3] = d out / d xyz
extern "C" int nphm_mlp_jacobian(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                                 float *out_dev, float *jac_dev, void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int rc = chain_ready(h, "nphm_mlp_jacobian");
    if (rc) return rc;
    NPHM_REQUIRE(n_queries >= 1 && n_points >= 0 && cond_dev && jac_dev, "nphm_mlp_jacobian: bad arguments");
    if (n_points == 0) return NPHM_OK;
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    const long long M = (long long)n_queries * n_points;
    const int out_dim = s.N[s.n_lin - 1];
    if ((rc = mlp_prepare(h, cond_dev, n_queries, stream))) return rc;
    float *out = out_dev;
    if (!out) {
        if ((rc = c.out_tmp.reserve((size_t)M * out_dim * sizeof(float)))) return rc;
        out = c.out_tmp.as<float>();
    }
    if ((rc = value_pass(h, xyz_dev, n_queries, n_points, true, out, stream))) return rc;
    // tangent pass: rows (point, j), j = 0..2; tangents between the layers packed, the last layer row-major for the layout kernel
    int max_ks = 1;
    for (int l = 0; l + 1 < s.n_lin; ++l) max_ks = std::max(max_ks, c.fwd[l].packed_ksteps_out());
    for (int i = 0; i < 2; ++i)
        if ((rc = c.Tp[i].reserve(packed_bytes(3 * M, max_ks)))) return rc;
    const int ld_last = c.ld[s.n_lin - 1];
    if ((rc = c.Tlast.reserve((size_t)3 * M * ld_last * sizeof(float)))) return rc;
    for (int l = 0; l < s.n_lin; ++l) {
        const bool last = l == s.n_lin - 1;
        tcl::LinearParams p;
        p.M = 3 * M;
        if (l == 0) { p.K1 = 0; p.K2 = 3; p.a2_onehot = 1; }
        else { p.Ap = c.Tp[(l - 1) & 1].as<uint8_t>(); p.a_ksteps = c.fwd[l].ksteps; }
        if (last) {
            p.mode = tcl::kModeLinear;
            p.C = c.Tlast.as<float>(); p.ldc = ld_last;
        } else {
            p.mode = tcl::kModeMult; p.Mul = c.S[l].as<float>(); p.ldmul = c.ld[l]; p.mul_div = 3; p.mul_blocked = 1;
            p.Cp = c.Tp[l & 1].as<uint8_t>(); p.c_ksteps = c.fwd[l].packed_ksteps_out();
            if (l + 1 == s.skip) { p.app_onehot = 1; p.app_w = 3; }               // d xyz / d xyz_j = e_j
        }
        if ((rc = tcl::launch_linear(c.fwd[l], p, stream))) return rc;
    }
    const long long total = M * out_dim * 3;
    chain::jacobian_layout_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, stream>>>(c.Tlast.as<float>(), ld_last, M, out_dim,
                                                                                      jac_dev);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

// adjoint pass: grad_cond [q][cond_dim] = sum_n (d out_n / d cond)^T grad_out_n ; grad_xyz [q][n][3] optional
extern "C" int nphm_mlp_backward_inputs(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                                        const float *grad_out_dev, float *grad_cond_dev, float *grad_xyz_dev, void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int rc = chain_ready(h, "nphm_mlp_backward_inputs");
    if (rc) return rc;
    NPHM_REQUIRE(n_queries >= 1 && n_points > 0 && cond_dev && grad_out_dev && (grad_cond_dev || grad_xyz_dev),
                 "nphm_mlp_backward_inputs: bad arguments");
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    const long long M = (long long)n_queries * n_points;
    const int L = s.n_lin - 1, out_dim = s.N[L];
    if (xyz_dev) {
        if ((rc = mlp_prepare(h, cond_dev, n_queries, stream))) return rc;
        if ((rc = c.out_tmp.reserve((size_t)M * out_dim * sizeof(float)))) return rc;
        if ((rc = value_pass(h, xyz_dev, n_queries, n_points, true, c.out_tmp.as<float>(), stream))) return rc;
        c.value_rows = M;
    } else {
        // xyz_dev == NULL: the activation derivatives of the previous nphm_mlp_jacobian / nphm_mlp_inverse_jacobian call on this
        // handle are reused (the joint fitter differentiates at the same points it just took the Jacobian at)
        NPHM_REQUIRE(c.value_rows == M && c.have_deriv, "nphm_mlp_backward_inputs: no matching value pass to reuse");
    }
    float *S[kMaxLayers];
    for (int l = 0; l < L; ++l) S[l] = c.S[l].as<float>();
    return adjoint_pass(h, M, n_points, grad_out_dev, S, grad_cond_dev, grad_xyz_dev, [](int, const Adjoint &) { return NPHM_OK; },
                        stream);
}

extern "C" int nphm_mlp_inverse_jacobian(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries, long long n_points,
                                         float *out_dev, float *jinv_dev, void *stream_)
{
    NPHM_REQUIRE(h && h->loaded && h->dims.N[h->dims.n_lin - 1] == 3, "nphm_mlp_inverse_jacobian: needs a 3-output stack");
    int rc = nphm_mlp_jacobian(h, xyz_dev, cond_dev, n_queries, n_points, out_dev, jinv_dev, stream_);
    if (rc || n_points == 0) return rc;
    const long long M = (long long)n_queries * n_points;
    chain::inverse_plus_identity_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, static_cast<cudaStream_t>(stream_)>>>(jinv_dev, M);
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

// ------------------------------------------------------------------------------------------------ training (first order)
// Reference: the deformation network of stage-2 training, scripts/training/train_corresp.py -> training_corresp.py:154-176:
// two forwards (correspondences, then zero-regulariser samples) and one loss.backward() that needs the gradients w.r.t. the
// weights, the condition and the points.  In training mode the reference adds randn(B, N, 32) / 200 to the compressed identity
// code per point (deepSDF.py:220-221): those columns of the condition are no longer constant over a query, so they ride with xyz
// (layer 0 reads [xyz | noise], the layer in front of the skip appends [xyz | noise]); the rest stays folded into the per-query
// constants.  The activations of a forward live in a caller-owned workspace, because both forwards precede the backward.
namespace nphm {
namespace chain {

constexpr int kMaxNoise = 36;                 // 3 + noise + a ones column within the skinny weight-gradient kernel
constexpr unsigned long long kTrainMagic = 0x314e5254'4d48504eull;

struct TrainHeader {
    unsigned long long magic, weight_gen;
    const void *handle;
    long long rows, n_points;
    int n_queries, noise_dim;
};
constexpr size_t kHeaderBytes = 256;

struct TrainLayout { size_t x, hp[kMaxLayers], s[kMaxLayers], total; };

static TrainLayout train_layout(const StackDims &s, long long M, int nd)
{
    auto align = [](size_t b) { return (b + 255) / 256 * 256; };
    TrainLayout t{};
    size_t off = kHeaderBytes;
    t.x = off;
    off += align((size_t)M * (3 + nd) * sizeof(float));
    for (int l = 0; l + 1 < s.n_lin; ++l) {
        const int extra = l + 1 == s.skip ? 3 + nd : 0;
        t.hp[l] = off;
        off += packed_bytes(M, (s.N[l] + extra + 15) / 16);
    }
    for (int l = 0; l + 1 < s.n_lin; ++l) {
        t.s[l] = off;
        off += (size_t)ceil_div(M, 128) * 128 * pad4(s.N[l]) * sizeof(float);
    }
    t.total = off;
    return t;
}

static bool noise_layer(const StackDims &s, int l) { return l == 0 || l + 1 == s.skip || l == s.skip; }

// layers 0, skip - 1 and skip with `nd` noise columns behind xyz (no-op for nd == 0: the inference packing is used)
static int train_pack(nphm_mlp *h, int nd, cudaStream_t stream)
{
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    if (nd == 0 || (c.train_noise == nd && c.train_gen == h->weight_gen)) return NPHM_OK;
    for (int l = 0; l < s.n_lin; ++l) {
        if (!noise_layer(s, l)) continue;
        const int K = l == 0 ? 3 + nd : (l == s.skip ? s.N[l - 1] + 3 + nd : s.K[l]);
        const int extra = l + 1 == s.skip ? 3 + nd : 0;
        int rc = c.train_fwd[l].pack(h->weights.W[l].as<float>(), s.in_total[l], s.N[l], K, 0, 0, false, l == s.skip ? kInvSqrt2 : 1.0f,
                                     stream, 1, 0, nullptr, 0, extra, kChainNt);
        if (rc) return rc;
    }
    c.train_noise = nd;
    c.train_gen = h->weight_gen;
    return NPHM_OK;
}

static const tcl::PackedLinear &train_fwd(MlpChain &c, const StackDims &s, int l, int nd)
{
    return nd > 0 && noise_layer(s, l) ? c.train_fwd[l] : c.fwd[l];
}

// the workspace header, written on the stream (a host-to-device copy from pageable memory could synchronise)
__global__ void write_header_kernel(TrainHeader hd, TrainHeader *dst) { *dst = hd; }

// x[r] = [xyz[r] | noise[r]]
__global__ void concat_inputs_kernel(const float *__restrict__ xyz, const float *__restrict__ noise, int nd, long long M, float *__restrict__ x)
{
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int w = 3 + nd;
    if (idx >= M * w) return;
    const long long r = idx / w;
    const int k = (int)(idx % w);
    x[idx] = k < 3 ? xyz[r * 3 + k] : noise[r * nd + k - 3];
}

static ChainIO train_io(nphm_mlp *h, uint8_t *ws, const TrainLayout &t, int nd)
{
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    ChainIO io;
    io.x = reinterpret_cast<const float *>(ws + t.x);
    io.xw = 3 + nd;
    for (int l = 0; l < s.n_lin; ++l) {
        io.fwd[l] = &train_fwd(c, s, l, nd);
        if (l + 1 == s.n_lin) break;
        io.Hp[l] = ws + t.hp[l];
        io.S[l] = reinterpret_cast<float *>(ws + t.s[l]);
    }
    return io;
}

}  // namespace chain
}  // namespace nphm

static int train_args(nphm_mlp *h, const char *who, const float *xyz_dev, const float *cond_dev, const float *noise_dev, int noise_dim,
                      int n_queries, long long n_points, void *workspace_dev)
{
    int rc = chain_ready(h, who);
    if (rc) return rc;
    NPHM_REQUIRE(n_queries >= 1 && n_points >= 1, "%s: bad sizes", who);
    NPHM_REQUIRE(noise_dim >= 0 && noise_dim <= std::min(h->dims.cond_dim, chain::kMaxNoise),
                 "%s: noise width %d outside [0, %d]", who, noise_dim, std::min(h->dims.cond_dim, chain::kMaxNoise));
    NPHM_REQUIRE(xyz_dev && cond_dev && workspace_dev && (noise_dim == 0 || noise_dev), "%s: NULL pointer", who);
    return NPHM_OK;
}

extern "C" long long nphm_mlp_train_workspace_bytes(const nphm_mlp *h, int n_queries, long long n_points, int noise_dim)
{
    if (!h || n_queries < 1 || n_points < 1 || noise_dim < 0 || noise_dim > std::min(h->dims.cond_dim, chain::kMaxNoise)) {
        set_error("nphm_mlp_train_workspace_bytes: bad arguments");
        return -1;
    }
    return (long long)chain::train_layout(h->dims, (long long)n_queries * n_points, noise_dim).total;
}

extern "C" int nphm_mlp_forward_train(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, const float *noise_dev, int noise_dim,
                                      int n_queries, long long n_points, float *out_dev, void *workspace_dev, void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int rc = train_args(h, "nphm_mlp_forward_train", xyz_dev, cond_dev, noise_dev, noise_dim, n_queries, n_points, workspace_dev);
    if (rc) return rc;
    NPHM_REQUIRE(out_dev, "nphm_mlp_forward_train: NULL output");
    const long long M = (long long)n_queries * n_points;
    const chain::TrainLayout t = chain::train_layout(h->dims, M, noise_dim);
    uint8_t *ws = static_cast<uint8_t *>(workspace_dev);
    if ((rc = chain::train_pack(h, noise_dim, stream))) return rc;
    if ((rc = mlp_prepare(h, cond_dev, n_queries, stream))) return rc;
    chain::concat_inputs_kernel<<<(unsigned)ceil_div(M * (3 + noise_dim), 256), 256, 0, stream>>>(xyz_dev, noise_dev, noise_dim, M,
                                                                                                   reinterpret_cast<float *>(ws + t.x));
    NPHM_CUDA_CHECK(cudaGetLastError());
    if ((rc = value_pass_io(h, chain::train_io(h, ws, t, noise_dim), n_queries, n_points, out_dev, stream))) return rc;
    const chain::TrainHeader hd{chain::kTrainMagic, h->weight_gen, h, M, n_points, n_queries, noise_dim};
    chain::write_header_kernel<<<1, 1, 0, stream>>>(hd, reinterpret_cast<chain::TrainHeader *>(ws));
    NPHM_CUDA_CHECK(cudaGetLastError());
    return NPHM_OK;
}

extern "C" int nphm_mlp_backward_train(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, const float *noise_dev, int noise_dim,
                                       int n_queries, long long n_points, const float *grad_out_dev, float *const *grad_w_dev,
                                       float *const *grad_b_dev, float *grad_cond_dev, float *grad_xyz_dev, void *workspace_dev,
                                       void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    int rc = train_args(h, "nphm_mlp_backward_train", xyz_dev, cond_dev, noise_dev, noise_dim, n_queries, n_points, workspace_dev);
    if (rc) return rc;
    NPHM_REQUIRE(grad_out_dev, "nphm_mlp_backward_train: NULL grad_out");
    MlpChain &c = *h->chain;
    const StackDims &s = h->dims;
    const long long M = (long long)n_queries * n_points;
    const int L = s.n_lin - 1;
    uint8_t *ws = static_cast<uint8_t *>(workspace_dev);
    const int out_dim = s.N[L];
    // The adjoints travel between the layers as fp16 hi + lo pairs, whose lo half (and, for tiny values, the hi half) is subnormal
    // below 6e-5: a training loss's grad_out (~1e-5 and less) would lose most of its digits.  The pass runs on grad_out scaled by a
    // power of two that brings max |grad_out| to [512, 1024); every output is scaled back exactly.
    if ((rc = c.wg_flags.reserve(2 * sizeof(unsigned int)))) return rc;
    unsigned int *const flags = c.wg_flags.as<unsigned int>(), *const bad = flags + 1;
    NPHM_CUDA_CHECK(cudaMemsetAsync(flags, 0, 2 * sizeof(unsigned int), stream));
    if ((rc = wg::abs_max(grad_out_dev, M * out_dim, flags, stream))) return rc;
    chain::TrainHeader hd;
    unsigned int gmax_bits = 0;
    NPHM_CUDA_CHECK(cudaMemcpyAsync(&hd, ws, sizeof(hd), cudaMemcpyDeviceToHost, stream));
    NPHM_CUDA_CHECK(cudaMemcpyAsync(&gmax_bits, flags, sizeof(gmax_bits), cudaMemcpyDeviceToHost, stream));
    NPHM_CUDA_CHECK(cudaStreamSynchronize(stream));
    NPHM_REQUIRE(hd.magic == chain::kTrainMagic && hd.handle == h,
                 "nphm_mlp_backward_train: the workspace does not hold a training forward of this network");
    NPHM_REQUIRE(hd.rows == M && hd.n_points == n_points && hd.n_queries == n_queries && hd.noise_dim == noise_dim,
                 "nphm_mlp_backward_train: the workspace holds a forward of %d x %lld points (noise %d), not %d x %lld (noise %d)",
                 hd.n_queries, hd.n_points, hd.noise_dim, n_queries, n_points, noise_dim);
    NPHM_REQUIRE(hd.weight_gen == h->weight_gen, "nphm_mlp_backward_train: the workspace holds a forward of older weights");
    if (!grad_w_dev && !grad_b_dev && !grad_cond_dev && !grad_xyz_dev) return NPHM_OK;
    float gmax;
    memcpy(&gmax, &gmax_bits, sizeof(gmax));
    NPHM_REQUIRE(std::isfinite(gmax), "nphm_mlp_backward_train: grad_out is not finite");
    int e = 0;
    if (gmax > 0.f) std::frexp(gmax, &e);
    e = std::max(-100, std::min(100, 10 - e));
    const float up = std::ldexp(1.0f, e), down = std::ldexp(1.0f, -e);
    if ((rc = c.wg_grad.reserve((size_t)M * out_dim * sizeof(float)))) return rc;
    if ((rc = wg::scale(grad_out_dev, M * out_dim, up, c.wg_grad.as<float>(), nullptr, stream))) return rc;
    const chain::TrainLayout t = chain::train_layout(s, M, noise_dim);
    const ChainIO io = chain::train_io(h, ws, t, noise_dim);
    const int xw = io.xw;
    const bool cond_w0 = grad_w_dev && grad_w_dev[0], cond_ws = grad_w_dev && grad_w_dev[s.skip];
    if (cond_w0 && (rc = c.wg_sums0.reserve((size_t)n_queries * s.N[0] * sizeof(float)))) return rc;
    if (cond_ws && (rc = c.wg_sumss.reserve((size_t)n_queries * s.N[s.skip] * sizeof(float)))) return rc;
    // dW_l = sum_rows d_l^T in_l while d_l is alive, and the fixed-order per-query sums of d_0 / d_skip for the condition columns
    auto on_layer = [&](int l, const Adjoint &d) -> int {
        float *gw = grad_w_dev ? grad_w_dev[l] : nullptr, *gb = grad_b_dev ? grad_b_dev[l] : nullptr;
        int rc2 = NPHM_OK;
        if (l == L) {                                             // d_L = grad_out (row-major, out_dim wide): skinny, unscaled
            if (gw && (rc2 = wg::packed_rows(io.Hp[L - 1], io.fwd[L]->ksteps, s.N[L - 1], grad_out_dev, out_dim, out_dim, M, 1.0f, gw,
                                             s.in_total[L], true, nullptr, c.wg_scratch, bad, stream))) return rc2;
            if (gb) rc2 = wg::rows_column_sums(grad_out_dev, out_dim, out_dim, M, gb, stream);
            return rc2;
        }
        if (l == 0) {                                             // [xyz | noise] columns and the bias: skinny
            if ((gw || gb) && (rc2 = wg::packed_rows(d.packed, d.ksteps, d.width, io.x, xw, gw ? xw : 0, M, down, gw, s.in_total[0], false,
                                                     gb, c.wg_scratch, bad, stream))) return rc2;
            if (cond_w0) rc2 = wg::range_sums(d.packed, d.ksteps, d.width, M, n_points, c.wg_sums0.as<float>(), stream);
            return rc2;
        }
        if (gw && (rc2 = wg::packed_packed(d.packed, d.ksteps, d.width, io.Hp[l - 1], io.fwd[l]->ksteps, io.fwd[l]->K, M,
                                           (l == s.skip ? chain::kInvSqrt2 : 1.0f) * down, gw, s.in_total[l], c.wg_scratch, bad, stream)))
            return rc2;
        if (gb && (rc2 = wg::packed_rows(d.packed, d.ksteps, d.width, nullptr, 0, 0, M, down, nullptr, 0, false, gb, c.wg_scratch,
                                         bad, stream))) return rc2;
        if (l == s.skip && cond_ws) rc2 = wg::range_sums(d.packed, d.ksteps, d.width, M, n_points, c.wg_sumss.as<float>(), stream);
        return rc2;
    };
    if ((rc = adjoint_pass(h, M, n_points, c.wg_grad.as<float>(), io.S, grad_cond_dev, grad_xyz_dev, on_layer, stream))) return rc;
    if (grad_cond_dev && (rc = wg::scale(grad_cond_dev, (long long)n_queries * s.cond_dim, down, grad_cond_dev, bad, stream))) return rc;
    if (grad_xyz_dev && (rc = wg::scale(grad_xyz_dev, M * 3, down, grad_xyz_dev, bad, stream))) return rc;
    // condition columns: sum_q (sum_{p in q} d[p]) (x) cond_q, added to the noise columns (their input was cond + noise)
    if (cond_w0 && (rc = wg::cond_columns(c.wg_sums0.as<float>(), s.N[0], cond_dev, s.cond_dim, n_queries, down, noise_dim, grad_w_dev[0],
                                          s.in_total[0], 3, bad, stream))) return rc;
    if (cond_ws && (rc = wg::cond_columns(c.wg_sumss.as<float>(), s.N[s.skip], cond_dev, s.cond_dim, n_queries, chain::kInvSqrt2 * down,
                                          noise_dim, grad_w_dev[s.skip], s.in_total[s.skip], s.N[s.skip - 1] + 3, bad, stream))) return rc;
    // an adjoint beyond the fp16 range of the packed format (65504, 64x above the scaled grad_out) shows up as a non-finite output:
    // report it instead of handing inf / NaN to the optimiser
    unsigned int bad_host = 0;
    NPHM_CUDA_CHECK(cudaMemcpyAsync(&bad_host, bad, sizeof(bad_host), cudaMemcpyDeviceToHost, stream));
    NPHM_CUDA_CHECK(cudaStreamSynchronize(stream));
    NPHM_REQUIRE(!bad_host, "nphm_mlp_backward_train: non-finite gradient (an adjoint exceeded the fp16 range of the packed format, "
                            "or the weights / inputs are not finite)");
    return NPHM_OK;
}
