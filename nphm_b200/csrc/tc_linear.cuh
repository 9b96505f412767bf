// Generic fp32-accurate tcgen05 linear layer (tc_linear.cu): parameters, packed weights, launch.
#pragma once
#include "engine.cuh"
#include "tc_common.cuh"

namespace nphm {
namespace tcl {

constexpr int kModeLinear = 0, kModeSoftplus = 1, kModeMult = 2;

struct LinearParams {
    const float *A1 = nullptr; int lda1 = 0; int K1 = 0;     // [M x K1] fp32 row-major (may be absent: K1 = 0)
    const float *A2 = nullptr; int lda2 = 0; int K2 = 0;     // optional second input appended along K
    int a2_onehot = 0;                                       // A2 is not read: row r contributes e_{r mod K2}
    long long M = 0;
    const float *bias = nullptr; int ldb = 0; long long rows_per_bias = 0;   // bias row = row / rows_per_bias (0: one row for all)
    int mode = kModeLinear;
    float *C = nullptr; int ldc = 0;
    float *Dv = nullptr; int lddv = 0;                       // SOFTPLUS: derivative of the activation (optional)
    const float *Mul = nullptr; int ldmul = 0; long long mul_div = 1;        // MULT: C = t * Mul[row / mul_div][n]
    const float *row_scale = nullptr;                        // MULT: additional factor row_scale[row]
    int mul_blocked = 0, dv_blocked = 0;                     // Mul / Dv alone in the blocked layout (see `blocked`)
    // operand-ready ("packed") activations: per 128-row tile and k-step 8 KB = [128 x 16 fp16 hi | 128 x 16 fp16 lo] in UMMA core-
    // matrix order.  Cp: the epilogue writes its output split like that (unit u of 16 columns = k-step u of the next layer), so
    // the next launch takes it as Ap with one bulk copy per k-step and no conversion work in its main loop.
    const uint8_t *Ap = nullptr; int a_ksteps = 0; long long sAp = 0;        // replaces A1 / A2; 16 a_ksteps = packed K
    uint8_t *Cp = nullptr; int c_ksteps = 0; long long sCp = 0;              // optional, in addition to / instead of C
    int a_tile_steps = 0, c_tile_steps = 0;                  // pitch between the tiles in k-steps (default: a_ksteps / c_ksteps)
    // columns appended behind the layer's N outputs in Cp (the next layer's `cat([h, xyz])`): app[row][0..app_w) or, one-hot,
    // e_{row mod app_w} (the tangent seeds of a forward-mode pass)
    const float *app = nullptr; int app_ld = 0, app_w = 0, app_onehot = 0;
    int blocked = 0;                                         // A1 / Mul / C in 128-row tiles, feature-major inside a tile:
                                                             // (row, k) at (row / 128) * ld * 128 + k * 128 + row % 128
    // batched launch (gridDim.z): entry z reads A1 + z sA1, Mul + z sMul, row_scale + z sRow, writes C + z sC (strides in floats)
    // and uses weight set z/2 for z < 2 w_pairs, z - w_pairs beyond (the mirrored pairs of the ensemble share weights)
    int batch = 1; long long sA1 = 0, sC = 0, sMul = 0, sRow = 0; int w_pairs = 0;
    // filled by launch_linear from the packed weights
    const uint8_t *W = nullptr; long long w_stride = 0; int N = 0, Nt = 0, ksteps = 0, stages = 0;
};

struct PackedLinear {
    DeviceBuffer slabs;
    int N = 0, K = 0, Nt = 0, n_tiles = 0, ksteps = 0, sets = 1;
    size_t set_bytes = 0;
    // B[n][k] = scale * k_scale[k] * (transpose ? W[k_off + k][n_off + n] : W[n_off + n][k_off + k]),  n < N, k < K;
    // `sets` matrices W + s * w_set_stride (k_scale + s * k_scale_stride) packed back to back
    // n_extra: output columns reserved behind N in the tiling (LinearParams::app)
    int pack(const float *W_dev, int ldw, int N, int K, int n_off, int k_off, bool transpose, float scale, cudaStream_t stream,
             int sets = 1, long long w_set_stride = 0, const float *k_scale_dev = nullptr, long long k_scale_stride = 0,
             int n_extra = 0, int max_nt = 0);      // max_nt: widest output tile (default 256); narrower = more CTAs for few rows
    int packed_ksteps_out() const { return (N + n_extra + 15) / 16; }       // k-steps of the packed output (Cp) of this layer
    int n_extra = 0;
};

int launch_linear(const PackedLinear &w, LinearParams p, cudaStream_t stream);

}  // namespace tcl

// Weight gradients over the rows of a batch (tc_wgrad.cu).  Deterministic: per-row-range partials in `scratch`, summed in order.
// `bad` (optional, device): set to non-zero when a written output is not finite.
namespace wg {
// dst[n][k] = scale * sum_r D[r][n] A[r][k], n < N, k < K; D and A packed (tcgen05)
int packed_packed(const uint8_t *D, int d_ksteps, int N, const uint8_t *A, int a_ksteps, int K, long long M, float scale, float *dst,
                  int ld_dst, DeviceBuffer &scratch, unsigned int *bad, cudaStream_t stream);
// skinny products, SIMT: dst_w[p][w] (transpose: dst_w[w][p]) = scale * sum_r P[r][p] R[r][w], w < Wr (P packed, R row-major);
// dst_ones[p] = scale * sum_r P[r][p] (optional)
int packed_rows(const uint8_t *P, int p_ksteps, int Pw, const float *R, int ldr, int Wr, long long M, float scale, float *dst_w, int ld_w,
                bool transpose, float *dst_ones, DeviceBuffer &scratch, unsigned int *bad, cudaStream_t stream);
// out[range][p] = sum of P[r][p] over the rows of each range of rows_per_range rows (P packed), fixed order
int range_sums(const uint8_t *P, int p_ksteps, int Pw, long long M, long long rows_per_range, float *out, cudaStream_t stream);
// *out_dev = bit pattern of max |x|;  y = s * x
int abs_max(const float *x, long long n, unsigned int *out_dev, cudaStream_t stream);
int scale(const float *x, long long n, float s, float *y, unsigned int *bad, cudaStream_t stream);
// out[w] = sum_r R[r][w]  (R row-major)
int rows_column_sums(const float *R, int ldr, int W, long long M, float *out, cudaStream_t stream);
// dst[n][col0 + j] = scale * sum_q S[q][n] cond[q][j]  (added to what is there for j < n_add)
int cond_columns(const float *S, int N, const float *cond, int cond_dim, int Q, float scale, int n_add, float *dst, int ld, int col0,
                 unsigned int *bad, cudaStream_t stream);
}  // namespace wg
}  // namespace nphm
