// Handle types behind the C ABI.
#pragma once
#include "common.cuh"
#include "simt.cuh"
#include <algorithm>

namespace nphm {

struct DeviceBuffer {
    void *ptr = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);          // grows (never shrinks); contents are NOT preserved on growth
    template <class T> T *as() const { return reinterpret_cast<T *>(ptr); }
    DeviceBuffer() = default;
    DeviceBuffer(const DeviceBuffer &) = delete;
    DeviceBuffer &operator=(const DeviceBuffer &) = delete;
    ~DeviceBuffer();
};

struct StackDims {
    int n_lin, skip, cond_dim, cvec_stride, max_rows;
    int in_total[kMaxLayers], N[kMaxLayers], Npad[kMaxLayers], K[kMaxLayers], folded[kMaxLayers], coff[kMaxLayers];
    float scale[kMaxLayers];
};

struct NetWeights {
    DeviceBuffer W[kMaxLayers], b[kMaxLayers];   // copies in the reference layout (used for the per-query constants)
    DeviceBuffer Wt[kMaxLayers];                 // SIMT layout [set][k][Npad]
    int load(const StackDims &s, int n_sets, const float *const *w_dev, const float *const *b_dev, cudaStream_t stream);
};

int build_stack(StackDims &s, int cond_dim, int hidden, int n_layers, int out_dim);
void fill_descriptors(const StackDims &s, const NetWeights &w, int n_members, int n_symm, int lat_dim, int lat_glob,
                      int lat_loc, FoldedNet &net, PackSpec &spec);

}  // namespace nphm

namespace nphm { namespace fit { struct BackwardPacks; } }

struct nphm_ensemble {
    nphm_ensemble_config cfg;
    int n_members = 0, n_sets = 0, lat_dim = 0;
    bool loaded = false;
    nphm::StackDims dims;
    nphm::NetWeights weights;
    nphm::FoldedNet net;
    nphm::PackSpec spec;
    nphm::DeviceBuffer pos_w[3], pos_b[3], mean_anchors;
    // per-call scratch
    nphm::DeviceBuffer anchors, cvec, axes, host_latent, host_volume;
    // tensor-core path (tc_ensemble.cu)
    nphm::DeviceBuffer tc_weights, tc_consts, tc_coff, tc_l2slabs;
    bool tc_ready = false;
    bool tc_prune = false;          // opt-in member pruning (NPHM_IMPL_TC_PRUNED)
    float tc_prune_tau = 1e-8f;
    // fitting (fit.cu)
    nphm::DeviceBuffer fit_scratch, fit_apply_scratch;
    nphm::fit::BackwardPacks *fit_packs = nullptr;      // adjoint weights of the backward GEMMs, built on first use
};

namespace nphm { struct MlpChain; }

struct nphm_mlp {
    nphm_mlp_config cfg;
    bool loaded = false;
    nphm::StackDims dims;
    nphm::NetWeights weights;
    nphm::FoldedNet net;
    nphm::PackSpec spec;
    nphm::DeviceBuffer cvec;
    // tensor-core path (tc_mlp.cu)
    nphm::DeviceBuffer tc_weights, tc_consts, tc_coff;
    bool tc_ready = false;
    const int *tc_live = nullptr;   // set around a launch by the Broyden loop: device counter, 0 = skip the evaluation
    bool tc_records_fresh = false;  // set by the Broyden loop after its first evaluation: the per-query records of the tensor-core
                                    // kernel are still those of this condition, do not rebuild them
    // layer-by-layer tensor-core passes: any width, Jacobian, adjoint (mlp_chain.cu)
    nphm::MlpChain *chain = nullptr;
    unsigned long long weight_gen = 0;   // bumped by every nphm_mlp_load_weights: training workspaces of older weights are refused
};

namespace nphm {
int ensemble_prepare(nphm_ensemble *h, const float *latents_dev, int n_queries, cudaStream_t stream);
// tensor-core ensemble kernel (tc_ensemble.cu)
bool tc_ensemble_supported(const nphm_ensemble *h);
int tc_ensemble_pack(nphm_ensemble *h, cudaStream_t stream);
int tc_ensemble_launch(nphm_ensemble *h, const SimtQuery &q, cudaStream_t stream);
// tensor-core MLP kernel (tc_mlp.cu): deformation backbone configuration only
bool tc_mlp_supported(const nphm_mlp *h);
int tc_mlp_pack(nphm_mlp *h, cudaStream_t stream);
int tc_mlp_launch(nphm_mlp *h, const float *xyz, const float *cvec, int n_queries, long long n_points, float *out,
                  cudaStream_t stream);
// fitting (fit.cu)
void fit_packs_destroy(nphm_ensemble *h);
// layer chain (mlp_chain.cu)
int chain_pack(nphm_mlp *h, cudaStream_t stream);
void chain_destroy(nphm_mlp *h);
int mlp_prepare(nphm_mlp *h, const float *cond_dev, int n_queries, cudaStream_t stream);
}  // namespace nphm
