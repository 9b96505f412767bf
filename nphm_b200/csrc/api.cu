// C ABI of libnphm_b200.so: handles, weight packing, query entry points (see include/nphm_b200.h).
#include "engine.cuh"
#include <cstring>
#include <cmath>
#include <vector>

namespace nphm {

static thread_local char g_error[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int sm_count()
{
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev < 64 && cached[dev]) return cached[dev];
    int n = 148;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (dev < 64) cached[dev] = n;
    return n;
}

int DeviceBuffer::reserve(size_t bytes)
{
    if (bytes <= cap) return NPHM_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr; cap = 0;
    const size_t want = bytes + bytes / 4 + 256;
    NPHM_CUDA_CHECK(cudaMalloc(&ptr, want));
    cap = want;
    return NPHM_OK;
}
DeviceBuffer::~DeviceBuffer() { if (ptr) cudaFree(ptr); }

// Build the folded description of a DeepSDF-style stack: n_lin = n_layers + 1 linear layers, widths
// [d_in, hidden x n_layers, out_dim], the layer before `skip` is narrowed by d_in (reference
// EnsembledDeepSDF.py:80-96 / deepSDF.py:38-55), d_in = 3 + cond_dim.
int build_stack(StackDims &s, int cond_dim, int hidden, int n_layers, int out_dim)
{
    NPHM_REQUIRE(n_layers >= 2 && n_layers + 1 <= kMaxLayers, "unsupported number of layers %d", n_layers);
    NPHM_REQUIRE(hidden > cond_dim + 3, "hidden_dim %d must exceed 3 + condition width %d", hidden, cond_dim);
    s.n_lin = n_layers + 1;
    s.skip = n_layers / 2;
    s.cond_dim = cond_dim;
    const int d_in = 3 + cond_dim;
    int coff = 0, max_rows = 8;
    for (int l = 0; l < s.n_lin; ++l) {
        int in_w = l == 0 ? d_in : hidden;
        int out_w = l == s.n_lin - 1 ? out_dim : hidden;
        if (l + 1 == s.skip) out_w -= d_in;
        s.in_total[l] = in_w;
        s.N[l] = out_w;
        s.Npad[l] = round_up(out_w, 8);
        if (l == 0) { s.K[l] = 3; s.folded[l] = 1; s.scale[l] = 1.0f; }
        else if (l == s.skip) { s.K[l] = s.N[l - 1] + 3; s.folded[l] = 1; s.scale[l] = (float)(1.0 / std::sqrt(2.0)); }
        else { s.K[l] = in_w; s.folded[l] = 0; s.scale[l] = 1.0f; }
        s.coff[l] = coff;
        coff += s.Npad[l];
        max_rows = std::max(max_rows, std::max(s.K[l], s.N[l] + 3));
    }
    s.cvec_stride = coff;
    s.max_rows = std::max(max_rows, 8 + 8 * 8);     // narrow_layer scratch rows
    return NPHM_OK;
}

int NetWeights::load(const StackDims &s, int n_sets, const float *const *w_dev, const float *const *b_dev,
                     cudaStream_t stream)
{
    for (int l = 0; l < s.n_lin; ++l) {
        NPHM_REQUIRE(w_dev[l] && b_dev[l], "layer %d: NULL weight/bias pointer", l);
        const size_t wb = (size_t)n_sets * s.N[l] * s.in_total[l] * sizeof(float);
        const size_t bb = (size_t)n_sets * s.N[l] * sizeof(float);
        int rc;
        if ((rc = W[l].reserve(wb))) return rc;
        if ((rc = b[l].reserve(bb))) return rc;
        if ((rc = Wt[l].reserve((size_t)n_sets * s.K[l] * s.Npad[l] * sizeof(float)))) return rc;
        NPHM_CUDA_CHECK(cudaMemcpyAsync(W[l].ptr, w_dev[l], wb, cudaMemcpyDeviceToDevice, stream));
        NPHM_CUDA_CHECK(cudaMemcpyAsync(b[l].ptr, b_dev[l], bb, cudaMemcpyDeviceToDevice, stream));
        if ((rc = launch_pack_wt(W[l].as<float>(), n_sets, s.N[l], s.in_total[l], s.K[l], s.Npad[l], s.scale[l],
                                 Wt[l].as<float>(), stream))) return rc;
    }
    return NPHM_OK;
}

void fill_descriptors(const StackDims &s, const NetWeights &w, int n_members, int n_symm, int lat_dim, int lat_glob,
                      int lat_loc, FoldedNet &net, PackSpec &spec)
{
    net.n_layers = s.n_lin; net.skip = s.skip; net.n_members = n_members; net.n_symm = n_symm;
    net.cvec_stride = s.cvec_stride; net.max_rows = s.max_rows;
    spec.n_layers = s.n_lin; spec.n_members = n_members; spec.n_symm = n_symm;
    spec.lat_dim = lat_dim; spec.lat_glob = lat_glob; spec.lat_loc = lat_loc; spec.cond_dim = s.cond_dim;
    spec.cvec_stride = s.cvec_stride;
    for (int l = 0; l < s.n_lin; ++l) {
        net.L[l] = FoldedLayer{w.Wt[l].as<float>(), s.K[l], s.N[l], s.Npad[l], s.coff[l], l < s.n_lin - 1 ? 1 : 0};
        spec.L[l] = PackLayer{w.W[l].as<float>(), w.b[l].as<float>(), s.N[l], s.Npad[l], s.in_total[l], s.K[l],
                              s.folded[l], s.scale[l], s.coff[l]};
    }
}

}  // namespace nphm

using namespace nphm;

extern "C" const char *nphm_last_error(void) { return g_error; }
extern "C" int nphm_abi_version(void) { return 1; }

extern "C" int nphm_device_info(int *sms, int *major, int *minor)
{
    int dev = 0;
    NPHM_CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    NPHM_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    if (sms) *sms = prop.multiProcessorCount;
    if (major) *major = prop.major;
    if (minor) *minor = prop.minor;
    return NPHM_OK;
}

// ------------------------------------------------------------------------------------------------ ensemble
extern "C" int nphm_ensemble_create(const nphm_ensemble_config *cfg, nphm_ensemble **out)
{
    NPHM_REQUIRE(cfg && out, "nphm_ensemble_create: NULL argument");
    NPHM_REQUIRE(cfg->n_loc >= 1 && cfg->n_symm_pairs >= 0 && 2 * cfg->n_symm_pairs <= cfg->n_loc,
                 "nphm_ensemble_create: bad anchor counts n_loc=%d n_symm_pairs=%d", cfg->n_loc, cfg->n_symm_pairs);
    NPHM_REQUIRE(cfg->lat_dim_glob > 0 && cfg->lat_dim_loc > 0 && cfg->hidden_dim > 0 && cfg->pos_mlp_dim > 0,
                 "nphm_ensemble_create: non-positive width");
    auto *h = new nphm_ensemble();
    h->cfg = *cfg;
    h->n_members = cfg->n_loc + 1;
    h->n_sets = h->n_members - cfg->n_symm_pairs;
    h->lat_dim = cfg->lat_dim_glob + h->n_members * cfg->lat_dim_loc;
    int rc = build_stack(h->dims, cfg->lat_dim_glob + cfg->lat_dim_loc, cfg->hidden_dim, cfg->n_layers, 1);
    if (rc) { delete h; return rc; }
    *out = h;
    return NPHM_OK;
}

extern "C" void nphm_ensemble_destroy(nphm_ensemble *h)
{
    if (h) nphm::fit_packs_destroy(h);
    delete h;
}

extern "C" int nphm_ensemble_set_prune_threshold(nphm_ensemble *h, float tau)
{
    NPHM_REQUIRE(h && tau >= 0.f && tau < 1.f, "nphm_ensemble_set_prune_threshold: tau must be in [0, 1)");
    h->tc_prune_tau = tau;
    return NPHM_OK;
}

extern "C" int nphm_ensemble_load_weights(nphm_ensemble *h, const float *const *lin_w, const float *const *lin_b,
                                          const float *const *pos_w, const float *const *pos_b,
                                          const float *mean_anchors, void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    NPHM_REQUIRE(h && lin_w && lin_b && pos_w && pos_b && mean_anchors, "nphm_ensemble_load_weights: NULL argument");
    int rc = h->weights.load(h->dims, h->n_sets, lin_w, lin_b, stream);
    if (rc) return rc;
    const int G = h->cfg.lat_dim_glob, H = h->cfg.pos_mlp_dim, O = h->cfg.n_loc * 3;
    const size_t wsz[3] = {(size_t)H * G, (size_t)H * H, (size_t)O * H}, bsz[3] = {(size_t)H, (size_t)H, (size_t)O};
    for (int i = 0; i < 3; ++i) {
        NPHM_REQUIRE(pos_w[i] && pos_b[i], "nphm_ensemble_load_weights: NULL mlp_pos pointer");
        if ((rc = h->pos_w[i].reserve(wsz[i] * 4))) return rc;
        if ((rc = h->pos_b[i].reserve(bsz[i] * 4))) return rc;
        NPHM_CUDA_CHECK(cudaMemcpyAsync(h->pos_w[i].ptr, pos_w[i], wsz[i] * 4, cudaMemcpyDeviceToDevice, stream));
        NPHM_CUDA_CHECK(cudaMemcpyAsync(h->pos_b[i].ptr, pos_b[i], bsz[i] * 4, cudaMemcpyDeviceToDevice, stream));
    }
    if ((rc = h->mean_anchors.reserve((size_t)O * 4))) return rc;
    NPHM_CUDA_CHECK(cudaMemcpyAsync(h->mean_anchors.ptr, mean_anchors, (size_t)O * 4, cudaMemcpyDeviceToDevice, stream));
    fill_descriptors(h->dims, h->weights, h->n_members, h->cfg.n_symm_pairs, h->lat_dim, h->cfg.lat_dim_glob,
                     h->cfg.lat_dim_loc, h->net, h->spec);
    rc = tc_ensemble_pack(h, stream);
    if (rc) return rc;
    fit_packs_destroy(h);                      // packed from the previous weights, rebuilt by the next fitting call
    h->loaded = true;
    return NPHM_OK;
}

namespace nphm {
// per-query constants: anchors, cvec (SIMT) and the tensor-core constants when that kernel is used
int ensemble_prepare(nphm_ensemble *h, const float *latents_dev, int n_queries, cudaStream_t stream)
{
    int rc;
    if ((rc = h->anchors.reserve((size_t)n_queries * h->cfg.n_loc * 3 * sizeof(float)))) return rc;
    if ((rc = h->cvec.reserve((size_t)n_queries * h->n_members * h->dims.cvec_stride * sizeof(float)))) return rc;
    const float *pw[3] = {h->pos_w[0].as<float>(), h->pos_w[1].as<float>(), h->pos_w[2].as<float>()};
    const float *pb[3] = {h->pos_b[0].as<float>(), h->pos_b[1].as<float>(), h->pos_b[2].as<float>()};
    if ((rc = launch_anchors(latents_dev, n_queries, h->lat_dim, h->cfg.lat_dim_glob, h->cfg.pos_mlp_dim,
                             h->cfg.n_loc * 3, pw, pb, h->mean_anchors.as<float>(), h->anchors.as<float>(), stream)))
        return rc;
    return launch_cvec(h->spec, latents_dev, n_queries, h->cvec.as<float>(), stream);
}

}  // namespace nphm (closed for the C entry below)

// anchors = mlp_pos(z_glob) + mean anchors of n_queries latent codes (reference src/NPHM/models/EnsembledDeepSDF.py:228-229) without
// evaluating the ensemble: what the fitters obtain by `decoder(zeros(1,1,3), lat)[1]` (fitting.py:59, :211).
extern "C" int nphm_ensemble_anchors(nphm_ensemble *h, const float *latents_dev, int n_queries, float *out_anchors_dev, void *stream_)
{
    using namespace nphm;
    NPHM_REQUIRE(h && h->loaded && latents_dev && out_anchors_dev && n_queries >= 1, "nphm_ensemble_anchors: bad arguments");
    const float *pw[3] = {h->pos_w[0].as<float>(), h->pos_w[1].as<float>(), h->pos_w[2].as<float>()};
    const float *pb[3] = {h->pos_b[0].as<float>(), h->pos_b[1].as<float>(), h->pos_b[2].as<float>()};
    return launch_anchors(latents_dev, n_queries, h->lat_dim, h->cfg.lat_dim_glob, h->cfg.pos_mlp_dim, h->cfg.n_loc * 3, pw, pb,
                          h->mean_anchors.as<float>(), out_anchors_dev, static_cast<cudaStream_t>(stream_));
}

namespace nphm {
static int pick_impl(nphm_ensemble *h, int impl, bool *use_tc)
{
    NPHM_REQUIRE(impl == NPHM_IMPL_AUTO || impl == NPHM_IMPL_SIMT || impl == NPHM_IMPL_TC || impl == NPHM_IMPL_TC_PRUNED,
                 "unknown impl %d", impl);
    const bool tc_ok = tc_ensemble_supported(h);
    h->tc_prune = impl == NPHM_IMPL_TC_PRUNED;
    if (impl == NPHM_IMPL_TC_PRUNED) impl = NPHM_IMPL_TC;
    if (impl == NPHM_IMPL_TC && !tc_ok) {
        set_error("tcgen05 ensemble kernel does not support this configuration");
        return NPHM_ERR_UNSUPPORTED;
    }
    *use_tc = impl == NPHM_IMPL_TC || (impl == NPHM_IMPL_AUTO && tc_ok);
    return NPHM_OK;
}

static int ensemble_run(nphm_ensemble *h, SimtQuery &q, const float *latents_dev, float *out_anchors_dev, int impl,
                        cudaStream_t stream)
{
    NPHM_REQUIRE(h && h->loaded, "ensemble: weights not loaded");
    bool use_tc = false;
    int rc = pick_impl(h, impl, &use_tc);
    if (rc) return rc;
    if ((rc = ensemble_prepare(h, latents_dev, q.n_queries, stream))) return rc;
    q.cvec = h->cvec.as<float>();
    q.anchors = h->anchors.as<float>();
    q.blend = 1;
    if (q.n_points > 0) {
        rc = use_tc ? tc_ensemble_launch(h, q, stream) : launch_folded_net(h->net, q, stream);
        if (rc) return rc;
    }
    if (out_anchors_dev)
        NPHM_CUDA_CHECK(cudaMemcpyAsync(out_anchors_dev, h->anchors.ptr, (size_t)q.n_queries * h->cfg.n_loc * 3 * 4,
                                        cudaMemcpyDeviceToDevice, stream));
    return NPHM_OK;
}
}  // namespace nphm

extern "C" int nphm_ensemble_query(nphm_ensemble *h, const float *xyz_dev, const float *latents_dev, int n_queries,
                                   long long n_points, long long quirk_period, float *out_sdf_dev,
                                   float *out_anchors_dev, int impl, void *stream_)
{
    NPHM_REQUIRE(h, "nphm_ensemble_query: NULL handle");
    NPHM_REQUIRE(n_queries >= 1 && n_points >= 0 && quirk_period >= 0, "nphm_ensemble_query: bad sizes");
    NPHM_REQUIRE(latents_dev && (n_points == 0 || (xyz_dev && out_sdf_dev)), "nphm_ensemble_query: NULL pointer");
    SimtQuery q{};
    q.xyz = xyz_dev; q.axes = nullptr; q.res = 0; q.first = 0; q.total = n_points; q.n_points = n_points;
    q.n_queries = n_queries; q.quirk_period = quirk_period; q.out = out_sdf_dev;
    return ensemble_run(h, q, latents_dev, out_anchors_dev, impl, static_cast<cudaStream_t>(stream_));
}

extern "C" int nphm_ensemble_query_grid(nphm_ensemble *h, const float *latent_dev, const double gmin[3],
                                        const double gmax[3], int res, long long first, long long count,
                                        long long quirk_period, float *out_sdf_dev, float *out_anchors_dev, int impl,
                                        void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    NPHM_REQUIRE(h, "nphm_ensemble_query_grid: NULL handle");
    NPHM_REQUIRE(res >= 2 && res <= 2048, "nphm_ensemble_query_grid: res %d out of range", res);
    const long long total = (long long)res * res * res;
    NPHM_REQUIRE(first >= 0 && count >= 0 && first + count <= total && quirk_period >= 0,
                 "nphm_ensemble_query_grid: range [%lld, %lld) outside the %d^3 grid", first, first + count, res);
    NPHM_REQUIRE(latent_dev && gmin && gmax && (count == 0 || out_sdf_dev), "nphm_ensemble_query_grid: NULL pointer");
    int rc;
    if ((rc = h->axes.reserve((size_t)3 * res * sizeof(float)))) return rc;
    if ((rc = launch_grid_axes(gmin, gmax, res, h->axes.as<float>(), stream))) return rc;
    SimtQuery q{};
    q.xyz = nullptr; q.axes = h->axes.as<float>(); q.res = res; q.first = first; q.total = total;
    q.n_points = count; q.n_queries = 1; q.quirk_period = quirk_period; q.out = out_sdf_dev;
    return ensemble_run(h, q, latent_dev, out_anchors_dev, impl, stream);
}

extern "C" int nphm_ensemble_get_logits_host(nphm_ensemble *h, const float *latent_host, const double gmin[3],
                                             const double gmax[3], int res, long long quirk_period, float *out_host,
                                             int impl)
{
    NPHM_REQUIRE(h && latent_host && out_host, "nphm_ensemble_get_logits_host: NULL argument");
    const long long total = (long long)res * res * res;
    int rc;
    if ((rc = h->host_latent.reserve((size_t)h->lat_dim * 4))) return rc;
    if ((rc = h->host_volume.reserve((size_t)total * 4))) return rc;
    NPHM_CUDA_CHECK(cudaMemcpyAsync(h->host_latent.ptr, latent_host, (size_t)h->lat_dim * 4, cudaMemcpyHostToDevice, 0));
    rc = nphm_ensemble_query_grid(h, h->host_latent.as<float>(), gmin, gmax, res, 0, total, quirk_period,
                                  h->host_volume.as<float>(), nullptr, impl, nullptr);
    if (rc) return rc;
    NPHM_CUDA_CHECK(cudaMemcpyAsync(out_host, h->host_volume.ptr, (size_t)total * 4, cudaMemcpyDeviceToHost, 0));
    NPHM_CUDA_CHECK(cudaStreamSynchronize(0));
    return NPHM_OK;
}

// ------------------------------------------------------------------------------------------------ plain MLP
extern "C" int nphm_mlp_create(const nphm_mlp_config *cfg, nphm_mlp **out)
{
    NPHM_REQUIRE(cfg && out, "nphm_mlp_create: NULL argument");
    NPHM_REQUIRE(cfg->lat_dim > 0 && cfg->hidden_dim > 0 && cfg->out_dim >= 1 && cfg->out_dim <= 8,
                 "nphm_mlp_create: unsupported widths (out_dim must be 1..8)");
    auto *h = new nphm_mlp();
    h->cfg = *cfg;
    int rc = build_stack(h->dims, cfg->lat_dim, cfg->hidden_dim, cfg->n_layers, cfg->out_dim);
    if (rc) { delete h; return rc; }
    *out = h;
    return NPHM_OK;
}

extern "C" void nphm_mlp_destroy(nphm_mlp *h)
{
    if (h) chain_destroy(h);
    delete h;
}

extern "C" int nphm_mlp_load_weights(nphm_mlp *h, const float *const *w_dev, const float *const *b_dev, void *stream_)
{
    NPHM_REQUIRE(h && w_dev && b_dev, "nphm_mlp_load_weights: NULL argument");
    int rc = h->weights.load(h->dims, 1, w_dev, b_dev, static_cast<cudaStream_t>(stream_));
    if (rc) return rc;
    ++h->weight_gen;
    fill_descriptors(h->dims, h->weights, 1, 0, h->cfg.lat_dim, 0, 0, h->net, h->spec);
    rc = tc_mlp_pack(h, static_cast<cudaStream_t>(stream_));
    if (rc) return rc;
    if (h->dims.skip >= 1 && h->dims.skip < h->dims.n_lin - 1) {       // stacks the layer chain can run (mlp_chain.cu)
        rc = chain_pack(h, static_cast<cudaStream_t>(stream_));
        if (rc) return rc;
    }
    h->loaded = true;
    return NPHM_OK;
}

namespace nphm {
// folded constants of the condition (one row per query); must precede mlp_run on the same stream
int mlp_prepare(nphm_mlp *h, const float *cond_dev, int n_queries, cudaStream_t stream)
{
    int rc;
    if ((rc = h->cvec.reserve((size_t)n_queries * h->dims.cvec_stride * sizeof(float)))) return rc;
    return launch_cvec(h->spec, cond_dev, n_queries, h->cvec.as<float>(), stream);
}

// point pass with the constants of the last mlp_prepare; impl AUTO = tensor-core kernel when the shape allows it
int mlp_run(nphm_mlp *h, const float *xyz_dev, int n_queries, long long n_points, float *out_dev, int impl, cudaStream_t stream)
{
    if (n_points == 0) return NPHM_OK;
    const bool use_tc = impl == NPHM_IMPL_TC || (impl == NPHM_IMPL_AUTO && tc_mlp_supported(h) && h->tc_ready);
    if (use_tc) return tc_mlp_launch(h, xyz_dev, h->cvec.as<float>(), n_queries, n_points, out_dev, stream);
    SimtQuery q{};
    q.xyz = xyz_dev; q.total = n_points; q.n_points = n_points; q.n_queries = n_queries; q.quirk_period = 0;
    q.cvec = h->cvec.as<float>(); q.anchors = nullptr; q.blend = 0; q.out = out_dev;
    return launch_folded_net(h->net, q, stream);
}
}  // namespace nphm

extern "C" int nphm_mlp_query(nphm_mlp *h, const float *xyz_dev, const float *cond_dev, int n_queries,
                              long long n_points, float *out_dev, int impl, void *stream_)
{
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    NPHM_REQUIRE(h && h->loaded, "nphm_mlp_query: weights not loaded");
    NPHM_REQUIRE(n_queries >= 1 && n_points >= 0, "nphm_mlp_query: bad sizes");
    NPHM_REQUIRE(cond_dev && (n_points == 0 || (xyz_dev && out_dev)), "nphm_mlp_query: NULL pointer");
    NPHM_REQUIRE(impl == NPHM_IMPL_AUTO || impl == NPHM_IMPL_SIMT || impl == NPHM_IMPL_TC, "nphm_mlp_query: unknown impl %d", impl);
    const bool tc_ok = tc_mlp_supported(h) && h->tc_ready;
    if (impl == NPHM_IMPL_TC && !tc_ok) {
        set_error("tcgen05 MLP kernel supports only the deformation backbone (hidden 512, 6 layers, condition 232, 3 outputs)");
        return NPHM_ERR_UNSUPPORTED;
    }
    const bool use_tc = impl == NPHM_IMPL_TC || (impl == NPHM_IMPL_AUTO && tc_ok);
    int rc;
    if ((rc = mlp_prepare(h, cond_dev, n_queries, stream))) return rc;
    return mlp_run(h, xyz_dev, n_queries, n_points, out_dev, use_tc ? NPHM_IMPL_TC : NPHM_IMPL_SIMT, stream);
}
