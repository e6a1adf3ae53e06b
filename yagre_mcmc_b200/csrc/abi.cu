// abi.cu -- the extern "C" surface of libyagre_b200.so (include/yagre_b200.h).
// Plain pointers and sizes only; no torch types, no exceptions across the boundary.
#include "ensemble.h"
#include "big_linear.h"
#include "smem_plan.h"
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

int yg_pooled_impl(const double *w_mean, const double *w_m2, const unsigned long long *n_accept, int d, int64_t nc,
                   int64_t welford_n, double *partials, int n_part, double *out_dev, cudaStream_t st);

static thread_local char g_err[512] = "";

void yg_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {

constexpr int POOL_PARTS = 64;

// The per-chain state buffers, one row per StateBuf: the yg_state field, the bytes of one element, the elements per
// chain as a function of the parameter dimension d and the adaptive error model's data dimension dd, and the group.
// ALWAYS and DIAG buffers exist in every handle, AM buffers if cfg.adaptive, AEM buffers if cfg.aem (allocated by
// yg_set_problem, which learns dd).  yg_set_state zeroes DIAG unless YG_KEEP_DIAGNOSTICS, AM and AEM unless
// YG_KEEP_ADAPTATION.
enum Group { ALWAYS, DIAG, AM, AEM };
struct StateSpec {
    size_t field;                               // offsetof(yg_state, ..._dev)
    size_t elem;
    size_t (*per_chain)(size_t d, size_t dd);
    Group group;
};
const StateSpec kState[SB_COUNT] = {
    {offsetof(yg_state, theta_dev), sizeof(double), [](size_t d, size_t) { return d; }, ALWAYS},
    {offsetof(yg_state, logpost_dev), sizeof(double), [](size_t, size_t) { return (size_t)YG_MAX_LEVELS; }, ALWAYS},
    {offsetof(yg_state, n_accept_dev), sizeof(unsigned long long), [](size_t, size_t) { return (size_t)1; }, DIAG},
    {offsetof(yg_state, w_mean_dev), sizeof(double), [](size_t d, size_t) { return d; }, DIAG},
    // the large linear model keeps the diagonal of the Welford M2 only (big_linear.h)
    {offsetof(yg_state, w_m2_dev), sizeof(double), [](size_t d, size_t) { return d > YG_MAX_DIM ? d : d * d; }, DIAG},
    {offsetof(yg_state, prop_L_dev), sizeof(double), [](size_t d, size_t) { return d * d; }, AM},
    {offsetof(yg_state, am_mean_dev), sizeof(double), [](size_t d, size_t) { return d; }, AM},
    {offsetof(yg_state, am_m2_dev), sizeof(double), [](size_t d, size_t) { return d * d; }, AM},
    {offsetof(yg_state, aem_n_dev), sizeof(unsigned long long), [](size_t, size_t) { return (size_t)1; }, AEM},
    {offsetof(yg_state, aem_mean_dev), sizeof(double), [](size_t, size_t dd) { return dd; }, AEM},
    {offsetof(yg_state, aem_m2_dev), sizeof(double), [](size_t, size_t dd) { return dd; }, AEM},
    {offsetof(yg_state, aem_cache_dev), sizeof(double), [](size_t d, size_t) { return 3 * (d + 1) + 1; }, AEM},
};

bool has_group(const yg_ensemble *e, Group g) { return g == AM ? e->cfg.adaptive : (g == AEM ? e->cfg.aem : true); }

size_t buf_bytes(const yg_ensemble *e, int b)
{
    const StateSpec &s = kState[b];
    return s.elem * s.per_chain((size_t)e->cfg.dim, (size_t)e->aem_data_dim) * (size_t)e->cfg.n_chains;
}

// Bytes yg_get_state / yg_load_state copy: the state holds n_levels of logpost's YG_MAX_LEVELS rows.
size_t state_bytes(const yg_ensemble *e, int b)
{
    return b == SB_LOGPOST ? sizeof(double) * e->cfg.n_levels * e->cfg.n_chains : buf_bytes(e, b);
}

void *state_ptr(const yg_state *s, int b)
{
    void *p;
    memcpy(&p, reinterpret_cast<const char *>(s) + kState[b].field, sizeof(p));
    return p;
}

int check_handle(const yg_ensemble *e, bool need_problem, bool need_state)
{
    if (!e) {
        yg_set_error("null ensemble handle");
        return YG_ERR_INVALID;
    }
    if (need_problem && !e->problem_set) {
        yg_set_error("yg_set_problem has not been called");
        return YG_ERR_STATE;
    }
    if (need_state && !e->state_set) {
        yg_set_error("yg_set_state / yg_load_state has not been called");
        return YG_ERR_STATE;
    }
    return YG_OK;
}

int dev_alloc(void **p, size_t bytes)
{
    YG_CUDA_CHECK(cudaMalloc(p, bytes));
    YG_CUDA_CHECK(cudaMemset(*p, 0, bytes));
    return YG_OK;
}

// (Re)allocates the buffers of group g, zeroed.
int alloc_group(yg_ensemble *e, Group g)
{
    for (int b = 0; b < SB_COUNT; b++) {
        if (kState[b].group != g) continue;
        cudaFree(e->buf[b]);
        e->buf[b] = nullptr;
        const int rc = dev_alloc(&e->buf[b], buf_bytes(e, b));
        if (rc) return rc;
    }
    return YG_OK;
}

void copy_mat(double *dst, const double *src, int rows, int cols)
{
    if (src) memcpy(dst, src, sizeof(double) * rows * cols);
}

RunArgs make_args(yg_ensemble *e)
{
    RunArgs a;
    memset(&a, 0, sizeof(a));
    a.problem = static_cast<const DevProblemHeader *>(e->d_problem);    // the tensor path passes its header itself
    a.problem_bytes = (uint32_t)e->h_problem.size();
    a.thin = 1;
    a.n_chains = e->cfg.n_chains;
    a.chain_offset = e->cfg.chain_offset;
    a.seed = e->cfg.seed;
    a.step0 = e->step_index;
    a.welford_n0 = e->welford_n;
    a.am_t0 = e->am_steps;
    a.theta = static_cast<double *>(e->buf[SB_THETA]);
    a.logpost = static_cast<double *>(e->buf[SB_LOGPOST]);
    a.n_accept = static_cast<unsigned long long *>(e->buf[SB_N_ACCEPT]);
    a.w_mean = static_cast<double *>(e->buf[SB_W_MEAN]);
    a.w_m2 = static_cast<double *>(e->buf[SB_W_M2]);
    a.am_mean = static_cast<double *>(e->buf[SB_AM_MEAN]);
    a.am_m2 = static_cast<double *>(e->buf[SB_AM_M2]);
    a.prop_L = static_cast<double *>(e->buf[SB_PROP_L]);
    a.adaptive = e->cfg.adaptive;
    a.am_refresh = std::max(1, e->cfg.am_refresh);
    a.am_idle = e->cfg.am_idle_steps;
    a.am_collect = e->cfg.am_collection_steps;
    a.am_eps = e->cfg.am_eps;
    a.am_scale = e->cfg.am_scale > 0.0 ? e->cfg.am_scale : 2.4 * 2.4 / (double)e->cfg.dim;
    a.aem = e->cfg.aem;
    a.aem_min_data = e->cfg.aem_min_data;
    a.aem_heuristic = e->cfg.aem_heuristic;
    a.welford = e->cfg.acceptance_only ? 0 : 1;
    a.aem_n = static_cast<unsigned long long *>(e->buf[SB_AEM_N]);
    a.aem_mean = static_cast<double *>(e->buf[SB_AEM_MEAN]);
    a.aem_m2 = static_cast<double *>(e->buf[SB_AEM_M2]);
    a.aem_cache = static_cast<double *>(e->buf[SB_AEM_CACHE]);
    a.counters = e->counters;
    return a;
}

__global__ void broadcast_L_kernel(const DevProblemHeader *pb, double *prop_L, int64_t n)
{
    const int d = pb->dim;
    for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n; g += (int64_t)gridDim.x * blockDim.x)
        for (int k = 0; k < d * d; k++) prop_L[(int64_t)k * n + g] = pb->prop_L[k];
}

// Every chain of an adaptive ensemble restarts from the problem's proposal factor.
int broadcast_prop_L(yg_ensemble *e, cudaStream_t st)
{
    const size_t n = (size_t)e->cfg.n_chains;
    broadcast_L_kernel<<<(int)std::min<size_t>((n + 127) / 128, 2048), 128, 0, st>>>(
        static_cast<const DevProblemHeader *>(e->d_problem), static_cast<double *>(e->buf[SB_PROP_L]), (int64_t)n);
    YG_CUDA_CHECK(cudaGetLastError());
    return YG_OK;
}

bool is_diagonal(const double *M, int n)
{
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++)
            if (i != j && M[i * n + j] != 0.0) return false;
    return true;
}

// The blob builders read the configuration and the problem only.  yg_set_problem has checked the proposal kind, the
// pCN rules and that prop_L is lower triangular.

// Large linear model: the DevBigHeader blob (big_linear.h) of linear_dmma_kernel.cu.
int build_big_blob(const yg_config &c, const yg_problem *pb, std::vector<char> &blob)
{
    const int d = c.dim, nl = c.n_levels;
    if (c.adaptive || c.eq_mode != YG_EQ_EXACT || c.aem || nl > 3) {
        yg_set_error("large linear model (dim > %d or data_dim > %d): MRW / pCN / MLDA with up to two surrogates with "
                     "exact equality only (no adaptive proposal or adaptive error model)", YG_MAX_DIM, YG_MAX_DATA_DIM);
        return YG_ERR_UNSUPPORTED;
    }
    const bool dense_L = !is_diagonal(pb->prop_L, d);
    const int kp = d <= 16 ? 16 : (d <= 32 ? 32 : 64), ks = kp + 4;
    int np_l[3] = {0, 0, 0};              // operand rows per level, rounded up to 16
    bool dense_prior[3] = {false, false, false};
    double temper[3] = {1.0, 1.0, 1.0};   // tempering of each level (target.py:40-43)
    std::vector<double> Rp[3];            // chol(prior precision)' of the levels with a dense prior
    for (int l = 0; l < nl; l++) {
        const yg_level &L = pb->level[l];
        if (!L.data || !L.noise_prec || !L.prior_mean || !L.prior_prec || !L.G || !L.b || L.n_data < 1 ||
            L.data_dim < 1) {
            yg_set_error("level %d: linear level needs data, noise_prec, prior, G and b", l);
            return YG_ERR_INVALID;
        }
        if (L.tempered) {
            if (!(L.tempering >= 0.0 && L.tempering <= 1.0)) {       // tmlda.py:24-29
                yg_set_error("Invalid tempering parameter at index %d: %g (must be in [0, 1]).", l, L.tempering);
                return YG_ERR_INVALID;
            }
            temper[l] = L.tempering;
        }
        if (L.data_dim > YG_BIG_MAX_DATA_DIM) {
            yg_set_error("level %d: large linear model is limited to data_dim <= %d", l, YG_BIG_MAX_DATA_DIM);
            return YG_ERR_UNSUPPORTED;
        }
        if (!is_diagonal(L.noise_prec, L.data_dim)) {
            yg_set_error("level %d: large linear model needs diagonal measurement noise", l);
            return YG_ERR_UNSUPPORTED;
        }
        for (int r = 0; r < L.data_dim; r++)
            if (!(L.noise_prec[(size_t)r * L.data_dim + r] >= 0.0)) {
                yg_set_error("level %d: negative noise precision", l);
                return YG_ERR_INVALID;
            }
        dense_prior[l] = !is_diagonal(L.prior_prec, d);
        if (dense_prior[l]) {
            // P = Lp Lp' (lower Cholesky); R = Lp' so that ||R x||^2 = x' P x.  DenseCovarianceMatrix priors
            // (statistics/covariance.py:69-94) arrive here as their dense precision.
            Rp[l].assign((size_t)d * d, 0.0);
            std::vector<double> Lp((size_t)d * d, 0.0);
            for (int j = 0; j < d; j++) {
                double sdiag = L.prior_prec[(size_t)j * d + j];
                for (int k = 0; k < j; k++) sdiag -= Lp[(size_t)j * d + k] * Lp[(size_t)j * d + k];
                if (!(sdiag > 0.0)) {
                    yg_set_error("level %d: the dense prior precision is not positive definite", l);
                    return YG_ERR_INVALID;
                }
                Lp[(size_t)j * d + j] = sqrt(sdiag);
                for (int i = j + 1; i < d; i++) {
                    double v = 0.5 * (L.prior_prec[(size_t)i * d + j] + L.prior_prec[(size_t)j * d + i]);
                    for (int k = 0; k < j; k++) v -= Lp[(size_t)i * d + k] * Lp[(size_t)j * d + k];
                    Lp[(size_t)i * d + j] = v / Lp[(size_t)j * d + j];
                }
            }
            for (int i = 0; i < d; i++)
                for (int j = 0; j < d; j++) Rp[l][(size_t)i * d + j] = Lp[(size_t)j * d + i];
        }
        np_l[l] = (L.data_dim + (dense_prior[l] ? d : 0) + 15) & ~15;
    }
    // operands that leave too little shared memory for BIG_MIN_WARPS warps are read from this blob's global copy
    // (smem_plan.h: big_tensor_plan); inside the envelope that always suffices, so the refusal is a safety check only
    const BigTensorPlan plan = big_tensor_plan(np_l[0], np_l[1], kp / 4, dense_L, false, np_l[2]);
    if (plan.smem.warps < BIG_MIN_WARPS) {
        yg_set_error("large linear model: %zu bytes of G / data do not fit the shared memory of one SM",
                     sizeof(double) * (size_t)plan.resident);
        return YG_ERR_UNSUPPORTED;
    }
    const size_t tail_len = (size_t)plan.tail;
    blob.assign(sizeof(DevBigHeader) + sizeof(double) * tail_len, 0);
    DevBigHeader *h = reinterpret_cast<DevBigHeader *>(blob.data());
    double *tail = reinterpret_cast<double *>(blob.data() + sizeof(DevBigHeader));
    h->dim = d; h->kp = kp; h->ks = ks; h->n_levels = nl;
    h->J = nl >= 2 ? c.sub_chain_length : 1;
    h->tail_len = (int32_t)tail_len;
    h->proposal = pb->proposal;
    h->dense_L = dense_L ? 1 : 0;
    h->stream = plan.stream;
    // every item in the staged prefix in the order below, except the streamed operands: those follow the prefix
    size_t off = 0, soff = (size_t)plan.resident;
    auto place = [&](const size_t n, const int bit) {
        size_t &cur = (plan.stream & bit) ? soff : off;
        const size_t at = cur;
        cur += n;
        return (int32_t)at;
    };
    if (pb->proposal == YG_PROPOSAL_PCN) {
        const double t = 2.0 * pb->pcn_step;                      // pcn.py:30
        h->pcn_a = sqrt(1.0 - t);
        h->pcn_b = sqrt(t);
    }
    for (int l = 0; l < nl; l++) {
        const yg_level &L = pb->level[l];
        BigLevel &B = h->lvl[l];
        const int rows = L.data_dim + (dense_prior[l] ? d : 0);
        const int np = np_l[l];
        B.n_data = L.n_data; B.data_dim = L.data_dim; B.np = np; B.n_rows = rows;
        B.G_off = place((size_t)np * ks, l == 1 ? BIG_STREAM_G1 : (l == 2 ? BIG_STREAM_G2 : 0));
        B.bd_off = place((size_t)np, 0);
        const size_t goff = (size_t)B.G_off;
        // sum_rows ||F - d_row||^2_P = sum_col n P_col (F_col - mean_col)^2 + sum_col P_col sum_rows (d - mean)^2;
        // sqrt(n P_col) is folded into row `col` of G and into b - mean.  A tempered level scales the data rows by
        // fl(sqrt(t)) and q_const by t (t = 1: both factors are exactly 1, the operands those of an untempered level).
        const double st = sqrt(temper[l]);
        double q_const = 0.0;
        for (int r = 0; r < L.data_dim; r++) {
            double mean = 0.0;
            for (int i = 0; i < L.n_data; i++) mean += L.data[(size_t)i * L.data_dim + r];
            mean /= (double)L.n_data;
            double scatter = 0.0;
            for (int i = 0; i < L.n_data; i++) {
                const double dd = L.data[(size_t)i * L.data_dim + r] - mean;
                scatter += dd * dd;
            }
            const double prec = L.noise_prec[(size_t)r * L.data_dim + r];
            const double sw = st * sqrt((double)L.n_data * prec);
            for (int k = 0; k < d; k++) tail[goff + (size_t)r * ks + k] = sw * L.G[(size_t)r * d + k];
            tail[B.bd_off + r] = sw * (L.b[r] - mean);
            q_const += prec * scatter;
        }
        if (dense_prior[l]) {                    // d more rows: R and -R m
            for (int r = 0; r < d; r++) {
                double rm = 0.0;
                for (int k = 0; k < d; k++) {
                    tail[goff + (size_t)(L.data_dim + r) * ks + k] = Rp[l][(size_t)r * d + k];
                    rm += Rp[l][(size_t)r * d + k] * L.prior_mean[k];
                }
                tail[B.bd_off + L.data_dim + r] = -rm;
            }
        }
        B.q_const = temper[l] * q_const;
        B.pmean_off = place(kp, 0);
        for (int k = 0; k < d; k++) tail[B.pmean_off + k] = L.prior_mean[k];
        B.pprec_off = place(kp, 0);
        if (!dense_prior[l])
            for (int k = 0; k < d; k++) tail[B.pprec_off + k] = L.prior_prec[(size_t)k * d + k];
    }
    if (nl == 1) h->lvl[1] = h->lvl[0];
    h->propL_off = place(kp, 0);
    for (int k = 0; k < d; k++) tail[h->propL_off + k] = pb->prop_L[(size_t)k * d + k];
    h->pcn_mean_off = place(kp, 0);
    if (pb->proposal == YG_PROPOSAL_PCN && pb->pcn_mean)
        for (int k = 0; k < d; k++) tail[h->pcn_mean_off + k] = pb->pcn_mean[k];
    h->Ld_off = place(dense_L ? (size_t)kp * ks : 0, BIG_STREAM_LD);
    if (dense_L)
        for (int r = 0; r < d; r++)
            for (int k = 0; k <= r; k++) tail[h->Ld_off + (size_t)r * ks + k] = pb->prop_L[(size_t)r * d + k];
    return YG_OK;
}

}  // namespace

extern "C" const char *yg_last_error(void) { return g_err; }
extern "C" uint32_t yg_abi_version(void) { return YG_ABI_VERSION; }

extern "C" int yg_create(const yg_config *cfg, yg_ensemble **out)
{
    if (!cfg || !out) {
        yg_set_error("yg_create: null argument");
        return YG_ERR_INVALID;
    }
    *out = nullptr;
    if (cfg->abi_version != YG_ABI_VERSION) {
        yg_set_error("abi_version %u != library %u", cfg->abi_version, YG_ABI_VERSION);
        return YG_ERR_ABI;
    }
    const int max_dim = cfg->model == YG_MODEL_LINEAR ? YG_BIG_MAX_DIM : YG_MAX_DIM;
    if (cfg->n_chains < 1 || cfg->dim < 1 || cfg->dim > max_dim) {
        yg_set_error("n_chains=%lld dim=%d out of range (dim 1..%d)", (long long)cfg->n_chains, cfg->dim, max_dim);
        return cfg->dim > max_dim ? YG_ERR_UNSUPPORTED : YG_ERR_INVALID;
    }
    if (cfg->dim > YG_MAX_DIM && cfg->adaptive) {
        yg_set_error("adaptive Metropolis is limited to dim <= %d", YG_MAX_DIM);
        return YG_ERR_UNSUPPORTED;
    }
    if (cfg->n_levels < 1 || cfg->n_levels > YG_MAX_LEVELS) {
        yg_set_error("n_levels=%d: MRW (1), two-level delayed acceptance (2) and MLDA with two surrogates (3) "
                     "exist on the device", cfg->n_levels);
        return YG_ERR_UNSUPPORTED;
    }
    if (cfg->n_levels == 3 && (cfg->model == YG_MODEL_LV_RK4 || cfg->aem)) {
        yg_set_error("three levels: Gaussian targets and the linear model only, no adaptive error model");
        return YG_ERR_UNSUPPORTED;
    }
    if (cfg->n_levels >= 2 && cfg->sub_chain_length < 1) {
        yg_set_error("sub_chain_length must be >= 1");
        return YG_ERR_INVALID;
    }
    if (cfg->model != YG_MODEL_GAUSS && cfg->model != YG_MODEL_LINEAR && cfg->model != YG_MODEL_LV_RK4) {
        yg_set_error("unknown model %d", cfg->model);
        return YG_ERR_UNSUPPORTED;
    }
    if (cfg->model == YG_MODEL_LV_RK4 && cfg->dim != 2) {
        yg_set_error("the Lotka-Volterra model has two parameters (dim=%d)", cfg->dim);
        return YG_ERR_INVALID;
    }
    if (cfg->adaptive && cfg->dim < 2) {
        yg_set_error("Adaptivity not implemented for scalar chains.");      // chain/adaptive.py:41-43
        return YG_ERR_UNSUPPORTED;
    }
    if (cfg->adaptive && (cfg->am_idle_steps < 0 || cfg->am_collection_steps < 0 || cfg->am_refresh < 0)) {
        yg_set_error("adaptive Metropolis: idle / collection steps and the refresh interval must be >= 0");
        return YG_ERR_INVALID;
    }
    // the builder's rule (AMBuilder.regularisationParameter: eps >= 0); a NaN eps or scale would make every refresh
    // fail, and the chain would silently never adapt.  A scale <= 0 selects the default 2.4^2 / d (make_args).
    if (cfg->adaptive && (!std::isfinite(cfg->am_eps) || cfg->am_eps < 0.0 || !std::isfinite(cfg->am_scale))) {
        yg_set_error("adaptive Metropolis: the regularisation eps must be finite and >= 0, and the scale finite "
                     "(eps=%g, scale=%g)", cfg->am_eps, cfg->am_scale);
        return YG_ERR_INVALID;
    }
    if (cfg->aem) {
        if (cfg->n_levels != 2 || cfg->model != YG_MODEL_LINEAR || cfg->adaptive || cfg->dim > YG_MAX_DIM) {
            yg_set_error("adaptive error model: two levels, linear model (dim <= %d), no adaptive proposal", YG_MAX_DIM);
            return YG_ERR_UNSUPPORTED;   // aem.py:72-75: only defined for a hierarchy of Bayesian models
        }
        if (cfg->aem_min_data < 2) {
            yg_set_error("Smallest senisible data size for AEM is 2.");      // likelihood.py:99-100
            return YG_ERR_INVALID;
        }
    }
    if (cfg->eq_mode == YG_EQ_ISCLOSE && cfg->dim != 1) {
        yg_set_error("isclose equality is the ScalarParameter rule (dim must be 1)");
        return YG_ERR_INVALID;
    }
    int ndev = 0;
    YG_CUDA_CHECK(cudaGetDeviceCount(&ndev));
    if (cfg->device < 0 || cfg->device >= ndev) {
        yg_set_error("device %d not present (%d visible)", cfg->device, ndev);
        return YG_ERR_INVALID;
    }
    YG_CUDA_CHECK(cudaSetDevice(cfg->device));
    yg_ensemble *e = new (std::nothrow) yg_ensemble();
    if (!e) {
        yg_set_error("out of host memory");
        return YG_ERR_INVALID;
    }
    e->cfg = *cfg;
    if (cudaDeviceGetAttribute(&e->sm_count, cudaDevAttrMultiProcessorCount, cfg->device) != cudaSuccess) {
        yg_set_error("cudaDeviceGetAttribute(multiProcessorCount) failed: %s", cudaGetErrorString(cudaGetLastError()));
        delete e;
        return YG_ERR_CUDA;
    }
    int rc = YG_OK;
    if ((rc = alloc_group(e, ALWAYS)) || (rc = alloc_group(e, DIAG)) || (cfg->adaptive && (rc = alloc_group(e, AM))) ||
        (rc = dev_alloc((void **)&e->counters, sizeof(unsigned long long) * 8)) ||
        (rc = dev_alloc((void **)&e->pool_partials,
                        sizeof(double) * POOL_PARTS * (size_t)yg_pooled_len(std::min(cfg->dim, YG_MAX_DIM))))) {
        yg_destroy(e);
        return rc;
    }
    *out = e;
    return YG_OK;
}

extern "C" int yg_destroy(yg_ensemble *e)
{
    if (!e) return YG_OK;
    cudaSetDevice(e->cfg.device);
    for (void *p : e->buf) cudaFree(p);
    cudaFree(e->d_problem);
    cudaFree(e->counters);
    cudaFree(e->pool_partials);
    cudaFree(e->big_done);
    delete e;
    return YG_OK;
}

namespace {

// One-chain-per-thread and LV kernels: the DevProblemHeader blob (common.cuh).
int build_blob(const yg_config &c, const yg_problem *pb, std::vector<char> &blob)
{
    const int d = c.dim, nl = c.n_levels, model = c.model;
    // tail: per level data + design
    size_t tail_len = 0;
    for (int l = 0; l < nl; l++) {
        const yg_level &L = pb->level[l];
        if (model == YG_MODEL_GAUSS) {
            if (!L.g_mean || !L.g_prec) {
                yg_set_error("level %d: Gaussian target needs g_mean and g_prec", l);
                return YG_ERR_INVALID;
            }
            continue;
        }
        if (!L.data || !L.noise_prec || !L.prior_mean || !L.prior_prec || L.n_data < 1 || L.data_dim < 1 ||
            L.data_dim > YG_MAX_DATA_DIM) {
            yg_set_error("level %d: regression level needs data[n_data>=1, data_dim<=%d], noise_prec, prior", l,
                         YG_MAX_DATA_DIM);
            return YG_ERR_INVALID;
        }
        if (model == YG_MODEL_LINEAR && (!L.G || !L.b)) {
            yg_set_error("level %d: linear model needs G and b", l);
            return YG_ERR_INVALID;
        }
        if (model == YG_MODEL_LV_RK4) {
            if (!L.design || L.data_dim != 2 || L.rk4_steps < 1 || !(L.T > 0.0)) {
                yg_set_error("level %d: LV model needs design[n_data,2], data_dim=2, rk4_steps>=1, T>0", l);
                return YG_ERR_INVALID;
            }
        }
        tail_len += (size_t)L.n_data * L.data_dim;
        if (model == YG_MODEL_LV_RK4) tail_len += (size_t)L.n_data * 2;
    }
    tail_len = (tail_len + 1) & ~size_t(1);        // keep the blob a multiple of 16 bytes
    blob.assign(sizeof(DevProblemHeader) + sizeof(double) * tail_len, 0);
    DevProblemHeader *h = reinterpret_cast<DevProblemHeader *>(blob.data());
    double *tail = reinterpret_cast<double *>(blob.data() + sizeof(DevProblemHeader));
    h->model = model;
    h->dim = d;
    h->n_levels = nl;
    h->J = nl >= 2 ? c.sub_chain_length : 1;
    h->eq_mode = c.eq_mode;
    h->tail_len = (int32_t)tail_len;
    h->proposal = pb->proposal;
    if (pb->proposal == YG_PROPOSAL_PCN) {
        const double t = 2.0 * pb->pcn_step;                      // pcn.py:30
        h->pcn_a = sqrt(1.0 - t);
        h->pcn_b = sqrt(t);
        if (pb->pcn_mean) copy_mat(h->pcn_mean, pb->pcn_mean, 1, d);
    }
    copy_mat(h->prop_L, pb->prop_L, d, d);
    size_t off = 0;
    for (int l = 0; l < nl; l++) {
        const yg_level &L = pb->level[l];
        DevLevel &D = h->lvl[l];
        if (model == YG_MODEL_GAUSS) {
            copy_mat(D.g_mean, L.g_mean, 1, d);
            copy_mat(D.g_prec, L.g_prec, d, d);
            D.g_logconst = L.g_logconst;
            continue;
        }
        D.n_data = L.n_data;
        D.data_dim = L.data_dim;
        D.tempering = 1.0;
        if (L.tempered) {
            if (!(L.tempering >= 0.0 && L.tempering <= 1.0)) {       // tmlda.py:24-29
                yg_set_error("Invalid tempering parameter at index %d: %g (must be in [0, 1]).", l, L.tempering);
                return YG_ERR_INVALID;
            }
            D.tempering = L.tempering;
        }
        copy_mat(D.noise_prec, L.noise_prec, L.data_dim, L.data_dim);
        copy_mat(D.prior_mean, L.prior_mean, 1, d);
        copy_mat(D.prior_prec, L.prior_prec, d, d);
        D.data_off = (int32_t)off;
        memcpy(tail + off, L.data, sizeof(double) * L.n_data * L.data_dim);
        off += (size_t)L.n_data * L.data_dim;
        if (model == YG_MODEL_LINEAR) {
            copy_mat(D.G, L.G, L.data_dim, d);
            copy_mat(D.b, L.b, 1, L.data_dim);
        } else {
            D.alpha = L.alpha;
            D.gamma = L.gamma;
            D.T = L.T;
            D.rk4_steps = L.rk4_steps;
            D.design_off = (int32_t)off;
            memcpy(tail + off, L.design, sizeof(double) * L.n_data * 2);
            off += (size_t)L.n_data * 2;
        }
    }
    if (c.aem) {
        const yg_level &Lc = pb->level[0], &Lf = pb->level[1];
        if (Lc.data_dim != Lf.data_dim || pb->proposal != YG_PROPOSAL_MRW) {
            yg_set_error("adaptive error model: both levels must share the data dimension (MRW proposal)");
            return YG_ERR_INVALID;
        }
        if (Lc.tempered && Lc.tempering != 1.0) {
            // the error model's coarse log-posterior has no tempering factor (likelihood.py:74-84,140-145)
            yg_set_error("adaptive error model: a tempered level 0 (tempering %g) is not supported", Lc.tempering);
            return YG_ERR_UNSUPPORTED;
        }
        for (int i = 0; i < Lc.data_dim; i++)
            for (int j = 0; j < Lc.data_dim; j++)
                if (i != j && Lc.noise_prec[i * Lc.data_dim + j] != 0.0) {
                    // noise.py:29-33
                    yg_set_error("Currently, AEM is only implemented for independent measurement noise.");
                    return YG_ERR_UNSUPPORTED;
                }
    }
    return YG_OK;
}

}  // namespace

extern "C" int yg_set_problem(yg_ensemble *e, const yg_problem *pb)
{
    int rc = check_handle(e, false, false);
    if (rc) return rc;
    if (!pb || !pb->prop_L) {
        yg_set_error("yg_set_problem: problem / prop_L is null");
        return YG_ERR_INVALID;
    }
    const yg_config &c = e->cfg;
    const int d = c.dim, nl = c.n_levels;
    if (pb->proposal != YG_PROPOSAL_MRW && pb->proposal != YG_PROPOSAL_PCN) {
        yg_set_error("unknown proposal kind %d", pb->proposal);
        return YG_ERR_INVALID;
    }
    if (pb->proposal == YG_PROPOSAL_PCN) {
        if (!(pb->pcn_step > 0.0 && pb->pcn_step <= 0.5)) {       // pcn.py:42
            yg_set_error("pCN step size must lie in (0, 0.5], got %g", pb->pcn_step);
            return YG_ERR_INVALID;
        }
        if (nl != 1 || c.adaptive) {
            yg_set_error("pCN is a single-level, non-adaptive method (chain/method/pcn.py)");
            return YG_ERR_UNSUPPORTED;
        }
    }
    for (int i = 0; i < d; i++)
        for (int j = i + 1; j < d; j++)
            if (pb->prop_L[(size_t)i * d + j] != 0.0) {
                yg_set_error("prop_L must be lower triangular");
                return YG_ERR_INVALID;
            }
    bool big = false;
    if (c.model == YG_MODEL_LINEAR) {
        big = d > YG_MAX_DIM;
        for (int l = 0; l < nl; l++) big = big || pb->level[l].data_dim > YG_MAX_DATA_DIM;
    }
    std::vector<char> blob;
    if ((rc = big ? build_big_blob(c, pb, blob) : build_blob(c, pb, blob))) return rc;
    // Commit.  The handle changes from here on only, and holds no problem unless every step below succeeds.
    YG_CUDA_CHECK(cudaSetDevice(c.device));
    e->problem_set = false;
    cudaFree(e->d_problem);
    e->d_problem = nullptr;
    YG_CUDA_CHECK(cudaMalloc(&e->d_problem, blob.size()));
    YG_CUDA_CHECK(cudaMemcpy(e->d_problem, blob.data(), blob.size(), cudaMemcpyHostToDevice));
    e->h_problem.swap(blob);
    e->big = big;
    if (big && !e->big_done) {      // per-tile progress counters of the balanced (tile, step-range) schedule
        if ((rc = dev_alloc((void **)&e->big_done, sizeof(long long) * (((size_t)c.n_chains + 7) / 8)))) return rc;
    }
    if (c.aem) {
        e->aem_data_dim = pb->level[0].data_dim;
        if ((rc = alloc_group(e, AEM))) return rc;
    }
    e->problem_set = true;
    return YG_OK;
}

extern "C" int yg_set_state(yg_ensemble *e, const double *theta0_dev, int32_t flags, void *stream)
{
    int rc = check_handle(e, true, false);
    if (rc) return rc;
    if (!theta0_dev) {
        yg_set_error("theta0_dev is null");
        return YG_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t n = (size_t)e->cfg.n_chains;
    // a handle that never held a state has nothing to keep
    const bool keep_diag = (flags & YG_KEEP_DIAGNOSTICS) && e->state_set;
    const bool keep_adapt = (flags & YG_KEEP_ADAPTATION) && e->state_set;
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    YG_CUDA_CHECK(cudaMemcpyAsync(e->buf[SB_THETA], theta0_dev, buf_bytes(e, SB_THETA), cudaMemcpyDeviceToDevice, st));
    for (int b = 0; b < SB_COUNT; b++) {      // prop_L restarts from the problem's factor below, not from zeros
        const Group g = kState[b].group;
        const bool reset = g == DIAG ? !keep_diag : (g != ALWAYS && has_group(e, g) && !keep_adapt);
        if (reset && b != SB_PROP_L) YG_CUDA_CHECK(cudaMemsetAsync(e->buf[b], 0, buf_bytes(e, b), st));
    }
    if (!keep_diag) {
        YG_CUDA_CHECK(cudaMemsetAsync(e->counters, 0, sizeof(unsigned long long) * 8, st));
        e->welford_n = 0;
    }
    if (e->cfg.adaptive && !keep_adapt) {
        if ((rc = broadcast_prop_L(e, st))) return rc;
        e->am_steps = 0;
    }
    double *theta = static_cast<double *>(e->buf[SB_THETA]), *logpost = static_cast<double *>(e->buf[SB_LOGPOST]);
    for (int l = 0; l < e->cfg.n_levels; l++) {
        rc = e->big ? yg_launch_logpost_big(e, l, theta, (int64_t)n, logpost + (size_t)l * n, st)
                    : yg_launch_logpost(e, l, theta, (int64_t)n, logpost + (size_t)l * n, st);
        if (rc) return rc;
    }
    // e->step_index (the Philox stream position) is deliberately left alone: the reference's numpy
    // generator keeps advancing across run() calls, and so does this stream (yg_seek repositions it)
    e->state_set = true;
    return YG_OK;
}

extern "C" int yg_seek(yg_ensemble *e, int64_t step_index)
{
    int rc = check_handle(e, false, false);
    if (rc) return rc;
    if (step_index < 0) {
        yg_set_error("yg_seek: step_index must be >= 0");
        return YG_ERR_INVALID;
    }
    e->step_index = step_index;
    return YG_OK;
}

// Replaces the proposal factor between launches (pooled proposal covariance across GPUs, north_star;
// the reference's only hook for this is AdaptiveMRWProposal swapping its covariance, chain/adaptive.py:55-60).
extern "C" int yg_set_proposal_factor(yg_ensemble *e, const double *L_host, void *stream)
{
    int rc = check_handle(e, true, false);
    if (rc) return rc;
    const int d = e->cfg.dim;
    if (!L_host) {
        yg_set_error("yg_set_proposal_factor: L is null");
        return YG_ERR_INVALID;
    }
    for (int i = 0; i < d; i++)
        for (int j = 0; j < d; j++) {
            const double v = L_host[(size_t)i * d + j];
            if (!std::isfinite(v) || (j > i && v != 0.0) || (i == j && !(v > 0.0))) {
                yg_set_error("proposal factor must be finite, lower triangular with a positive diagonal");
                return YG_ERR_INVALID;
            }
        }
    cudaStream_t st = (cudaStream_t)stream;
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    if (e->big) {
        DevBigHeader *h = reinterpret_cast<DevBigHeader *>(e->h_problem.data());
        if (!h->dense_L && !is_diagonal(L_host, d)) {
            yg_set_error("large linear model: this handle was built for a diagonal proposal factor (its kernels and shared-"
                         "memory plan differ for a dense one): pass a dense factor to yg_set_problem to switch");
            return YG_ERR_UNSUPPORTED;
        }
        if (h->proposal != YG_PROPOSAL_MRW) {
            yg_set_error("the proposal factor of a pCN chain is the prior's (pcn.py:23-35) and cannot be replaced");
            return YG_ERR_UNSUPPORTED;
        }
        double *tail = reinterpret_cast<double *>(e->h_problem.data() + sizeof(DevBigHeader));
        for (int k = 0; k < d; k++) tail[h->propL_off + k] = L_host[(size_t)k * d + k];
        char *base = static_cast<char *>(e->d_problem) + sizeof(DevBigHeader);
        YG_CUDA_CHECK(cudaMemcpyAsync(base + sizeof(double) * h->propL_off, tail + h->propL_off, sizeof(double) * d,
                                      cudaMemcpyHostToDevice, st));
        if (h->dense_L) {
            for (int r = 0; r < d; r++)
                for (int k = 0; k < d; k++) tail[h->Ld_off + (size_t)r * h->ks + k] = (k <= r) ? L_host[(size_t)r * d + k] : 0.0;
            YG_CUDA_CHECK(cudaMemcpyAsync(base + sizeof(double) * h->Ld_off, tail + h->Ld_off,
                                          sizeof(double) * (size_t)h->kp * h->ks, cudaMemcpyHostToDevice, st));
        }
        return YG_OK;
    }
    DevProblemHeader *h = reinterpret_cast<DevProblemHeader *>(e->h_problem.data());
    if (h->proposal != YG_PROPOSAL_MRW) {
        yg_set_error("the proposal factor of a pCN chain is the prior's (pcn.py:23-35) and cannot be replaced");
        return YG_ERR_UNSUPPORTED;
    }
    copy_mat(h->prop_L, L_host, d, d);
    YG_CUDA_CHECK(cudaMemcpyAsync(static_cast<char *>(e->d_problem) + offsetof(DevProblemHeader, prop_L), h->prop_L,
                                  sizeof(h->prop_L), cudaMemcpyHostToDevice, st));
    return e->cfg.adaptive ? broadcast_prop_L(e, st) : YG_OK;
}

extern "C" int yg_run(yg_ensemble *e, int64_t n_steps, int32_t thin, const yg_outputs *out, const yg_noise *noise,
                      void *stream)
{
    int rc = check_handle(e, true, true);
    if (rc) return rc;
    if (n_steps < 0 || thin < 1) {
        yg_set_error("n_steps=%lld thin=%d invalid", (long long)n_steps, thin);
        return YG_ERR_INVALID;
    }
    if (n_steps == 0) return YG_OK;
    RunArgs a = make_args(e);
    a.n_steps = n_steps;
    a.thin = thin;
    if (out) {
        a.samples = out->samples_dev;
        a.accepted = out->accepted_dev;
        a.lp_out = out->logpost_dev;
        if ((a.samples || a.lp_out) && n_steps % thin) {
            yg_set_error("n_steps (%lld) must be a multiple of thin (%d) when samples are stored",
                         (long long)n_steps, thin);
            return YG_ERR_INVALID;
        }
    }
    if (noise && noise->mode != YG_NOISE_PHILOX) {
        if (noise->mode != YG_NOISE_INJECT && noise->mode != YG_NOISE_RECORD) {
            yg_set_error("unknown noise mode %d", noise->mode);
            return YG_ERR_INVALID;
        }
        if (!noise->z_dev || !noise->u_f_dev || (e->cfg.n_levels >= 2 && !noise->u_c_dev)) {
            yg_set_error("noise mode %d needs z_dev, u_f_dev%s", noise->mode,
                         e->cfg.n_levels >= 2 ? " and u_c_dev" : "");
            return YG_ERR_INVALID;
        }
        a.noise_mode = noise->mode;
        a.z = noise->z_dev;
        a.u_c = noise->u_c_dev;
        a.u_f = noise->u_f_dev;
    }
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    rc = e->big ? yg_launch_linear_big(e, a, (cudaStream_t)stream)
         : (e->cfg.model == YG_MODEL_LV_RK4) ? yg_launch_lv(e, a, (cudaStream_t)stream)
                                             : yg_launch_generic(e, a, (cudaStream_t)stream);
    if (rc) return rc;
    e->step_index += n_steps;
    e->welford_n += n_steps;
    if (e->cfg.adaptive) e->am_steps += n_steps;
    return YG_OK;
}

extern "C" int yg_get_state(yg_ensemble *e, const yg_state *dst, void *stream)
{
    int rc = check_handle(e, true, true);
    if (rc) return rc;
    if (!dst) return YG_ERR_INVALID;
    for (int b = 0; b < SB_COUNT; b++) {
        const Group g = kState[b].group;
        if (state_ptr(dst, b) && !has_group(e, g)) {
            yg_set_error("%s per-chain state of %s ensembles only",
                         b == SB_PROP_L ? "prop_L_dev is" : (g == AM ? "am_mean_dev / am_m2_dev are" : "aem_*_dev are"),
                         g == AM ? "adaptive" : "adaptive-error-model");
            return YG_ERR_INVALID;
        }
    }
    cudaStream_t st = (cudaStream_t)stream;
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    for (int b = 0; b < SB_COUNT; b++)
        if (void *p = state_ptr(dst, b))
            YG_CUDA_CHECK(cudaMemcpyAsync(p, e->buf[b], state_bytes(e, b), cudaMemcpyDeviceToDevice, st));
    return YG_OK;
}

extern "C" int yg_load_state(yg_ensemble *e, const yg_state *src, int64_t step_index, int64_t welford_n,
                             int64_t am_steps, void *stream)
{
    int rc = check_handle(e, true, false);
    if (rc) return rc;
    if (!src || !src->theta_dev || !src->logpost_dev) {
        yg_set_error("yg_load_state needs at least theta_dev and logpost_dev");
        return YG_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    for (int b = 0; b < SB_COUNT; b++) {
        const void *p = state_ptr(src, b);
        if (p && has_group(e, kState[b].group))       // pointers for groups the handle lacks are ignored
            YG_CUDA_CHECK(cudaMemcpyAsync(e->buf[b], p, state_bytes(e, b), cudaMemcpyDeviceToDevice, st));
    }
    e->step_index = step_index;
    e->welford_n = welford_n;
    e->am_steps = am_steps;
    e->state_set = true;
    return YG_OK;
}

extern "C" int yg_get_counters(yg_ensemble *e, int64_t *out_host, void *stream)
{
    int rc = check_handle(e, false, false);
    if (rc) return rc;
    if (!out_host) return YG_ERR_INVALID;
    unsigned long long c[8];
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    YG_CUDA_CHECK(cudaMemcpyAsync(c, e->counters, sizeof(c), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    YG_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    out_host[0] = e->step_index;
    out_host[1] = (int64_t)c[0];
    out_host[2] = (int64_t)c[1];
    out_host[3] = (int64_t)c[2];
    out_host[4] = (int64_t)c[3];
    out_host[5] = e->welford_n;
    out_host[6] = e->am_steps;
    out_host[7] = (int64_t)c[4];
    out_host[8] = (int64_t)c[5];
    out_host[9] = (int64_t)c[6];
    return YG_OK;
}

extern "C" int yg_logpost(yg_ensemble *e, int32_t level, const double *theta_dev, int64_t n, double *out_dev,
                          void *stream)
{
    int rc = check_handle(e, true, false);
    if (rc) return rc;
    if (level < 0 || level >= e->cfg.n_levels || !theta_dev || !out_dev || n < 1) {
        yg_set_error("yg_logpost: invalid arguments");
        return YG_ERR_INVALID;
    }
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    return e->big ? yg_launch_logpost_big(e, level, theta_dev, n, out_dev, (cudaStream_t)stream)
                  : yg_launch_logpost(e, level, theta_dev, n, out_dev, (cudaStream_t)stream);
}

extern "C" int yg_pooled_stats(yg_ensemble *e, double *out_dev, void *stream)
{
    int rc = check_handle(e, true, true);
    if (rc) return rc;
    if (!out_dev) return YG_ERR_INVALID;
    if (e->cfg.dim > YG_MAX_DIM) {
        yg_set_error("pooled statistics need the full second-moment matrix (dim <= %d)", YG_MAX_DIM);
        return YG_ERR_UNSUPPORTED;
    }
    YG_CUDA_CHECK(cudaSetDevice(e->cfg.device));
    return yg_pooled_impl(static_cast<const double *>(e->buf[SB_W_MEAN]), static_cast<const double *>(e->buf[SB_W_M2]),
                          static_cast<const unsigned long long *>(e->buf[SB_N_ACCEPT]), e->cfg.dim, e->cfg.n_chains,
                          e->welford_n, e->pool_partials, POOL_PARTS, out_dev, (cudaStream_t)stream);
}

extern "C" int yg_last_launch(yg_ensemble *e, int32_t *grid, int32_t *block, int32_t *smem_bytes, int64_t *launches)
{
    if (!e) return YG_ERR_INVALID;
    if (grid) *grid = e->last_grid;
    if (block) *block = e->last_block;
    if (smem_bytes) *smem_bytes = e->last_smem;
    if (launches) *launches = e->launches;
    return YG_OK;
}

extern "C" int yg_fp64_tensor_peak(int32_t device, double ms, double *tflops_out)
{
    if (!tflops_out) return YG_ERR_INVALID;
    return yg_dmma_peak(device, ms, tflops_out);
}

