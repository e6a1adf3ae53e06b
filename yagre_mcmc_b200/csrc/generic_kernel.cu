// generic_kernel.cu -- host dispatch of the one-chain-per-thread kernels (generic_kernel.cuh) over the
// capacity classes (D, DD) in {2, 4, 8}^2; the kernels are instantiated per D in generic_d{2,4,8}.cu.
#include "ensemble.h"
#include <algorithm>

int yg_launch_generic_d2(yg_ensemble *e, const RunArgs &a, cudaStream_t st, int cdd);
int yg_launch_generic_d4(yg_ensemble *e, const RunArgs &a, cudaStream_t st, int cdd);
int yg_launch_generic_d8(yg_ensemble *e, const RunArgs &a, cudaStream_t st, int cdd);
int yg_launch_logpost_d2(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st, int cdd);
int yg_launch_logpost_d4(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st, int cdd);
int yg_launch_logpost_d8(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st, int cdd);

namespace {
int cap_of(int n) { return n <= 2 ? 2 : (n <= 4 ? 4 : 8); }
}  // namespace

int yg_launch_generic(yg_ensemble *e, const RunArgs &a, cudaStream_t st)
{
    const DevProblemHeader *hp = reinterpret_cast<const DevProblemHeader *>(e->h_problem.data());
    const int cd = cap_of(hp->dim);
    const int cdd = cap_of(std::max(1, std::max(hp->lvl[0].data_dim, std::max(hp->lvl[1].data_dim, hp->lvl[2].data_dim))));
    int rc = YG_ERR_UNSUPPORTED;
    if (hp->dim <= 8 && std::max(hp->lvl[0].data_dim, std::max(hp->lvl[1].data_dim, hp->lvl[2].data_dim)) <= 8) {
#ifdef YG_DEV_22
        if (cd == 2) rc = yg_launch_generic_d2(e, a, st, cdd);
#else
        rc = cd == 2 ? yg_launch_generic_d2(e, a, st, cdd)
                     : (cd == 4 ? yg_launch_generic_d4(e, a, st, cdd) : yg_launch_generic_d8(e, a, st, cdd));
#endif
    }
    if (rc == YG_ERR_UNSUPPORTED) yg_set_error("unsupported dimensions d=%d data_dim=%d", hp->dim, hp->lvl[0].data_dim);
    return rc;
}

int yg_launch_logpost(yg_ensemble *e, int level, const double *theta, int64_t n, double *out, cudaStream_t st)
{
    const DevProblemHeader *hp = reinterpret_cast<const DevProblemHeader *>(e->h_problem.data());
    const int cd = cap_of(hp->dim);
    const int cdd = cap_of(std::max(1, std::max(hp->lvl[0].data_dim, std::max(hp->lvl[1].data_dim, hp->lvl[2].data_dim))));
    int rc = YG_ERR_UNSUPPORTED;
    if (hp->dim <= 8 && std::max(hp->lvl[0].data_dim, std::max(hp->lvl[1].data_dim, hp->lvl[2].data_dim)) <= 8) {
#ifdef YG_DEV_22
        if (cd == 2) rc = yg_launch_logpost_d2(e, level, theta, n, out, st, cdd);
#else
        rc = cd == 2 ? yg_launch_logpost_d2(e, level, theta, n, out, st, cdd)
                     : (cd == 4 ? yg_launch_logpost_d4(e, level, theta, n, out, st, cdd)
                                : yg_launch_logpost_d8(e, level, theta, n, out, st, cdd));
#endif
    }
    if (rc == YG_ERR_UNSUPPORTED) yg_set_error("unsupported dimensions d=%d data_dim=%d", hp->dim, hp->lvl[0].data_dim);
    return rc;
}
