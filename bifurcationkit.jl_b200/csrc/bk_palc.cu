// bk_palc.cu -- bk_palc_run: the PALC loop of bk_palc_loop.hpp on the device backend (SURVEY.md 8(b), optional entry).
// The backend is the library's own C ABI with device pointers, i.e. exactly the calls the plugin-surface loop makes
// (julia/BK200.jl under continuation(...), bifurcationkit.jl_b200/palc.py) -- same kernels, same order, same bits --
// minus the host-language dispatch and the per-call allocations between them.
#include <cstring>
#include "bk_common.cuh"
#include "bk_palc_loop.hpp"

namespace {

struct AbiFailure {
  int status;
};

struct DeviceBackend {
  using Vec = double*;
  bk_ctx* c;
  const bk_palc_opts* po;
  const bk_gmres_opts* go;
  double par[BK_MAX_PAR];

  DeviceBackend(bk_ctx* ctx, const bk_palc_opts* p, const bk_gmres_opts* g) : c(ctx), po(p), go(g) {
    memcpy(par, ctx->par, sizeof par);
  }
  void chk(int st) const {
    if (st < 0) throw AbiFailure{st};
  }
  long long size() const { return c->N; }
  Vec alloc() {
    double* p = nullptr;
    chk(bk_vec_alloc(c, c->N, &p));
    return p;
  }
  void release(Vec v) { bk_vec_free(c, v); }
  void copy(Vec dst, Vec src) { chk(bk_vec_copy(c, dst, src, c->N)); }
  void zero(Vec x) { chk(bk_vec_zero(c, x, c->N)); }
  void axpby(Vec y, double a, Vec x, double b) { chk(bk_vec_axpby(c, y, a, x, b, c->N)); }
  void scale(Vec x, double a) { chk(bk_vec_scale(c, x, a, c->N)); }
  double dot(Vec x, Vec y) {
    double d = 0;
    chk(bk_vec_dot(c, x, y, c->N, &d));
    return d;
  }
  double diffdot(Vec x, Vec x0, Vec tau) {
    double d = 0;
    chk(bk_vec_diffdot(c, x, x0, tau, c->N, &d));
    return d;
  }
  double norm2(Vec x) {
    double d = 0;
    chk(bk_vec_norm2(c, x, c->N, &d));
    return d;
  }
  double normC(Vec x) {
    double d = 0;
    chk(po->normc == 1 ? bk_vec_norminf(c, x, c->N, &d) : bk_vec_norm2(c, x, c->N, &d));
    return d;
  }
  void set(double p) {
    par[po->lens] = p;
    chk(bk_set_params(c, par, BK_MAX_PAR));
  }
  void residual(Vec x, double p, Vec out) {
    set(p);
    chk(bk_residual(c, x, out));
  }
  void jacobian(Vec x, double p) {
    set(p);
    chk(bk_jac_set_state(c, x));
  }
  bool linsolve(Vec rhs, Vec out, int& iters) {
    int32_t cv = 0, it = 0;
    chk(bk_gmres(c, rhs, out, 0.0, 1.0, go, &cv, &it, nullptr));
    iters = it;
    return cv != 0;
  }
  bool bls(Vec dR, Vec dzu, double dzp, Vec R, double n, double xiu, double xip, double dotscale, Vec dX, double& dl, int& iters) {
    int32_t cv = 0;
    if (po->bls == 1) {
      int32_t it[2] = {0, 0};
      chk(bk_bls_bordering(c, dR, dzu, dzp, R, n, xiu, xip, 0, 0.0, dotscale, go, po->bls_check_precision, po->bls_k > 0 ? po->bls_k : 1,
                           po->bls_tol, dX, &dl, &cv, it));
      iters = it[0] + it[1];
    } else {
      int32_t it = 0;
      chk(bk_bls_matrixfree(c, dR, dzu, dzp, R, n, xiu, xip, 0, 0.0, dotscale, go, dX, &dl, &cv, &it));
      iters = it;
    }
    return cv != 0;
  }
};

struct CallbackThunk {
  bk_palc_callback cb;
  void* user;
};
bool thunk(void* t, int step, const double* row, double* z_u, double z_p) {
  auto* k = static_cast<CallbackThunk*>(t);
  return k->cb(k->user, step, row, z_u, z_p) != 0;
}

}  // namespace

extern "C" int32_t bk_palc_run(bk_ctx* c, const bk_palc_opts* po, const bk_gmres_opts* go, const double* u0, double p0,
                               const double* u1, double p1, double* rows, int32_t max_rows, bk_palc_callback cb, void* user,
                               double* u_final, bk_palc_result* result) {
  BK_ENTER(c);
  BkRange nvtx_range("bk_palc_run");
  BK_CHECK(c, po && go && u0 && rows && max_rows >= 1, "bk_palc_run: opts, linsolver, u0 and rows are required");
  BK_CHECK(c, po->lens >= 0 && po->lens < BK_MAX_PAR, "bk_palc_run: lens out of range");
  BK_CHECK(c, !c->cplx && c->N == c->N0, "bk_palc_run: real contexts only");
  BK_CHECK(c, c->kind != BK_SPARSE,
           "bk_palc_run: a BK_SPARSE context has no residual (F is the caller's function); run the continuation loop on the host");
  BK_CHECK(c, po->newton_maxit >= 1 && po->dsmin > 0 && po->dsmax >= po->dsmin, "bk_palc_run: bad step / Newton limits");
  const long long N = c->N;
  bkpalc::Opts o;
  o.ds = po->ds, o.dsmin = po->dsmin, o.dsmax = po->dsmax, o.a = po->a, o.p_min = po->p_min, o.p_max = po->p_max;
  o.theta = po->theta, o.eta = po->eta, o.newton_tol = po->newton_tol, o.fd_eps = po->fd_eps;
  o.max_steps = po->max_steps, o.newton_maxit = po->newton_maxit, o.tangent = po->tangent;
  double saved_par[BK_MAX_PAR];
  memcpy(saved_par, c->par, sizeof saved_par);
  int status = BK_OK;
  // host inputs are uploaded once; everything in between stays on the device
  double *d0 = nullptr, *d1 = nullptr, *df = nullptr;
  auto stage = [&](const double* h, double** d) -> int {
    if (bk_is_device_ptr(h)) {
      *d = const_cast<double*>(h);
      return BK_OK;
    }
    BK_TRY(bk_vec_alloc(c, N, d));
    return bk_vec_upload(c, *d, h, N);
  };
  BK_TRY(stage(u0, &d0));
  if (u1) BK_TRY(stage(u1, &d1));
  if (u_final) {
    if (bk_is_device_ptr(u_final))
      df = u_final;
    else
      BK_TRY(bk_vec_alloc(c, N, &df));
  }
  bkpalc::Result R;
  try {
    DeviceBackend be(c, po, go);
    bkpalc::Loop<DeviceBackend> loop(be, o);
    CallbackThunk t{cb, user};
    R = loop.run(d0, p0, d1, u1 != nullptr, p1, rows, max_rows, cb ? &thunk : nullptr, &t, df);
  } catch (const AbiFailure& f) {
    status = f.status;  // bk_last_error holds the message of the failing call
  } catch (const bkpalc::StartupFailure& f) {
    status = bk_fail(c, BK_ERR_STATE, f.what(), __FILE__, __LINE__);
  } catch (const std::exception& f) {
    status = bk_fail(c, BK_ERR_STATE, f.what(), __FILE__, __LINE__);
  }
  memcpy(c->par, saved_par, sizeof saved_par);  // the caller's parameter tuple is left as it was
  if (status == BK_OK && u_final && df != u_final) status = bk_vec_download(c, u_final, df, N);
  if (d0 != u0) bk_vec_free(c, d0);
  if (d1 && d1 != u1) bk_vec_free(c, d1);
  if (df && df != u_final) bk_vec_free(c, df);
  if (result) {
    result->nrows = R.nrows, result->steps = R.steps, result->nfail = R.nfail, result->stopped = R.stopped;
    result->work_newton = R.work_newton, result->work_linear = R.work_linear;
    result->p_final = R.z_p, result->ds_final = R.ds;
  }
  return status;
}
