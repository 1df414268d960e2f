// Device-resident EP sweep for the chain  prior -> x -> LinearChannel -> z -> likelihood.
//
// reference: algos/message_passing.py:330-357 (iterate), :249-269 (forward /
// backward pass, update_variables), :70-127 (constant damping), :187-209 (NaN
// check); algos/callbacks.py:250-286 (EarlyStoppingEP); algos/metrics.py:5-14.
//
// One iteration = 9 stages on one stream (7 launches: S1 and S2 run inside the projections P1 and P3
// when the operator passes are GEMVs), B instances in lock step, no host round trip (edge
// numbering e1..e8 as in SURVEY 3.3):
//   F1  factor_message(prior)   e8 -> e1 (=e2)
//   P1  project  V_R^T b2       -> tz
//   S1  rescale fwd             -> coef, vx(lin)
//   P2  expand   U_R coef       -> part
//   Z   z_update: e3 (=e4), likelihood e5 (=e6), posterior of z
//   P3  project  U_R^T b6       -> tx        (reused by the next iteration's S1)
//   S2  rescale bwd             -> coef, vz(lin)
//   P4  expand   V_R coef       -> part
//   X   x_update: e7 (=e8), posterior of x, MSE / tolerance records, early stop
// Each operator is streamed exactly twice per iteration (once as A^T x, once
// as A c): 16*R*(N+M) bytes per instance-iteration.
#include "trb_moments.cuh"
#include "trb_updates.cuh"

using namespace trb;

namespace {

constexpr int kUpThreads = 512;

constexpr int kUnroll = 2;  // elements per thread whose loads are issued together (2 CTAs of 512 threads per SM)

// stats[b*4 + {0,1}] = sum (r_new - r_old)^2, sum r_new^2 for z
// light (schedule 2): only the scalars of e3 and the constant Gaussian-likelihood
// message e5 are updated; e3's vector, the posterior mean of z and its tolerance
// statistics wait for the last iteration of the run.
__global__ void __launch_bounds__(kUpThreads, 2)
k_z_update(trb_sweep sw, int G, int first, int light, double* __restrict__ stats, trb_peers peers) {
  __shared__ double sh[33 * 2];
  __shared__ int sh_flag;
  const int b = blockIdx.y;  // grid (C, B): a cluster of C CTAs per instance
  if (sw.active && !sw.active[b]) return;
  const int T = blockDim.x * cluster_nctarank();
  const int gtid = cluster_ctarank() * blockDim.x + threadIdx.x;
  const int B = sw.B, M = sw.M, ld = sw.ldm;
  const size_t off = (size_t)b * ld;
  double* ea = sw.edge_a;
  const double a6 = ea[5 * B + b];
  const double a3n = clip_a_new(sw.vlin[b], a6, sw.lin_amin, sw.lin_amax);  // base_channel.py:9-12
  const double a3 = damp(sw.damp3, ea[2 * B + b], a3n);
  const double ainv3 = a6 + a3n;
  const int ns = slots_of(b, sw.R, B, G);
  const double* part = sw.part + (size_t)b * sw.nslots * ld;
  const double* b6 = ((first && sw.b6_init) ? sw.b6_init : sw.b5) + off;
  double* b3 = sw.b3 + off;
  double* b5 = sw.b5 + off;
  double* rz = sw.rz + off;
  double* scr = sw.scr_m + off;
  const double* y = sw.y + off;
  const bool const_lik = factor_is_constant_message(sw.lik.kind);
  // every overwritten value is first copied to the one-iteration-back state (the reference's
  // old_message_dag, message_passing.py:356): no separate copy kernel per iteration
  const bool snap = sw.snap_edge_a != nullptr;
  const int step = T * kUnroll;
  int flag = 0;
  double vsum = 0.0;
  // row-sharded operator: the expansion is the sum of the ranks' vectors, read
  // from peer memory once every rank has published this exchange (trb_comm.cu)
  const bool use_peers = peers.n > 0 && !light;
  if (use_peers && !peers_wait(peers)) flag |= TRB_FLAG_COMM_TIMEOUT;
  // pass 1: e3 (= e4) and the likelihood moments at (a3, b3)
  for (int base = gtid; base < (light ? 0 : M); base += step) {
    double rx[kUnroll], b6v[kUnroll], b3o[kUnroll], yv[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int i = base + u * T;
      rx[u] = 0.0;
      if (i < M) {
        if (use_peers) rx[u] = peers_sum(peers, off + i);
        else for (int sl = 0; sl < ns; ++sl) rx[u] += part[(size_t)sl * ld + i];
        b6v[u] = b6[i];
        b3o[u] = b3[i];
        yv[u] = y[i];
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int i = base + u * T;
      if (i < M) {
        const double b3n = rx[u] * ainv3 - b6v[u];
        if (b3n != b3n) flag |= TRB_FLAG_NAN_B;
        const double b3v = damp(sw.damp3, b3o[u], b3n);
        if (snap) sw.snap_b3[off + i] = b3o[u];
        b3[i] = b3v;
        if (!const_lik) {
          const RV m = factor_moments(sw.lik, a3, b3v, yv[u]);
          scr[i] = m.r;
          vsum += m.v;
        }
      }
    }
  }
  double a5n;
  if (const_lik) {
    a5n = sw.lik.p0;  // gaussian_likelihood.py:68-71
  } else {
    const double v = cluster_sum(vsum, sh) / M;
    a5n = clip_a_new(v, a3, sw.lik.amin, sw.lik.amax);  // base_likelihood.py:25-28
  }
  const double a5 = damp(sw.damp5, ea[4 * B + b], a5n);
  const double ainv5 = a3 + a5n;
  const double a_hat = a3 + a5;
  double red[2] = {0.0, 0.0};
  // pass 2: e5 (= e6) and the posterior of z
  for (int base = gtid; base < M; base += step) {
    double b3v[kUnroll], src[kUnroll], b5o[kUnroll], ro[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int i = base + u * T;
      if (i < M) {
        b3v[u] = b3[i];
        src[u] = const_lik ? y[i] : scr[i];
        b5o[u] = b5[i];
        ro[u] = rz[i];
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int i = base + u * T;
      if (i < M) {
        const double b5n = const_lik ? src[u] * sw.lik.p0 : src[u] * ainv5 - b3v[u];
        if (b5n != b5n) flag |= TRB_FLAG_NAN_B;
        const double b5v = damp(sw.damp5, b5o[u], b5n);
        if (snap) sw.snap_b5[off + i] = b5o[u];
        b5[i] = b5v;
        if (light) continue;
        const double rnew = (b3v[u] + b5v) / a_hat;  // base.py:152-161
        if (snap) sw.snap_rz[off + i] = ro[u];
        rz[i] = rnew;
        red[0] += (rnew - ro[u]) * (rnew - ro[u]);
        red[1] += rnew * rnew;
      }
    }
  }
  cluster_sum_n<2>(red, sh);
  if (a3n != a3n || a5n != a5n) flag |= TRB_FLAG_NAN_A;
  if (a3n < 0 || a5n < 0) flag |= TRB_FLAG_NEG_A;
  const int all = cluster_or(flag, &sh_flag);
  if (gtid == 0) z_tail(sw, b, light, stats, a3, a5, a_hat, all, red[0], red[1]);
}

__global__ void __launch_bounds__(kUpThreads, 2)
k_x_update(trb_sweep sw, int G, int it_host, double* __restrict__ stats, trb_peers peers) {
  __shared__ double sh[33 * 4];
  __shared__ int sh_flag;
  const int b = blockIdx.y;  // grid (C, B): a cluster of C CTAs per instance
  if (sw.active && !sw.active[b]) return;
  // it < 0 (replayed CUDA graph): the iteration index is the instance's own count of
  // completed iterations, which equals the host's index while the instance is active
  const int it = it_host >= 0 ? it_host : sw.n_iter[b];
  const int T = blockDim.x * cluster_nctarank();
  const int gtid = cluster_ctarank() * blockDim.x + threadIdx.x;
  const int B = sw.B, N = sw.N, ld = sw.ldn;
  const size_t off = (size_t)b * ld;
  double* ea = sw.edge_a;
  const double a1 = ea[1 * B + b];  // e2 (= e1)
  const double a7n = clip_a_new(sw.vlin[b], a1, sw.lin_amin, sw.lin_amax);  // base_channel.py:14-17
  const double a7 = damp(sw.damp7, ea[6 * B + b], a7n);
  const double ainv7 = a1 + a7n;
  const double a_hat = a1 + a7;
  const int ns = slots_of(b, sw.R, B, G);
  const double* part = sw.part + (size_t)b * sw.nslots * ld;
  const bool null_space = (sw.R_total > 0 ? sw.R_total : sw.R) < N;
  const double* b1 = sw.b1 + off;
  double* b7 = sw.b7 + off;
  double* rx = sw.rx + off;
  const double* xt = sw.x_true ? sw.x_true + off : nullptr;
  const int step = T * kUnroll;
  int flag = 0;
  const bool use_peers = peers.n > 0;  // row-sharded operator, see k_z_update
  if (use_peers && !peers_wait(peers)) flag |= TRB_FLAG_COMM_TIMEOUT;
  const bool snap = sw.snap_edge_a != nullptr;  // see k_z_update
  double red[4] = {0.0, 0.0, 0.0, 0.0};  // sum dr^2, sum r^2, sum (r-x)^2, sum (r+x)^2
  for (int base = gtid; base < N; base += step) {
    double rzv[kUnroll], b1v[kUnroll], b7o[kUnroll], ro[kUnroll], xv[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int i = base + u * T;
      rzv[u] = 0.0;
      xv[u] = 0.0;
      if (i < N) {
        if (use_peers) rzv[u] = peers_sum(peers, off + i);
        else for (int sl = 0; sl < ns; ++sl) rzv[u] += part[(size_t)sl * ld + i];
        b1v[u] = b1[i];
        b7o[u] = b7[i];
        ro[u] = rx[i];
        if (xt) xv[u] = xt[i];
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const int i = base + u * T;
      if (i < N) {
        double r = rzv[u];
        if (null_space) r = b1v[u] / a1 + r;
        const double b7n = r * ainv7 - b1v[u];
        if (b7n != b7n) flag |= TRB_FLAG_NAN_B;
        const double b7v = damp(sw.damp7, b7o[u], b7n);
        if (snap) {
          sw.snap_b7[off + i] = b7o[u];
          sw.snap_rx[off + i] = ro[u];
        }
        b7[i] = b7v;
        const double rnew = (b1v[u] + b7v) / a_hat;
        rx[i] = rnew;
        red[0] += (rnew - ro[u]) * (rnew - ro[u]);
        red[1] += rnew * rnew;
        red[2] += (rnew - xv[u]) * (rnew - xv[u]);  // metrics.py:5-6
        red[3] += (rnew + xv[u]) * (rnew + xv[u]);  // metrics.py:9-14
      }
    }
  }
  cluster_sum_n<4>(red, sh);
  const double d2 = red[0], n2 = red[1], e_pos = red[2], e_neg = red[3];
  if (a7n != a7n) flag |= TRB_FLAG_NAN_A;
  if (a7n < 0) flag |= TRB_FLAG_NEG_A;
  const int all = cluster_or(flag, &sh_flag);
  if (gtid == 0) x_tail(sw, b, it, stats, a7, a_hat, all, d2, n2, e_pos, e_neg);
}

// ---- chunked update kernels ---------------------------------------------------------------
// The z / x updates are maps over the instance vector plus a few sums.  One CTA (or cluster) per
// instance walks its vector in rounds of a few loads per thread behind a chain of dependent
// accesses (flag -> scalars -> elements -> further slots), and the latencies add up (ncu,
// profiles/r02c_ncu_update_kernels.json: these kernels follow the SM clock and the length of that
// chain, not HBM).  Here an instance is cut into chunks of kChunk elements, one small CTA each
// (grid (chunks, B), 3-4 CTAs per SM), every thread
// issues ALL its loads at once -- flag, scalars and elements (trb_updates.cuh) -- the CTA's sums
// meet in thread 0 after ONE barrier, and go to a scratch row of the instance; the thread whose
// chunk arrives last (acq_rel counter, column 3 of `stats`) adds the chunks in chunk order -- the
// result does not depend on the arrival order -- and writes the instance's scalars (z_tail /
// x_tail).  Per element the arithmetic is that of k_z_update / k_x_update, bit for bit.
// Chunk = 1024 elements for both; threads x elements per thread as measured at the north-star
// shape (ncu, us per launch): z 256 x 4 22.7 (128 x 8: 25.4), x 128 x 8 40.1 (256 x 4: 41.6) -- the
// x update has the longer per-thread prologue to amortise.  Registers: all loads of a thread stay
// in registers (85 at 3 CTAs per SM, 128 at 4).
constexpr int kChunk = 1024;
constexpr int kZcThreads = 256, kZcE = kChunk / kZcThreads, kZcCtasPerSm = 3;
constexpr int kXcThreads = 128, kXcE = kChunk / kXcThreads, kXcCtasPerSm = 4;
constexpr int kZPartials = 3, kXPartials = 5;  // sums + flags per chunk

// Gaussian likelihood (constant message e5, gaussian_likelihood.py:68-71): no sum is needed
// before the second half of the update, so the whole z update is one pass.
__global__ void __launch_bounds__(kZcThreads, kZcCtasPerSm)
k_z_update_chunked(trb_sweep sw, int G, int first, double* __restrict__ stats, trb_peers peers) {
  __shared__ double sh[2 * 8];
  __shared__ int shi[8];
  const int b = blockIdx.y, chunk = blockIdx.x, nchunk = gridDim.x;
  // every load first: flag, scalars, elements (independent addresses), then the first look
  const int act = sw.active ? sw.active[b] : 1;
  const ZRaw raw = z_raw(sw, b);
  const int ns = slots_of(b, sw.R, sw.B, G);
  const int start = chunk * kChunk + (int)threadIdx.x;
  ZLoads<kZcE> l;
  z_load<kZcE>(sw, b, ns, first, &peers, start, kZcThreads, l);
  if (!act) return;
  const ZScalars z = z_scalars(sw, raw);
  int flag = z_scalar_flags(z);
  if (peers.n > 0 && !peers_wait(peers)) flag |= TRB_FLAG_COMM_TIMEOUT;
  double red[2] = {0.0, 0.0};
  z_compute<kZcE>(sw, b, ns, &peers, z, start, kZcThreads, l, red, flag);
  cta_sums_to_thread0<2>(red, flag, sh, shi);
  if (threadIdx.x != 0) return;
  double* partials = sw.scr_m + (size_t)b * sw.ldm;  // free here: the likelihood parks nothing
  partials[chunk * kZPartials + 0] = red[0];
  partials[chunk * kZPartials + 1] = red[1];
  partials[chunk * kZPartials + 2] = (double)flag;
  unsigned int* cnt = reinterpret_cast<unsigned int*>(stats) + (size_t)b * 8 + 6;
  if (!chunk_arrive_last(cnt, nchunk)) return;
  double d2 = 0.0, n2 = 0.0;
  int all = 0;
  for (int c = 0; c < nchunk; ++c) {
    d2 += __ldcg(partials + c * kZPartials + 0);
    n2 += __ldcg(partials + c * kZPartials + 1);
    all |= (int)__ldcg(partials + c * kZPartials + 2);
  }
  z_tail(sw, b, 0, stats, z.a3, z.a5, z.a_hat, all, d2, n2);
}

__global__ void __launch_bounds__(kXcThreads, kXcCtasPerSm)
k_x_update_chunked(trb_sweep sw, int G, int it_host, double* __restrict__ stats, trb_peers peers) {
  __shared__ double sh[4 * 8];
  __shared__ int shi[8];
  const int b = blockIdx.y, chunk = blockIdx.x, nchunk = gridDim.x;
  const int act = sw.active ? sw.active[b] : 1;
  const XRaw raw = x_raw(sw, b);
  const int ns = slots_of(b, sw.R, sw.B, G);
  const int start = chunk * kChunk + (int)threadIdx.x;
  XLoads<kXcE> l;
  x_load<kXcE>(sw, b, ns, &peers, start, kXcThreads, l);
  if (!act) return;
  const XScalars x = x_scalars(sw, raw);
  int flag = x_scalar_flags(x);
  if (peers.n > 0 && !peers_wait(peers)) flag |= TRB_FLAG_COMM_TIMEOUT;
  double red[4] = {0.0, 0.0, 0.0, 0.0};
  x_compute<kXcE>(sw, b, ns, &peers, x, start, kXcThreads, l, red, flag);
  cta_sums_to_thread0<4>(red, flag, sh, shi);
  if (threadIdx.x != 0) return;
  double* partials = sw.scr_n + (size_t)b * sw.ldn;  // free here: the prior's scratch, rewritten by the next F1
#pragma unroll
  for (int k = 0; k < 4; ++k) partials[chunk * kXPartials + k] = red[k];
  partials[chunk * kXPartials + 4] = (double)flag;
  unsigned int* cnt = reinterpret_cast<unsigned int*>(stats) + (size_t)b * 8 + 7;
  if (!chunk_arrive_last(cnt, nchunk)) return;
  const int it = it_host >= 0 ? it_host : sw.n_iter[b];  // see k_x_update
  double t[4] = {0.0, 0.0, 0.0, 0.0};
  int all = 0;
  for (int c = 0; c < nchunk; ++c) {
#pragma unroll
    for (int k = 0; k < 4; ++k) t[k] += __ldcg(partials + c * kXPartials + k);
    all |= (int)__ldcg(partials + c * kXPartials + 4);
  }
  x_tail(sw, b, it, stats, x.a7, x.a_hat, all, t[0], t[1], t[2], t[3]);
}

// One-iteration-back snapshot of the message state, per instance:
//   active instance                      -> save   (old_message_dag = message_dag.copy(), :356)
//   stopped on NaN / divergence, once    -> restore (reset_message_dag, :196-197, callbacks.py:281-283)
// restore_only: the update kernels keep the one-iteration-back state themselves (every value
// is copied to its snap_* buffer before it is overwritten), so nothing is saved here.
__global__ void __launch_bounds__(256)
k_snapshot(trb_sweep sw, int restore_only) {
  const int b = blockIdx.y;  // grid (chunks, B), plain CTAs: pure copies
  const int B = sw.B;
  const size_t gtid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t T = (size_t)gridDim.x * blockDim.x;
  const int flags = sw.flags[b];
  const bool save = sw.active[b] != 0 && !restore_only;
  const bool restore = !save && (flags & (TRB_FLAG_DIVERGED | TRB_FLAG_NAN_A | TRB_FLAG_NAN_B)) &&
                       !(flags & TRB_FLAG_RESTORED);
  if (!save && !restore) return;
  auto copy = [&](double* live, double* snap, size_t n) {
    double* dst = save ? snap : live;
    const double* src = save ? live : snap;
    for (size_t i = gtid; i < n; i += T) dst[i] = src[i];
  };
  copy(sw.b1 + (size_t)b * sw.ldn, sw.snap_b1 + (size_t)b * sw.ldn, sw.N);
  copy(sw.b7 + (size_t)b * sw.ldn, sw.snap_b7 + (size_t)b * sw.ldn, sw.N);
  copy(sw.rx + (size_t)b * sw.ldn, sw.snap_rx + (size_t)b * sw.ldn, sw.N);
  copy(sw.b3 + (size_t)b * sw.ldm, sw.snap_b3 + (size_t)b * sw.ldm, sw.M);
  copy(sw.b5 + (size_t)b * sw.ldm, sw.snap_b5 + (size_t)b * sw.ldm, sw.M);
  copy(sw.rz + (size_t)b * sw.ldm, sw.snap_rz + (size_t)b * sw.ldm, sw.M);
  copy(sw.tx + (size_t)b * sw.R, sw.snap_tx + (size_t)b * sw.R, sw.R);
  if (blockIdx.x != 0) return;
  if (threadIdx.x < 8) {
    double* live = sw.edge_a + (size_t)threadIdx.x * B + b;
    double* snap = sw.snap_edge_a + (size_t)threadIdx.x * B + b;
    if (save) *snap = *live; else *live = *snap;
  }
  if (threadIdx.x == 8) { if (save) sw.snap_vx[b] = sw.vx[b]; else sw.vx[b] = sw.snap_vx[b]; }
  if (threadIdx.x == 9) { if (save) sw.snap_vz[b] = sw.vz[b]; else sw.vz[b] = sw.snap_vz[b]; }
}

// after every CTA of k_snapshot is done: remember which instances were rolled back
__global__ void k_snapshot_mark(trb_sweep sw) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= sw.B) return;
  const int flags = sw.flags[b];
  if (sw.active[b] == 0 && (flags & (TRB_FLAG_DIVERGED | TRB_FLAG_NAN_A | TRB_FLAG_NAN_B)) &&
      !(flags & TRB_FLAG_RESTORED))
    sw.flags[b] = flags | TRB_FLAG_RESTORED;
}

// Schedules 1, 2: U_R^T b5' for the Gaussian-likelihood message b5' = d5 b5 + (1-d5) y/var
// (gaussian_likelihood.py:68-71, message_passing.py:119-127), from tx = U_R^T b5.
__global__ void __launch_bounds__(256)
k_tx_recur(trb_sweep sw) {
  const int b = blockIdx.y;
  if (sw.active && !sw.active[b]) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= sw.R) return;
  const size_t o = (size_t)b * sw.R + i;
  const double told = sw.tx[o];
  if (sw.snap_tx) sw.snap_tx[o] = told;  // one-iteration-back state, see k_z_update
  sw.tx[o] = damp(sw.damp5, told, sw.lik.p0 * sw.ty[o]);
}

}  // namespace

// Which update kernels run chunked (trb_set_update_kernels, TRB_UPDATE_KERNELS=<mask>): bit 0 the x
// update, bit 1 the z update with a Gaussian likelihood.  A cleared bit: one CTA / cluster per
// instance.  Default: both.
constexpr int kUpdateKernelsAll = 3;
static int g_update_kernels = -1;

static int update_kernels() {
  if (g_update_kernels < 0) {
    const char* e = getenv("TRB_UPDATE_KERNELS");
    g_update_kernels = e ? (atoi(e) & kUpdateKernelsAll) : kUpdateKernelsAll;
  }
  return g_update_kernels;
}

extern "C" void trb_set_update_kernels(int mask) {
  g_update_kernels = mask < 0 ? -1 : (mask & kUpdateKernelsAll);
}

#define TRB_TRY(expr)      \
  do {                     \
    int rc_ = (expr);      \
    if (rc_) return rc_;   \
  } while (0)

static int check_sweep(const trb_sweep* sw) {
  TRB_CHECK_ARG(sw, "null sweep descriptor");
  TRB_CHECK_ARG(sw->B > 0 && sw->N > 0 && sw->M > 0 && sw->R > 0, "bad shape");
  // every per-instance launch of the sweep puts the instance index in gridDim.y
  TRB_CHECK_ARG(sw->B <= 65535, "B > 65535");
  TRB_CHECK_ARG(sw->R <= sw->N && sw->R <= sw->M, "R must be <= min(N, M)");
  TRB_CHECK_ARG(sw->y, "null observation");
  TRB_CHECK_ARG(sw->edge_a && sw->b1 && sw->b3 && sw->b5 && sw->b7, "null message buffer");
  TRB_CHECK_ARG(sw->rx && sw->rz && sw->vx && sw->vz, "null posterior buffer");
  TRB_CHECK_ARG(sw->tz && sw->tx && sw->coef && sw->part && sw->scr_n && sw->scr_m && sw->vlin &&
                    sw->stats,
                "null scratch buffer");
  TRB_CHECK_ARG(sw->active && sw->flags && sw->n_iter, "null status buffer");
  TRB_CHECK_ARG(sw->es_mode == 0 || (sw->es_mode == 1 && (sw->es_tol < 0 || sw->snap_edge_a)),
                "the variance early stopping needs the snapshot buffers");
  TRB_CHECK_ARG(!sw->snap_edge_a || (sw->snap_b1 && sw->snap_b3 && sw->snap_b5 && sw->snap_b7 &&
                                     sw->snap_rx && sw->snap_rz && sw->snap_vx && sw->snap_vz &&
                                     sw->snap_tx),
                "incomplete snapshot buffers");
  return TRB_OK;
}

// Row-sharded operator: reduce this rank's slots and push the result into every
// rank's exchange buffer, then publish; the following update kernel adds the
// ranks' vectors from its own memory (trb_comm.cu).
int trb_reduce_slots_push(int B, int R, int n, int ld, const double* part, const trb_push* push,
                          void* stream);
int trb_factor_message_snap(const trb_factor* f, int B, int n, int ld, const double* a_in,
                            const double* b_in, const double* y, double* a_io, double* b_io,
                            double* a_copy, double damping, double* scratch, int* flags,
                            const int* active, double* snap_b, double* snap_a, double* snap_a_copy,
                            void* stream);
int trb_lin_rescale_snap(int dir, int B, int R, int Nz, int Nx, int rank, int null_space,
                         const double* s, const double* s2, int64_t stride_s, const double* az,
                         const double* ax, const double* tz, const double* tx, double* coef, double* v,
                         const int* active, double* snap_tx, void* stream);
int trb_lin_project_rescale(const double* A, int64_t strideA, int R, int n, int ld, int B,
                            const double* vec, int ldvec, double* t_out, const int* active, int dir,
                            int Nz, int Nx, int rank, int null_space, const double* s, const double* s2,
                            int64_t stride_s, const double* az, const double* ax, const double* t_other,
                            double* coef, double* v, double* snap_tx, void* stream);
// The push is NOT gated by `active`: every rank takes the same stop decision in the same
// iteration (the update kernels are computed redundantly on bit-identical sums), and a stopped
// instance's `part` is no longer rewritten by trb_lin_expand, so the ranks go on pushing and
// publishing identical stale vectors for the rest of the call while the consumers return before
// peers_wait -- the sequence numbers keep advancing in lock step on all ranks, which is what the
// double buffering of trb_comm.cu relies on.
static int exchange_expansion(const trb_sweep* sw, int n, int ld, cudaStream_t st) {
  trb_comm* comm = sw->comm;
  TRB_CHECK_ARG((size_t)sw->B * ld <= trb_comm_capacity(comm), "exchange buffer too small");
  trb_push push;
  trb_comm_begin_exchange(comm, &push);  // the reduction kernel's last CTA publishes
  return trb_reduce_slots_push(sw->B, sw->R, n, ld, sw->part, &push, st);
}

// One stage of the iteration (see the header comment of this file).  `first`:
// this is the first iteration after the messages were initialised.
// pre_reduced: the expansion result already sits, fully summed, in slot 0 of
// `part` (GEMM / multi-GPU back ends) instead of in per-CTA slots.
extern "C" int trb_sweep_stage(const trb_sweep* sw, int stage, int it, int first, int pre_reduced,
                               void* stream) {
  int rc = check_sweep(sw);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int B = sw->B;
  double* ea = sw->edge_a;
  const bool needs_ops = (stage == TRB_STAGE_PROJECT_Z || stage == TRB_STAGE_PROJECT_X_INIT ||
                          stage == TRB_STAGE_EXPAND_X || stage == TRB_STAGE_PROJECT_X ||
                          stage == TRB_STAGE_EXPAND_Z || stage == TRB_STAGE_PROJECT_Y);
  TRB_CHECK_ARG(!needs_ops || (sw->Vt && sw->Ut), "null operator");
  const bool needs_s = (stage == TRB_STAGE_RESCALE_FWD || stage == TRB_STAGE_RESCALE_BWD);
  TRB_CHECK_ARG(!needs_s || (sw->s && sw->s2), "null spectrum");
  const int R_total = sw->R_total > 0 ? sw->R_total : sw->R;
  const int null_space = R_total < sw->N;
  // operator passes as shared-operator DMMA GEMMs (trb_gemm.cu): the expansion
  // lands fully summed in slot 0 of `part`, like a pre-reduced back end
  const bool shared_ops = sw->strideV == 0 && sw->strideU == 0;
  TRB_CHECK_ARG(sw->gemv_impl != 3 || shared_ops, "gemv_impl 3 (GEMM) needs a shared operator");
  const bool gemm = shared_ops && (sw->gemv_impl == 3 || (sw->gemv_impl == 0 && B >= 16));
  if (gemm) pre_reduced = 1;
  trb_comm* comm = sw->comm;
  TRB_CHECK_ARG(!comm || (!gemm && sw->s_full && sw->s2_full && sw->R_total >= sw->R),
                "a row-sharded sweep needs GEMV operator passes, s_full, s2_full and R_total");
  // few instances over many CTAs: the expansion stages leave the slot sum in slot 0
  const bool reduce_first = !pre_reduced && !comm && sw->nslots > kTrbDirectSlots;
  if (reduce_first && (stage == TRB_STAGE_Z_UPDATE || stage == TRB_STAGE_X_UPDATE)) pre_reduced = 1;
  int G = 0;
  if (stage == TRB_STAGE_Z_UPDATE || stage == TRB_STAGE_Z_UPDATE_LIGHT ||
      stage == TRB_STAGE_X_UPDATE) {
    if (pre_reduced) {
      G = 0;  // ns = 1
    } else {
      const trb_expand_geom geo = trb_expand_geometry(B, sw->R);
      TRB_CHECK_ARG(sw->nslots == geo.nslots, "nslots must equal trb_lin_expand_slots(B, R)");
      G = geo.G;
    }
  }
  switch (stage) {
    case TRB_STAGE_PRIOR: {  // F1: reads e8, writes e1 and its pass-through copy e2
      const double* b8 = (first && sw->b8_init) ? sw->b8_init : sw->b7;
      double* sa = sw->snap_edge_a;
      return trb_factor_message_snap(&sw->prior, B, sw->N, sw->ldn, ea + 7 * B, b8, nullptr, ea + 0 * B,
                                     sw->b1, ea + 1 * B, sw->damp1, sw->scr_n, sw->flags, sw->active,
                                     sa ? sw->snap_b1 : nullptr, sa, sa ? sa + 1 * B : nullptr, stream);
    }
    case TRB_STAGE_PROJECT_Z:  // P1: tz = V_R^T b2
      if (gemm)
        return trb_lin_project_gemm(sw->Vt, sw->R, sw->N, sw->ldn, B, sw->b1, sw->ldn, sw->tz,
                                    stream);
      return trb_lin_project(sw->Vt, sw->strideV, sw->R, sw->N, sw->ldn, B, sw->b1, sw->ldn,
                             sw->tz, sw->active, sw->gemv_impl, stream);
    case TRB_STAGE_PROJECT_X_INIT: {  // tx = U_R^T b6 for the initial e6
      const double* b6 = sw->b6_init ? sw->b6_init : sw->b5;
      if (gemm)
        return trb_lin_project_gemm(sw->Ut, sw->R, sw->M, sw->ldm, B, b6, sw->ldm, sw->tx, stream);
      return trb_lin_project(sw->Ut, sw->strideU, sw->R, sw->M, sw->ldm, B, b6, sw->ldm, sw->tx,
                             sw->active, sw->gemv_impl, stream);
    }
    case TRB_STAGE_RESCALE_FWD:  // S1: coef = s res (tz + s tx), forward variance
    case TRB_STAGE_RESCALE_BWD:  // S2: coef for rz, backward variance
      if (comm) {  // variance from the whole (replicated) spectrum, coefficients from the shard
        const int dir = stage == TRB_STAGE_RESCALE_BWD;
        rc = trb_lin_rescale(dir, B, R_total, sw->N, sw->M, sw->rank, null_space, sw->s_full,
                             sw->s2_full, 0, ea + 1 * B, ea + 5 * B, nullptr, nullptr, nullptr,
                             sw->vlin, sw->active, stream);
        if (rc) return rc;
        return trb_lin_rescale_snap(dir, B, sw->R, sw->N, sw->M, sw->rank < sw->R ? sw->rank : sw->R,
                                    null_space, sw->s, sw->s2, sw->stride_s, ea + 1 * B, ea + 5 * B,
                                    sw->tz, sw->tx, sw->coef, nullptr, sw->active,
                                    (dir == 0 && sw->schedule == 0 && sw->snap_edge_a) ? sw->snap_tx : nullptr,
                                    stream);
      }
      if (stage == TRB_STAGE_RESCALE_BWD)
        return trb_lin_rescale(1, B, sw->R, sw->N, sw->M, sw->rank, null_space, sw->s, sw->s2,
                               sw->stride_s, ea + 1 * B, ea + 5 * B, sw->tz, sw->tx, sw->coef,
                               sw->vlin, sw->active, stream);
      // general schedule: P3 overwrites tx later in this iteration, so its old value is kept here
      // (schedules 1 and 2 update tx in k_tx_recur, which keeps it)
      return trb_lin_rescale_snap(0, B, sw->R, sw->N, sw->M, sw->rank, null_space, sw->s, sw->s2,
                                  sw->stride_s, ea + 1 * B, ea + 5 * B, sw->tz, sw->tx, sw->coef,
                                  sw->vlin, sw->active,
                                  (sw->schedule == 0 && sw->snap_edge_a) ? sw->snap_tx : nullptr, stream);
    case TRB_STAGE_EXPAND_X:  // P2: rx = U_R coef
      if (gemm)
        return trb_lin_expand_gemm(sw->Ut, sw->R, sw->M, sw->ldm, B, sw->coef, sw->part,
                                   sw->nslots * sw->ldm, stream);
      rc = trb_lin_expand(sw->Ut, sw->strideU, sw->R, sw->M, sw->ldm, B, sw->coef, sw->part,
                          sw->active, sw->gemv_impl, stream);
      if (rc) return rc;
      if (comm) return exchange_expansion(sw, sw->M, sw->ldm, st);
      if (!reduce_first) return rc;
      return trb_reduce_slots_inplace(B, sw->R, sw->M, sw->ldm, sw->part, stream);
    case TRB_STAGE_Z_UPDATE:          // Z: e3, likelihood e5, posterior z
    case TRB_STAGE_Z_UPDATE_LIGHT: {  // schedule 2: scalars and e5 only
      const int light = stage == TRB_STAGE_Z_UPDATE_LIGHT;
      TRB_CHECK_ARG(!light || sw->lik.kind == TRB_GAUSSIAN_LIKELIHOOD,
                    "the light z update needs a Gaussian likelihood");
      trb_launch_scope scope_(0, st);
      trb_peers peers = {};
      if (comm && !light) peers = *trb_comm_last(comm);
      const int zchunks = (sw->M + kChunk - 1) / kChunk;
      if ((update_kernels() & 2) && !light && sw->lik.kind == TRB_GAUSSIAN_LIKELIHOOD &&
          zchunks * kZPartials <= sw->ldm) {
        k_z_update_chunked<<<dim3(zchunks, B), kZcThreads, 0, st>>>(*sw, G, first, sw->stats, peers);
        TRB_CHECK_LAUNCH();
        return TRB_OK;
      }
      cudaError_t le = trb_launch_cluster(k_z_update, trb_cluster_size(B, sw->M), B, kUpThreads, st,
                                          *sw, G, first, light, sw->stats, peers);
      if (le != cudaSuccess)
        return trb_set_error(TRB_ERR_CUDA, "k_z_update: %s", cudaGetErrorString(le));
      TRB_CHECK_LAUNCH();
      return TRB_OK;
    }
    case TRB_STAGE_TX_RECUR: {
      TRB_CHECK_ARG(sw->ty && sw->lik.kind == TRB_GAUSSIAN_LIKELIHOOD,
                    "the tx recurrence needs ty and a Gaussian likelihood");
      trb_launch_scope scope_(0, st);
      k_tx_recur<<<dim3((sw->R + 255) / 256, B), 256, 0, st>>>(*sw);
      TRB_CHECK_LAUNCH();
      return TRB_OK;
    }
    case TRB_STAGE_PROJECT_Y: {  // ty = U_R^T y
      TRB_CHECK_ARG(sw->ty, "null ty");
      if (gemm)
        return trb_lin_project_gemm(sw->Ut, sw->R, sw->M, sw->ldm, B, sw->y, sw->ldm, sw->ty,
                                    stream);
      return trb_lin_project(sw->Ut, sw->strideU, sw->R, sw->M, sw->ldm, B, sw->y, sw->ldm, sw->ty,
                             nullptr, sw->gemv_impl, stream);
    }
    case TRB_STAGE_PROJECT_X:  // P3: tx = U_R^T b6 (new)
      if (gemm)
        return trb_lin_project_gemm(sw->Ut, sw->R, sw->M, sw->ldm, B, sw->b5, sw->ldm, sw->tx,
                                    stream);
      return trb_lin_project(sw->Ut, sw->strideU, sw->R, sw->M, sw->ldm, B, sw->b5, sw->ldm,
                             sw->tx, sw->active, sw->gemv_impl, stream);
case TRB_STAGE_EXPAND_Z:  // P4: rz = [b2/a2 +] V_R coef
      if (gemm)
        return trb_lin_expand_gemm(sw->Vt, sw->R, sw->N, sw->ldn, B, sw->coef, sw->part,
                                   sw->nslots * sw->ldn, stream);
      rc = trb_lin_expand(sw->Vt, sw->strideV, sw->R, sw->N, sw->ldn, B, sw->coef, sw->part,
                          sw->active, sw->gemv_impl, stream);
      if (rc) return rc;
      if (comm) return exchange_expansion(sw, sw->N, sw->ldn, st);
      if (!reduce_first) return rc;
      return trb_reduce_slots_inplace(B, sw->R, sw->N, sw->ldn, sw->part, stream);
    case TRB_STAGE_X_UPDATE: {  // X: e7, posterior x, records, early stopping
      trb_launch_scope scope_(0, st);
      trb_peers peers = {};
      if (comm) peers = *trb_comm_last(comm);
      const int xchunks = (sw->N + kChunk - 1) / kChunk;
      if ((update_kernels() & 1) && xchunks * kXPartials <= sw->ldn) {
        k_x_update_chunked<<<dim3(xchunks, B), kXcThreads, 0, st>>>(*sw, G, it, sw->stats, peers);
        TRB_CHECK_LAUNCH();
        return TRB_OK;
      }
      cudaError_t le = trb_launch_cluster(k_x_update, trb_cluster_size(B, sw->N), B, kUpThreads, st,
                                          *sw, G, it, sw->stats, peers);
      if (le != cudaSuccess)
        return trb_set_error(TRB_ERR_CUDA, "k_x_update: %s", cudaGetErrorString(le));
      TRB_CHECK_LAUNCH();
      return TRB_OK;
    }
    case TRB_STAGE_SNAPSHOT: {
      if (!sw->snap_edge_a) return TRB_OK;
      trb_launch_scope scope_(0, st);
      const int big = sw->N > sw->M ? sw->N : sw->M;
      int chunks = (big + 511) / 512;  // plain copies: spread a large instance over many CTAs
      const int cap = (4 * trb_device_sm_count() + B - 1) / B;
      if (chunks > cap) chunks = cap < 1 ? 1 : cap;
      // it == -2: restore only (end of a trb_sweep_run whose update kernels kept the state)
      k_snapshot<<<dim3(chunks, B), 256, 0, st>>>(*sw, it == -2 ? 1 : 0);
      k_snapshot_mark<<<(B + 255) / 256, 256, 0, st>>>(*sw);
      TRB_CHECK_LAUNCH();
      return TRB_OK;
    }
  }
  return trb_set_error(TRB_ERR_INVALID, "trb_sweep_stage: unknown stage %d", stage);
}

// ---- rescale inside the projection (P1+S1, P3+S2) --------------------------------------
// The rescale is 4 vectors of R per instance: as a kernel of its own it costs a launch and an idle
// GPU on both sides (~18 us at the north-star size, twice per iteration).  The projecting GEMV
// writes the coefficient of a row next to its projection and the variance from the spectrum
// (trb_linear.cu, RescaleFused): no launch, no wait on other CTAs.
static int g_fuse_rescale = -1;

extern "C" void trb_set_fused_rescale(int enabled) { g_fuse_rescale = enabled ? 1 : 0; }

static bool rescale_fusable(const trb_sweep* sw) {
  if (g_fuse_rescale < 0) {
    const char* e = getenv("TRB_FUSE_RESCALE");
    g_fuse_rescale = (e && e[0] == '0') ? 0 : 1;
  }
  if (!g_fuse_rescale || sw->comm || !sw->s || !sw->s2 || !sw->Vt || !sw->Ut) return false;
  const bool shared_ops = sw->strideV == 0 && sw->strideU == 0;
  if (shared_ops && (sw->gemv_impl == 3 || (sw->gemv_impl == 0 && sw->B >= 16))) return false;  // GEMM passes
  return sw->gemv_impl == 0 || sw->gemv_impl == 2;
}

// TRB_ERR_UNSUPPORTED: nothing was launched, the caller runs the two stages one by one
static int project_and_rescale(const trb_sweep* sw, int dir, cudaStream_t st) {
  const int B = sw->B;
  double* ea = sw->edge_a;
  const int R_total = sw->R_total > 0 ? sw->R_total : sw->R;
  const int null_space = R_total < sw->N;
  if (dir == 0)  // P1 + S1: tz = V_R^T b2, coef = s res (tz + s tx), forward variance
    return trb_lin_project_rescale(sw->Vt, sw->strideV, sw->R, sw->N, sw->ldn, B, sw->b1, sw->ldn, sw->tz,
                                   sw->active, 0, sw->N, sw->M, sw->rank, null_space, sw->s, sw->s2,
                                   sw->stride_s, ea + 1 * B, ea + 5 * B, sw->tx, sw->coef, sw->vlin,
                                   (sw->schedule == 0 && sw->snap_edge_a) ? sw->snap_tx : nullptr, (void*)st);
  // P3 + S2: tx = U_R^T b6 (new), coef for rz, backward variance
  return trb_lin_project_rescale(sw->Ut, sw->strideU, sw->R, sw->M, sw->ldm, B, sw->b5, sw->ldm, sw->tx,
                                 sw->active, 1, sw->N, sw->M, sw->rank, null_space, sw->s, sw->s2,
                                 sw->stride_s, ea + 1 * B, ea + 5 * B, sw->tz, sw->coef, sw->vlin, nullptr,
                                 (void*)st);
}

// One whole iteration, stage by stage (see the header comment of this file).
static int enqueue_iteration(const trb_sweep* sw, int it, int first, int fresh, bool light,
                             cudaStream_t st) {
  void* stream = (void*)st;
  const int schedule = sw->schedule;
  const bool fuse = rescale_fusable(sw);
  TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_PRIOR, it, first, 0, stream));
  if (first) {  // tx of the initial e6 (S1 needs it)
    if (fresh == 2) {  // e6 was initialised to b = 0: U_R^T 0 = 0, no pass over U needed
      cudaError_t e = cudaMemsetAsync(sw->tx, 0, sizeof(double) * (size_t)sw->B * sw->R, st);
      if (e != cudaSuccess)
        return trb_set_error(TRB_ERR_CUDA, "trb_sweep_run: %s", cudaGetErrorString(e));
    } else {
      TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_PROJECT_X_INIT, it, first, 0, stream));
    }
  }
  int fused = fuse ? project_and_rescale(sw, 0, st) : TRB_ERR_UNSUPPORTED;
  if (fused != TRB_OK && fused != TRB_ERR_UNSUPPORTED) return fused;
  if (fused != TRB_OK) {
    TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_PROJECT_Z, it, first, 0, stream));
    TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_RESCALE_FWD, it, first, 0, stream));
  }
  if (!light) TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_EXPAND_X, it, first, 0, stream));
  TRB_TRY(trb_sweep_stage(sw, light ? TRB_STAGE_Z_UPDATE_LIGHT : TRB_STAGE_Z_UPDATE, it, first, 0,
                          stream));
  fused = (fuse && schedule == 0) ? project_and_rescale(sw, 1, st) : TRB_ERR_UNSUPPORTED;
  if (fused != TRB_OK && fused != TRB_ERR_UNSUPPORTED) return fused;
  if (fused != TRB_OK) {
    TRB_TRY(trb_sweep_stage(sw, schedule ? TRB_STAGE_TX_RECUR : TRB_STAGE_PROJECT_X, it, first, 0,
                            stream));
    TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_RESCALE_BWD, it, first, 0, stream));
  }
  TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_EXPAND_Z, it, first, 0, stream));
  TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_X_UPDATE, it, first, 0, stream));
  // The update kernels copy every value they overwrite to the one-iteration-back state, so a
  // stopped instance is rolled back once, at the end of trb_sweep_run.  Schedule 2 skips the z
  // branch (b3, rz are not rewritten every iteration) and keeps the copy kernel.
  if (schedule == 2) TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_SNAPSHOT, it, first, 0, stream));
  return TRB_OK;
}

// ---- CUDA-graph replay of the identical middle iterations ----------------------
// An iteration of a small instance is a dozen ~2 us kernels: launch latency, not
// HBM, bounds it.  One iteration is captured (on a private stream: torch's
// default stream is the legacy stream, which cannot be captured) with the
// iteration index read from the device (k_x_update, it < 0) and replayed on the
// caller's stream.  The last captured graph is cached per host thread, keyed by
// the descriptor bytes.
constexpr int kGraphMinIters = 4;
constexpr double kGraphMaxBytes = 1e9;  // per iteration: beyond ~150 us of streaming, launches are hidden
bool trb_profile_events_enabled();
void trb_profile_add_launches(long long n0, long long n1);
long long trb_profile_launch_count(int kind);
static int g_graphs_enabled = -1;

static bool graph_eligible(const trb_sweep* sw) {
  if (g_graphs_enabled < 0) {
    const char* e = getenv("TRB_CUDA_GRAPHS");
    g_graphs_enabled = (e && e[0] == '0') ? 0 : 1;
  }
  if (!g_graphs_enabled || sw->comm || trb_profile_events_enabled()) return false;
  const bool shared = sw->strideV == 0 && sw->strideU == 0;
  const double bytes = 16.0 * sw->R * ((double)sw->N + sw->M) * (shared ? 1 : sw->B);
  return bytes <= kGraphMaxBytes;
}

struct GraphCache {
  trb_sweep key;
  int light = 0;
  int kernel_choice = -1;  // fused rescale / chunked updates at capture time
  cudaGraphExec_t exec = nullptr;
  long long launches[2] = {0, 0};
  cudaStream_t capture_stream = nullptr;
};
static thread_local GraphCache g_graph;

static int run_graph(const trb_sweep* sw, bool light, int count, cudaStream_t st) {
  GraphCache& gc = g_graph;
  const int kernel_choice = update_kernels() | (rescale_fusable(sw) ? 4 : 0);
  if (!gc.exec || gc.light != (int)light || gc.kernel_choice != kernel_choice ||
      memcmp(&gc.key, sw, sizeof(trb_sweep)) != 0) {
    if (gc.exec) {
      cudaGraphExecDestroy(gc.exec);
      gc.exec = nullptr;
    }
    if (!gc.capture_stream &&
        cudaStreamCreateWithFlags(&gc.capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
      cudaGetLastError();
      return TRB_ERR_UNSUPPORTED;
    }
    const long long n0 = trb_profile_launch_count(0), n1 = trb_profile_launch_count(1);
    if (cudaStreamBeginCapture(gc.capture_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
      cudaGetLastError();
      return TRB_ERR_UNSUPPORTED;
    }
    const int rc = enqueue_iteration(sw, -1, 0, 0, light, gc.capture_stream);
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(gc.capture_stream, &graph);
    gc.launches[0] = trb_profile_launch_count(0) - n0;
    gc.launches[1] = trb_profile_launch_count(1) - n1;
    trb_profile_add_launches(-gc.launches[0], -gc.launches[1]);  // captured, not launched
    if (rc != TRB_OK || ce != cudaSuccess || !graph) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      return rc != TRB_OK ? rc : TRB_ERR_UNSUPPORTED;
    }
    const cudaError_t ie = cudaGraphInstantiate(&gc.exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ie != cudaSuccess) {
      gc.exec = nullptr;
      cudaGetLastError();
      return TRB_ERR_UNSUPPORTED;
    }
    gc.key = *sw;
    gc.light = (int)light;
    gc.kernel_choice = kernel_choice;
  }
  for (int i = 0; i < count; ++i) {
    const cudaError_t le = cudaGraphLaunch(gc.exec, st);
    if (le != cudaSuccess)
      return trb_set_error(TRB_ERR_CUDA, "trb_sweep_run: graph launch: %s", cudaGetErrorString(le));
  }
  trb_profile_add_launches(gc.launches[0] * count, gc.launches[1] * count);
  return TRB_OK;
}

extern "C" void trb_set_cuda_graphs(int enabled) { g_graphs_enabled = enabled ? 1 : 0; }

int trb_sweep_run_persistent(const trb_sweep* sw, int it0, int n_iter, int fresh, cudaStream_t st);

extern "C" int trb_sweep_run(const trb_sweep* sw, int it0, int n_iter, int fresh, void* stream) {
  int rc = check_sweep(sw);
  if (rc) return rc;
  TRB_CHECK_ARG(it0 >= 0 && n_iter >= 0, "bad iteration range");
  TRB_CHECK_ARG(fresh >= 0 && fresh <= 2, "fresh must be 0, 1 or 2");
  const int schedule = sw->schedule;
  TRB_CHECK_ARG(schedule >= 0 && schedule <= 2, "schedule must be 0, 1 or 2");
  if (schedule) {
    TRB_CHECK_ARG(sw->lik.kind == TRB_GAUSSIAN_LIKELIHOOD, "schedules 1, 2 need a Gaussian likelihood");
    TRB_CHECK_ARG(sw->ty && !sw->b6_init, "schedules 1, 2 need ty and e6 initialised like e5");
    TRB_CHECK_ARG(schedule == 1 || (sw->damp3 == 0.0 && sw->es_tol < 0),
                  "schedule 2 needs damp3 = 0 and no early stopping");
  }
  cudaStream_t st = (cudaStream_t)stream;
  // one launch-bound instance: all iterations inside one cooperative launch (trb_persist.cu)
  {
    const int rc_p = trb_sweep_run_persistent(sw, it0, n_iter, fresh, st);
    if (rc_p != TRB_ERR_UNSUPPORTED) return rc_p;
  }
  if (n_iter > 0) {  // arrival counters of the chunked updates: stats[:, 2:4]
    const cudaError_t e = cudaMemset2DAsync(reinterpret_cast<char*>(sw->stats) + 16, 32, 0, 16, sw->B, st);
    if (e != cudaSuccess) return trb_set_error(TRB_ERR_CUDA, "trb_sweep_run: %s", cudaGetErrorString(e));
  }
  int k = 0;
  while (k < n_iter) {
    const int first = (fresh && k == 0) ? 1 : 0;
    const bool light = schedule == 2 && k + 1 < n_iter;  // z branch deferred to the last iteration
    // launch-bound sweeps (small instances): the identical middle iterations are
    // captured once into a CUDA graph and replayed
    if (!first) {
      int last = n_iter;                 // iterations [k, last) are identical
      if (schedule == 2) last = light ? n_iter - 1 : k;
      const int count = last - k;
      if (count >= kGraphMinIters && graph_eligible(sw)) {
        int rc_g = run_graph(sw, light, count, st);
        if (rc_g == TRB_OK) {
          k += count;
          continue;
        }
        if (rc_g != TRB_ERR_UNSUPPORTED) return rc_g;  // else: fall through to plain launches
      }
    }
    TRB_TRY(enqueue_iteration(sw, it0 + k, first, fresh, light, st));
    ++k;
  }
  // roll back the instances that stopped on NaN / divergence in this call (restore only)
  if (schedule != 2 && n_iter > 0) TRB_TRY(trb_sweep_stage(sw, TRB_STAGE_SNAPSHOT, -2, 0, 0, stream));
  return TRB_OK;
}
