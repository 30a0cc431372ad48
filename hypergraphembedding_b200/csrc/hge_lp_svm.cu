// Personalized link-prediction classifiers (evaluation_util._personalized_classifier_prediction) on
// sm_100a: one RBF C-SVC per owner named by an asked link, trained on the owner's members (+1)
// against min(non-members, 2 x members) non-members drawn from the owner's Philox stream (-1), then
// one decision value per link.  oracle/lp_svm_ref.py restates the training sets and the solver.
//
//   grouping   links stably sorted by owner, the named owners numbered (PairGroups, hge_expand.cuh)
//   negatives  one warp per owner: Floyd's selection over the positions 0 .. n_o - 1 of the owner's
//              ascending non-member list (position -> id is a binary search over the sorted member
//              row, so no per-item flags), then the positions ranked into ascending order
//   solve      libsvm's dual C-SVC (Solver::Solve without shrinking): WSS3 working-set selection,
//              the two-variable update with clipping, stop at max_up -yG + max_low yG < tol, rho as
//              calculate_rho.  Kernel entries fp32 (||x - z||^2 a sequential fp32 sum over the d
//              components, each operation rounded on its own), gradient and alpha fp64 without
//              contraction; ties in the selections go to the largest index (libsvm's >= / <= scans).
//              Owners of at most 32 points: a warp each, one point per lane, the kernel matrix in
//              shared memory.  Larger owners: a CTA each, the points gathered (transposed) into a
//              workspace and the two kernel columns of each iteration computed on the fly.  Both
//              paths evaluate every quantity with the same functions, so the path taken changes no
//              bit; every selection is an exact arg-max, so no reduction order shows in the result.
//   predict    one warp per link: sum of alpha_i y_i K(x_i, x_item) over its owner's points (fixed
//              lane striding and shuffle tree) minus rho; the link is kept when that is > 0.
//
// A degenerate owner trains nothing and has no points: rho = +inf without members (every link
// rejected), -inf when every item is a member (every link kept).
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <chrono>
#include <math.h>
#include <vector>

#include "hge_common.cuh"
#include "hge_expand.cuh"
#include "hge_incidence.cuh"
#include "hge_philox.cuh"

namespace {

constexpr int kBlock = 256;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kWarpPoints = 32;          // warp path: owners of at most this many points
constexpr int kWarpsPerBlock = 8;
constexpr int kSolveBlock = 256;         // CTA path
constexpr double kTau = 1e-12;           // libsvm's TAU
constexpr int64_t kDefaultWorkspaceMb = 2048;
// CTA-path workspace per training point: gradient and alpha (16), the two kernel columns (8), plus
// 4 * d for the gathered point
constexpr int64_t kBytesPerPoint = 24;

struct SvmParams {
  float gamma;
  double C, tol;
};

// K(a, b) = exp(-gamma ||a - b||^2) in fp32; component c of a is a[c * sa]
__device__ __forceinline__ float rbf(const float* __restrict__ a, int64_t sa, const float* __restrict__ b,
                                     int64_t sb, int d, float gamma) {
  float s = 0.f;
  for (int c = 0; c < d; ++c) {
    const float t = __fsub_rn(a[c * sa], b[c * sb]);
    s = __fadd_rn(s, __fmul_rn(t, t));
  }
  return expf(__fmul_rn(-gamma, s));
}

// Q_ij = y_i y_j K_ij as libsvm caches it (float)
__device__ __forceinline__ float qval(double yi, double yj, float k) { return (yi == yj) ? k : -k; }

__device__ __forceinline__ bool better(double v, int i, double bv, int bi, bool largest) {
  return (largest ? v > bv : v < bv) || (v == bv && i > bi);
}

__device__ __forceinline__ void warp_best(double& v, int& i, bool largest) {
  for (int o = 16; o; o >>= 1) {
    const double ov = __shfl_xor_sync(kFull, v, o);
    const int oi = __shfl_xor_sync(kFull, i, o);
    if (better(ov, oi, v, i, largest)) {
      v = ov;
      i = oi;
    }
  }
}

// best (value, index) of the block; every thread gets it.  sv / si: shared [32]
__device__ void block_best(double& v, int& i, bool largest, double* sv, int* si) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  warp_best(v, i, largest);
  __syncthreads();
  if (lane == 0) {
    sv[w] = v;
    si[w] = i;
  }
  __syncthreads();
  v = lane < nw ? sv[lane] : (largest ? -INFINITY : INFINITY);
  i = lane < nw ? si[lane] : -1;
  warp_best(v, i, largest);
}

// -y G when t is in I_up (a candidate for the first index of the working set), else -inf
__device__ __forceinline__ double up_value(double y, double G, double A, double C) {
  const bool up = y > 0 ? A < C : A > 0;
  return up ? -(y * G) : -INFINITY;
}

// I_low member t: Gmax2 candidate y G and WSS3's objective decrease for (i, t)
__device__ __forceinline__ void low_values(double y, double G, double A, double C, double Gmax, float Qit,
                                           double yi, double& g2, double& obj) {
  g2 = -INFINITY;
  obj = INFINITY;
  const bool low = y > 0 ? A > 0 : A < C;
  if (!low) return;
  g2 = y * G;
  const double grad_diff = __dadd_rn(Gmax, y * G);
  if (grad_diff > 0) {
    // QD[i] + QD[j] - 2 y_i Q_i[j] (y_j = +1), + 2 y_i Q_i[j] (y_j = -1); QD = K(x, x) = 1
    double quad = __dsub_rn(2.0, y * __dmul_rn(2.0 * yi, (double)Qit));
    if (!(quad > 0)) quad = kTau;
    obj = -__ddiv_rn(__dmul_rn(grad_diff, grad_diff), quad);
  }
}

// libsvm's two-variable update with clipping (C_i = C_j = C): new alpha_i, alpha_j
__device__ __forceinline__ void smo_step(double yi, double yj, double Gi, double Gj, double Ai, double Aj,
                                         float Qij, double C, double& ai, double& aj) {
  ai = Ai;
  aj = Aj;
  if (yi != yj) {
    double quad = __dadd_rn(2.0, (double)__fmul_rn(2.f, Qij));
    if (quad <= 0) quad = kTau;
    const double delta = __ddiv_rn(__dsub_rn(-Gi, Gj), quad);
    const double diff = __dsub_rn(ai, aj);
    ai = __dadd_rn(ai, delta);
    aj = __dadd_rn(aj, delta);
    if (diff > 0) {
      if (aj < 0) {
        aj = 0;
        ai = diff;
      }
    } else {
      if (ai < 0) {
        ai = 0;
        aj = -diff;
      }
    }
    if (diff > 0) {   // diff > C_i - C_j
      if (ai > C) {
        ai = C;
        aj = __dsub_rn(C, diff);
      }
    } else {
      if (aj > C) {
        aj = C;
        ai = __dadd_rn(C, diff);
      }
    }
  } else {
    double quad = __dsub_rn(2.0, (double)__fmul_rn(2.f, Qij));
    if (quad <= 0) quad = kTau;
    const double delta = __ddiv_rn(__dsub_rn(Gi, Gj), quad);
    const double sum = __dadd_rn(ai, aj);
    ai = __dsub_rn(ai, delta);
    aj = __dadd_rn(aj, delta);
    if (sum > C) {
      if (ai > C) {
        ai = C;
        aj = __dsub_rn(sum, C);
      }
    } else {
      if (aj < 0) {
        aj = 0;
        ai = sum;
      }
    }
    if (sum > C) {
      if (aj > C) {
        aj = C;
        ai = __dsub_rn(sum, C);
      }
    } else {
      if (ai < 0) {
        ai = 0;
        aj = sum;
      }
    }
  }
}

__device__ __forceinline__ double grad_update(double G, float Qi, float Qj, double dai, double daj) {
  return __dadd_rn(G, __dadd_rn(__dmul_rn((double)Qi, dai), __dmul_rn((double)Qj, daj)));
}

// calculate_rho, fed the points in index order
struct RhoAcc {
  int64_t nfree = 0;
  double ub = INFINITY, lb = -INFINITY, sum = 0;
  __device__ void add(double y, double G, double A, double C) {
    const double yG = y * G;
    if (A >= C) {
      if (y < 0) ub = fmin(ub, yG); else lb = fmax(lb, yG);
    } else if (A <= 0) {
      if (y > 0) ub = fmin(ub, yG); else lb = fmax(lb, yG);
    } else {
      ++nfree;
      sum = __dadd_rn(sum, yG);
    }
  }
  __device__ double value() const {
    return nfree > 0 ? __ddiv_rn(sum, (double)nfree) : __ddiv_rn(__dadd_rn(ub, lb), 2.0);
  }
};

__device__ __forceinline__ int64_t max_iter(int64_t n) { return n > 100000 ? 100 * n : 10000000; }

// ---- grouping / training sets -------------------------------------------------------------------

// per named owner: members m, points n (0 for a degenerate owner, whose rho is set here)
__global__ void k_owner_sizes(int64_t U, const int32_t* __restrict__ ug, const int64_t* __restrict__ mptr,
                              int64_t items, int32_t* __restrict__ msize, int64_t* __restrict__ npts,
                              double* __restrict__ rho, int64_t* __restrict__ iters) {
  for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u <= U; u += (int64_t)gridDim.x * blockDim.x) {
    if (u == U) {
      npts[U] = 0;
      continue;
    }
    const int32_t o = ug[u];
    const int64_t m = mptr[o + 1] - mptr[o], others = items - m;
    const bool degenerate = m == 0 || others == 0;
    msize[u] = (int32_t)m;
    npts[u] = degenerate ? 0 : m + (others < 2 * m ? others : 2 * m);
    iters[u] = 0;
    if (degenerate) rho[u] = m == 0 ? INFINITY : -INFINITY;
  }
}

// training points of every named owner u at pid[poff[u] ..]: its members, then its negatives, both
// ascending.  One warp per owner; every lane draws the same words of the owner's stream.
__global__ void __launch_bounds__(kBlock) k_training_sets(
    int64_t U, const int32_t* __restrict__ ug, const int64_t* __restrict__ mptr, const int32_t* __restrict__ midx,
    int64_t items, const int64_t* __restrict__ poff, uint64_t seed, uint32_t phase, int32_t* __restrict__ pid,
    int32_t* __restrict__ scratch) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t u = blockIdx.x * (int64_t)(kBlock / 32) + (threadIdx.x >> 5); u < U; u += nw) {
    const int64_t base = poff[u], n = poff[u + 1] - base;
    if (n == 0) continue;
    const int32_t o = ug[u];
    const int32_t* mem = midx + mptr[o];
    const int64_t m = mptr[o + 1] - mptr[o], others = items - m, k = n - m;
    for (int64_t t = lane; t < m; t += 32) pid[base + t] = mem[t];
    int32_t* neg = pid + base + m;
    if (k == others) {   // every non-member, nothing drawn
      for (int64_t p = lane; p < k; p += 32) neg[p] = hge_nonmember(mem, m, p);
      continue;
    }
    int32_t* pos = scratch + base + m;
    HgeStreamRng rng(seed, phase, (uint64_t)o);
    for (int64_t s = 0; s < k; ++s) {
      const int64_t j = others - k + s;
      const int32_t t = (int32_t)rng.below((uint32_t)(j + 1));
      bool hit = false;
      for (int64_t q = lane; q < s; q += 32) hit |= pos[q] == t;
      hit = __any_sync(kFull, hit);
      if (lane == 0) pos[s] = hit ? (int32_t)j : t;
      __syncwarp();
    }
    for (int64_t q = lane; q < k; q += 32) {
      const int32_t v = pos[q];
      int64_t r = 0;
      for (int64_t x = 0; x < k; ++x) r += pos[x] < v;
      neg[r] = hge_nonmember(mem, m, v);
    }
    __syncwarp();
  }
}

// ---- solver: warp path --------------------------------------------------------------------------

__global__ void __launch_bounds__(kWarpsPerBlock * 32) k_smo_warp(
    int64_t count, const int32_t* __restrict__ list, const int64_t* __restrict__ poff,
    const int32_t* __restrict__ msize, const int32_t* __restrict__ pid, const float* __restrict__ vec, int d,
    SvmParams prm, double* __restrict__ coef, double* __restrict__ rho, int64_t* __restrict__ iters) {
  __shared__ float ks[kWarpsPerBlock][kWarpPoints][kWarpPoints + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const double C = prm.C;
  for (int64_t li = blockIdx.x * (int64_t)kWarpsPerBlock + w; li < count;
       li += (int64_t)gridDim.x * kWarpsPerBlock) {
    const int32_t u = list[li];
    const int64_t base = poff[u];
    const int n = (int)(poff[u + 1] - base), m = msize[u];
    const bool on = lane < n;
    const int32_t id = on ? pid[base + lane] : 0;
    const double y = lane < m ? 1.0 : -1.0;
    for (int s = 0; s < n; ++s) {
      const int32_t other = __shfl_sync(kFull, id, s);
      if (on) ks[w][lane][s] = rbf(vec + (int64_t)id * d, 1, vec + (int64_t)other * d, 1, d, prm.gamma);
    }
    __syncwarp();
    double G = -1.0, A = 0.0;
    int64_t it = 0;
    const int64_t cap = max_iter(n);
    while (it < cap) {
      double Gmax = on ? up_value(y, G, A, C) : -INFINITY;
      int i = Gmax > -INFINITY ? lane : -1;
      warp_best(Gmax, i, true);
      if (i < 0) break;
      const double yi = i < m ? 1.0 : -1.0;
      const float Qi = on ? qval(yi, y, ks[w][i][lane]) : 0.f;
      double g2 = -INFINITY, obj = INFINITY;
      if (on) low_values(y, G, A, C, Gmax, Qi, yi, g2, obj);
      int j = obj < INFINITY ? lane : -1;
      int dummy = 0;
      warp_best(obj, j, false);
      warp_best(g2, dummy, true);
      if (__dadd_rn(Gmax, g2) < prm.tol || j < 0) break;
      const double yj = j < m ? 1.0 : -1.0;
      const float Qj = on ? qval(yj, y, ks[w][j][lane]) : 0.f;
      const double Gi = __shfl_sync(kFull, G, i), Gj = __shfl_sync(kFull, G, j);
      const double Ai = __shfl_sync(kFull, A, i), Aj = __shfl_sync(kFull, A, j);
      const float Qij = __shfl_sync(kFull, Qi, j);
      double ai, aj;
      smo_step(yi, yj, Gi, Gj, Ai, Aj, Qij, C, ai, aj);
      const double dai = __dsub_rn(ai, Ai), daj = __dsub_rn(aj, Aj);
      if (on) G = grad_update(G, Qi, Qj, dai, daj);
      if (lane == i) A = ai;
      if (lane == j) A = aj;
      ++it;
    }
    RhoAcc acc;
    for (int s = 0; s < n; ++s) {
      const double Gs = __shfl_sync(kFull, G, s), As = __shfl_sync(kFull, A, s);
      acc.add(s < m ? 1.0 : -1.0, Gs, As, C);
    }
    if (on) coef[base + lane] = y * A;
    if (lane == 0) {
      rho[u] = acc.value();
      iters[u] = it;
    }
    __syncwarp();
  }
}

// ---- solver: CTA path ---------------------------------------------------------------------------

// one CTA per owner list[b]; its workspace starts at point woff[b] of the batch's arrays
__global__ void __launch_bounds__(kSolveBlock) k_smo_block(
    const int32_t* __restrict__ list, const int64_t* __restrict__ woff, const int64_t* __restrict__ poff,
    const int32_t* __restrict__ msize, const int32_t* __restrict__ pid, const float* __restrict__ vec, int d,
    SvmParams prm, float* __restrict__ wx, double* __restrict__ wg, double* __restrict__ wa,
    float* __restrict__ wqi, float* __restrict__ wqj, double* __restrict__ coef, double* __restrict__ rho,
    int64_t* __restrict__ iters) {
  __shared__ double sv[32];
  __shared__ int si[32];
  const int32_t u = list[blockIdx.x];
  const int64_t base = poff[u], off = woff[blockIdx.x];
  const int n = (int)(poff[u + 1] - base), m = msize[u];
  const double C = prm.C;
  float* X = wx + off * d;   // X[c * n + t]: component c of point t
  double* G = wg + off;
  double* A = wa + off;
  float* Qi = wqi + off;
  float* Qj = wqj + off;
  for (int64_t e = threadIdx.x; e < (int64_t)n * d; e += blockDim.x) {
    const int64_t t = e / d, c = e - t * d;
    X[c * n + t] = vec[(int64_t)pid[base + t] * d + c];
  }
  for (int t = threadIdx.x; t < n; t += blockDim.x) {
    G[t] = -1.0;
    A[t] = 0.0;
  }
  __syncthreads();
  int64_t it = 0;
  const int64_t cap = max_iter(n);
  while (it < cap) {
    double Gmax = -INFINITY;
    int i = -1;
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      const double v = up_value(t < m ? 1.0 : -1.0, G[t], A[t], C);
      if (v > -INFINITY && better(v, t, Gmax, i, true)) {
        Gmax = v;
        i = t;
      }
    }
    block_best(Gmax, i, true, sv, si);
    if (i < 0) break;
    const double yi = i < m ? 1.0 : -1.0;
    for (int t = threadIdx.x; t < n; t += blockDim.x)
      Qi[t] = qval(yi, t < m ? 1.0 : -1.0, rbf(X + i, n, X + t, n, d, prm.gamma));
    __syncthreads();
    double g2 = -INFINITY, obj = INFINITY;
    int j = -1, dummy = 0;
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      double tg2, tobj;
      low_values(t < m ? 1.0 : -1.0, G[t], A[t], C, Gmax, Qi[t], yi, tg2, tobj);
      g2 = fmax(g2, tg2);
      if (tobj < INFINITY && better(tobj, t, obj, j, false)) {
        obj = tobj;
        j = t;
      }
    }
    block_best(obj, j, false, sv, si);
    block_best(g2, dummy, true, sv, si);
    if (__dadd_rn(Gmax, g2) < prm.tol || j < 0) break;
    const double yj = j < m ? 1.0 : -1.0;
    for (int t = threadIdx.x; t < n; t += blockDim.x)
      Qj[t] = qval(yj, t < m ? 1.0 : -1.0, rbf(X + j, n, X + t, n, d, prm.gamma));
    const double Gi = G[i], Gj = G[j], Ai = A[i], Aj = A[j];
    const float Qij = Qi[j];
    __syncthreads();   // Qj complete; G / A read before they change
    double ai, aj;
    smo_step(yi, yj, Gi, Gj, Ai, Aj, Qij, C, ai, aj);
    const double dai = __dsub_rn(ai, Ai), daj = __dsub_rn(aj, Aj);
    for (int t = threadIdx.x; t < n; t += blockDim.x) G[t] = grad_update(G[t], Qi[t], Qj[t], dai, daj);
    if (threadIdx.x == 0) {
      A[i] = ai;
      A[j] = aj;
    }
    __syncthreads();
    ++it;
  }
  for (int t = threadIdx.x; t < n; t += blockDim.x) coef[base + t] = (t < m ? 1.0 : -1.0) * A[t];
  if (threadIdx.x == 0) {
    RhoAcc acc;
    for (int t = 0; t < n; ++t) acc.add(t < m ? 1.0 : -1.0, G[t], A[t], C);
    rho[u] = acc.value();
    iters[u] = it;
  }
}

// ---- prediction ---------------------------------------------------------------------------------

// one warp per sorted link i (link order[i], owner rank[i] - 1)
__global__ void __launch_bounds__(kBlock) k_predict(
    int64_t num_links, const int32_t* __restrict__ order, const int32_t* __restrict__ rank,
    const int32_t* __restrict__ items, const int64_t* __restrict__ poff, const int32_t* __restrict__ pid,
    const double* __restrict__ coef, const double* __restrict__ rho, const float* __restrict__ vec, int d,
    float gamma, uint8_t* __restrict__ keep, double* __restrict__ decision) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * (kBlock / 32);
  for (int64_t i = blockIdx.x * (int64_t)(kBlock / 32) + (threadIdx.x >> 5); i < num_links; i += nw) {
    const int32_t p = order[i];
    const int64_t u = rank[i] - 1, base = poff[u], n = poff[u + 1] - base;
    const float* x = vec + (int64_t)items[p] * d;
    double s = 0;
    for (int64_t t = lane; t < n; t += 32) {
      const double c = coef[base + t];
      if (c != 0) s = __dadd_rn(s, __dmul_rn(c, (double)rbf(vec + (int64_t)pid[base + t] * d, 1, x, 1, d, gamma)));
    }
    for (int o = 16; o; o >>= 1) s = __dadd_rn(s, __shfl_xor_sync(kFull, s, o));
    if (lane == 0) {
      const double f = __dsub_rn(s, rho[u]);
      keep[p] = f > 0 ? 1 : 0;
      if (decision) decision[p] = f;
    }
  }
}

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

}  // namespace

extern "C" {

int hge_lp_svm_predict(hge_ctx* ctx, hge_incidence* inc, int owner_side, const float* item_vectors, int d,
                       const int32_t* link_items, const int32_t* link_owners, int64_t num_links, uint64_t seed,
                       double C, double gamma, double tol, int64_t workspace_mb, uint8_t* out_keep,
                       double* out_decision, int64_t* out_counts, int32_t* owner_ids, double* owner_rho,
                       int64_t* owner_iters, int64_t* owner_offset, int32_t* point_ids, double* point_coef,
                       int64_t point_capacity, double* phase_ms) {
  HGE_REQUIRE(ctx && inc, "hge_lp_svm_predict: NULL argument");
  HGE_REQUIRE(!inc->sharded, "hge_lp_svm_predict: needs a whole (not sharded) incidence");
  HGE_REQUIRE(owner_side == 0 || owner_side == 1, "hge_lp_svm_predict: owner_side must be 0 (nodes) or 1 (edges)");
  HGE_REQUIRE(d >= 1, "hge_lp_svm_predict: d must be >= 1");
  HGE_REQUIRE(C > 0 && gamma > 0 && tol > 0, "hge_lp_svm_predict: C, gamma and tol must be positive");
  HGE_REQUIRE(num_links >= 0 && num_links < (1ll << 31) &&
                  (num_links == 0 || (item_vectors && link_items && link_owners && out_keep)),
              "hge_lp_svm_predict: bad links");
  HGE_REQUIRE(workspace_mb >= 0 && point_capacity >= 0, "hge_lp_svm_predict: negative size");
  HGE_CUDA(cudaSetDevice(ctx->device));
  if (out_counts) out_counts[0] = out_counts[1] = out_counts[2] = 0;
  if (num_links == 0) return HGE_OK;
  const double t0 = now_ms();
  auto mark = [&](int k, double& last) -> int {
    if (!phase_ms) return HGE_OK;
    HGE_CUDA(cudaStreamSynchronize(ctx->stream));
    const double t = now_ms();
    phase_ms[k] = t - last;
    last = t;
    return HGE_OK;
  };
  double last = t0;
  // owner = edge: members are its nodes, items the nodes; owner = node: its edges, items the edges
  const int64_t owners = owner_side == 1 ? inc->E : inc->N, items = owner_side == 1 ? inc->N : inc->E;
  const int64_t* mptr = owner_side == 1 ? inc->e2n_ptr : inc->n2e_ptr;
  const int32_t* midx = owner_side == 1 ? inc->e2n_idx : inc->n2e_idx;
  const uint32_t phase = owner_side == 1 ? HGE_PHASE_LP_EDGE_OWNERS : HGE_PHASE_LP_NODE_OWNERS;
  const int64_t L = num_links;

  // 1. links stably sorted by owner, the named owners, their training-set sizes
  PairGroups grp(ctx);
  int bad = 0;
  HGE_TRY(grp.build(ctx, L, link_items, items, link_owners, owners, &bad));
  HGE_REQUIRE(!(bad & kBadX), "hge_lp_svm_predict: a link names an item outside [0, %lld)", (long long)items);
  HGE_REQUIRE(!(bad & kBadGroup), "hge_lp_svm_predict: a link names an owner outside [0, %lld)", (long long)owners);
  const int64_t U = grp.U;
  DevBuf<int32_t> msize(ctx);
  DevBuf<int64_t> npts(ctx), poff(ctx), iters(ctx);
  DevBuf<double> rho(ctx);
  DevBuf<char> temp(ctx);
  HGE_TRY(msize.alloc((size_t)U));
  HGE_TRY(npts.alloc((size_t)U + 1));
  HGE_TRY(poff.alloc((size_t)U + 1));
  HGE_TRY(iters.alloc((size_t)U));
  HGE_TRY(rho.alloc((size_t)U));
  k_owner_sizes<<<grid_for(ctx, U + 1), kBlock, 0, ctx->stream>>>(U, grp.ug.p, mptr, items, msize.p, npts.p, rho.p,
                                                                 iters.p);
  HGE_CHECK_LAUNCH(ctx);
  size_t bytes = 0;
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, npts.p, poff.p, U + 1, ctx->stream));
  HGE_TRY(temp.alloc(bytes));
  HGE_CUDA(cub::DeviceScan::ExclusiveSum(temp.p, bytes, npts.p, poff.p, U + 1, ctx->stream));
  ctx->launches++;
  std::vector<int64_t> h_poff((size_t)U + 1);
  HGE_TRY(read_back(ctx, poff.p, h_poff.data(), (size_t)U + 1));
  const int64_t T = h_poff[(size_t)U];
  HGE_REQUIRE(!(point_ids || point_coef) || T <= point_capacity,
              "hge_lp_svm_predict: the model has %lld training points, more than point_capacity %lld",
              (long long)T, (long long)point_capacity);
  HGE_TRY(mark(0, last));

  // 2. training sets
  DevBuf<int32_t> pid(ctx), scratch(ctx);
  DevBuf<double> coef(ctx);
  HGE_TRY(pid.alloc((size_t)T));
  HGE_TRY(coef.alloc((size_t)T));
  HGE_TRY(scratch.alloc((size_t)T));
  k_training_sets<<<grid_for(ctx, U, kBlock / 32), kBlock, 0, ctx->stream>>>(U, grp.ug.p, mptr, midx, items, poff.p,
                                                                           seed, phase, pid.p, scratch.p);
  HGE_CHECK_LAUNCH(ctx);
  scratch.reset();
  HGE_TRY(mark(1, last));

  // 3. solve: small owners a warp each in one launch, larger ones a CTA each in batches whose
  //    workspace fits the budget (a single larger owner is its own batch)
  const SvmParams prm = {(float)gamma, C, tol};
  std::vector<int32_t> small, large;
  std::vector<int64_t> large_off;   // each large owner's first point in its batch's workspace
  std::vector<size_t> batch_end;    // end of each batch in `large`
  const int64_t mb = workspace_mb ? workspace_mb : kDefaultWorkspaceMb;
  const int64_t budget = mb << 20, per_point = kBytesPerPoint + 4 * (int64_t)d;
  int64_t used = 0, batch_points = 0;
  std::vector<int64_t> batch_pts;
  for (int64_t u = 0; u < U; ++u) {
    const int64_t n = h_poff[(size_t)u + 1] - h_poff[(size_t)u];
    if (n == 0) continue;
    if (n <= kWarpPoints) {
      small.push_back((int32_t)u);
      continue;
    }
    if (!large.empty() && used + n * per_point > budget) {
      batch_end.push_back(large.size());
      batch_pts.push_back(batch_points);
      used = batch_points = 0;
    }
    large.push_back((int32_t)u);
    large_off.push_back(batch_points);
    used += n * per_point;
    batch_points += n;
  }
  if (!large.empty()) {
    batch_end.push_back(large.size());
    batch_pts.push_back(batch_points);
  }
  DevBuf<int32_t> d_small(ctx), d_large(ctx);
  DevBuf<int64_t> d_off(ctx);
  if (!small.empty()) {
    HGE_TRY(d_small.alloc(small.size()));
    HGE_CUDA(cudaMemcpyAsync(d_small.p, small.data(), small.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                             ctx->stream));
    const int64_t cnt = (int64_t)small.size();
    k_smo_warp<<<grid_for(ctx, cnt, kWarpsPerBlock), kWarpsPerBlock * 32, 0, ctx->stream>>>(
        cnt, d_small.p, poff.p, msize.p, pid.p, item_vectors, d, prm, coef.p, rho.p, iters.p);
    HGE_CHECK_LAUNCH(ctx);
  }
  if (!large.empty()) {
    HGE_TRY(d_large.alloc(large.size()));
    HGE_TRY(d_off.alloc(large.size()));
    HGE_CUDA(cudaMemcpyAsync(d_large.p, large.data(), large.size() * sizeof(int32_t), cudaMemcpyHostToDevice,
                             ctx->stream));
    HGE_CUDA(cudaMemcpyAsync(d_off.p, large_off.data(), large_off.size() * sizeof(int64_t), cudaMemcpyHostToDevice,
                             ctx->stream));
    size_t b0 = 0;
    for (size_t b = 0; b < batch_end.size(); ++b) {
      const size_t b1 = batch_end[b];
      const int64_t P = batch_pts[b];
      DevBuf<float> wx(ctx), wqi(ctx), wqj(ctx);
      DevBuf<double> wg(ctx), wa(ctx);
      int rc = wx.alloc((size_t)P * d);
      if (rc == HGE_OK) rc = wg.alloc((size_t)P);
      if (rc == HGE_OK) rc = wa.alloc((size_t)P);
      if (rc == HGE_OK) rc = wqi.alloc((size_t)P);
      if (rc == HGE_OK) rc = wqj.alloc((size_t)P);
      if (rc == HGE_ERR_NOMEM)
        hge_set_error("hge_lp_svm_predict: %lld owners with %lld training points need %lld bytes of workspace, "
                      "more than the device holds", (long long)(b1 - b0), (long long)P, (long long)(P * per_point));
      HGE_TRY(rc);
      k_smo_block<<<(unsigned)(b1 - b0), kSolveBlock, 0, ctx->stream>>>(
          d_large.p + b0, d_off.p + b0, poff.p, msize.p, pid.p, item_vectors, d, prm, wx.p, wg.p, wa.p, wqi.p,
          wqj.p, coef.p, rho.p, iters.p);
      HGE_CHECK_LAUNCH(ctx);
      b0 = b1;
    }
  }
  std::vector<int64_t> h_iters((size_t)U);
  HGE_TRY(read_back(ctx, iters.p, h_iters.data(), (size_t)U));
  int64_t capped = 0;
  for (int64_t u = 0; u < U; ++u) {
    const int64_t n = h_poff[(size_t)u + 1] - h_poff[(size_t)u];
    if (n > 0 && h_iters[(size_t)u] >= std::max<int64_t>(10000000, 100 * n)) ++capped;
  }
  HGE_TRY(mark(2, last));

  // 4. one decision value per link
  k_predict<<<grid_for(ctx, L, kBlock / 32), kBlock, 0, ctx->stream>>>(
      L, grp.order, grp.rank.p, link_items, poff.p, pid.p, coef.p, rho.p, item_vectors, d, prm.gamma, out_keep,
      out_decision);
  HGE_CHECK_LAUNCH(ctx);
  if (owner_ids)
    HGE_CUDA(cudaMemcpyAsync(owner_ids, grp.ug.p, (size_t)U * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
  if (owner_rho)
    HGE_CUDA(cudaMemcpyAsync(owner_rho, rho.p, (size_t)U * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  if (owner_iters)
    HGE_CUDA(cudaMemcpyAsync(owner_iters, iters.p, (size_t)U * sizeof(int64_t), cudaMemcpyDeviceToDevice,
                             ctx->stream));
  if (owner_offset)
    HGE_CUDA(cudaMemcpyAsync(owner_offset, poff.p, ((size_t)U + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice,
                             ctx->stream));
  if (point_ids && T)
    HGE_CUDA(cudaMemcpyAsync(point_ids, pid.p, (size_t)T * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
  if (point_coef && T)
    HGE_CUDA(cudaMemcpyAsync(point_coef, coef.p, (size_t)T * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
  if (out_counts) {
    out_counts[0] = U;
    out_counts[1] = T;
    out_counts[2] = capped;
  }
  HGE_TRY(mark(3, last));
  return HGE_OK;
}

}  // extern "C"
