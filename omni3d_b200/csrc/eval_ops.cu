// eval_ops.cu — Omni3D AP evaluation on the device: per-(image, category) greedy matching (Omni3Deval.evaluateImg) and
// the precision / recall / score tables (Omni3Deval.accumulate), cubercnn/evaluation/omni3d_evaluation.py:1172-1313,
// 1433-1551.  Compiled with -fmad=false: the 2D IoU (pycocotools bbIou) and the precision ratios must round exactly as
// the host's fp64 arithmetic does, so no a*b+c may be contracted.
#include <math.h>
#include <stdint.h>

#include "c3d_common.cuh"

namespace {

constexpr int kMaxA = 8, kMaxT = 16;
constexpr int kMatchWarps = 4;        // groups per 128-thread block
constexpr int kAccThreads = 64;       // (threshold, maxDet) curves of one (category, range) per block

struct MatchParams {
  double iou_start[kMaxT];            // min(iouThrs[t], 1 - 1e-10), computed on the host
  double lo[kMaxA], hi[kMaxA];        // inclusive range bounds
  double prox_thresh;
  int32_t A, T, mode3d, eval_prox;
};

// pycocotools maskApi.c bbIou for one (dt, gt) pair with iscrowd = 0: same branches, same operation order
__device__ __forceinline__ double bb_iou(const double* D, const double* G) {
  const double ga = G[2] * G[3], da = D[2] * D[3];
  const double w = fmin(D[2] + D[0], G[2] + G[0]) - fmax(D[0], G[0]);
  if (w <= 0) return 0.0;
  const double h = fmin(D[3] + D[1], G[3] + G[1]) - fmax(D[1], G[1]);
  if (h <= 0) return 0.0;
  const double i = w * h;
  const double u = da + ga - i;
  return i / u;
}

__device__ __forceinline__ bool outside(double v, double lo, double hi) { return v < lo || v > hi; }

// One warp per (image, category) group; lane l runs the greedy chains c = l, l + 32, ... of the A x T (range,
// threshold) pairs.  A range only changes which GTs are ignored, so a chain walks the group's regular GTs in annotation
// order and then its ignored ones: the reference's stable "ignored last" permutation without building it.
__global__ void __launch_bounds__(kMatchWarps * 32) eval_match_kernel(
    MatchParams P, int32_t G, const int32_t* __restrict__ dt_off, const int32_t* __restrict__ gt_off,
    const double* __restrict__ dt_box, const double* __restrict__ dt_rng, const double* __restrict__ gt_box,
    const double* __restrict__ gt_rng, const uint8_t* __restrict__ gt_ignore, const int64_t* __restrict__ gt_id,
    const float* __restrict__ iou3d, const int64_t* __restrict__ pair_off, int64_t NL, int64_t NG,
    int32_t* __restrict__ match, uint8_t* __restrict__ flags, int32_t* __restrict__ npig, uint8_t* __restrict__ gtm) {
  const int lane = threadIdx.x & 31;
  const int64_t g = (int64_t)blockIdx.x * kMatchWarps + (threadIdx.x >> 5);
  if (g >= G) return;
  const int32_t d0 = dt_off[g], nd = dt_off[g + 1] - d0;
  const int32_t g0 = gt_off[g], ng = gt_off[g + 1] - g0;
  const int A = P.A, T = P.T;
  if (lane < A) {
    int32_t n = 0;
    for (int j = 0; j < ng; ++j)
      n += !(gt_ignore[g0 + j] || outside(gt_rng[g0 + j], P.lo[lane], P.hi[lane]));
    npig[g * A + lane] = n;
  }
  if (nd == 0) return;
  const int64_t p0 = P.mode3d ? pair_off[g] : 0;
  const bool prox = P.eval_prox && ng > 0;
  for (int c = lane; c < A * T; c += 32) {
    const int a = c / T, t = c % T;
    const double lo = P.lo[a], hi = P.hi[a];
    uint8_t* used = gtm + (int64_t)c * NG + g0;
    for (int j = 0; j < ng; ++j) used[j] = 0;
    for (int d = 0; d < nd; ++d) {
      const double* D = dt_box + (int64_t)(d0 + d) * 4;
      double cur = P.iou_start[t];
      int m = -1, mig = 0;
      for (int pass = 0; pass < 2; ++pass) {
        // "if dt matched to reg gt, and on ignore gt, stop": no ignored GT is looked at once a regular one matched
        if (pass == 1 && m >= 0) break;
        for (int j = 0; j < ng; ++j) {
          const int ig = gt_ignore[g0 + j] || outside(gt_rng[g0 + j], lo, hi);
          if (ig != pass) continue;
          if (prox && !(bb_iou(D, gt_box + (int64_t)(g0 + j) * 4) > P.prox_thresh)) continue;
          if (used[j]) continue;
          const double v = P.mode3d ? (double)iou3d[p0 + (int64_t)d * ng + j] : bb_iou(D, gt_box + (int64_t)(g0 + j) * 4);
          if (v < cur) continue;       // the loop's own comparison: NaN and ties behave as in the reference
          cur = v;
          m = j;
          mig = pass;
        }
      }
      bool near = false;               // in proximity of any GT of the group, matched or not
      for (int j = 0; prox && j < ng && !near; ++j) near = bb_iou(D, gt_box + (int64_t)(g0 + j) * 4) > P.prox_thresh;
      int ig = 0, nz = 0;
      if (m >= 0) {
        used[m] = 1;
        ig = mig;
        nz = gt_id[g0 + m] != 0;       // dtMatches holds the GT id: a match to id 0 reads as unmatched
      }
      if (!nz && outside(dt_rng[d0 + d], lo, hi)) ig = 1;
      if (prox && !near) ig = 1;
      const int64_t o = (int64_t)c * NL + d0 + d;
      match[o] = m >= 0 ? g0 + m : -1;
      flags[o] = (uint8_t)(ig | (nz << 1));
    }
  }
}

// smallest integer c in [0, n] with c / n >= r in fp64 (the reference's searchsorted(tp / npig, r, 'left') target)
__device__ __forceinline__ int32_t recall_count(double r, int32_t n) {
  int32_t c = (int32_t)ceil(r * (double)n);
  if (c < 0) c = 0;
  if (c > n) c = n;
  while (c > 0 && (double)(c - 1) / (double)n >= r) --c;
  while (c < n && (double)c / (double)n < r) ++c;
  return c;
}

// One block per (category, range); thread (t, m) owns one precision-recall curve over the category's detections in
// score order, keeping those of per-group rank < maxDets[m].  Pass 1 counts; pass 2 walks backwards carrying the suffix
// maximum of tp / (tp + fp + eps) (the reference's envelope) and, at the detection where tp first reaches c, writes
// every recall threshold whose target count is c.
__global__ void __launch_bounds__(kAccThreads) eval_accumulate_kernel(
    int32_t K, int32_t A, int32_t T, int32_t M, int32_t R, const int32_t* __restrict__ grp_off,
    const int32_t* __restrict__ npig, const int32_t* __restrict__ ent_off, const int32_t* __restrict__ ent_idx,
    const int32_t* __restrict__ ent_rank, const double* __restrict__ ent_score, const uint8_t* __restrict__ flags,
    int64_t NL, const double* __restrict__ rec_thrs, const int32_t* __restrict__ max_dets, double* __restrict__ precision,
    double* __restrict__ recall, double* __restrict__ scores) {
  const int k = blockIdx.x, a = blockIdx.y;
  __shared__ int32_t s_npig[kAccThreads];
  int32_t n = 0;
  for (int32_t g = grp_off[k] + threadIdx.x; g < grp_off[k + 1]; g += blockDim.x) n += npig[(int64_t)g * A + a];
  s_npig[threadIdx.x] = n;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < blockDim.x; ++i) n += s_npig[i];
    s_npig[0] = n;
  }
  __syncthreads();
  const int32_t np = s_npig[0];
  const int c = threadIdx.x;
  if (c >= T * M) return;
  const int t = c / M, m = c % M;
  const int64_t KAM = (int64_t)K * A * M, col = (int64_t)k * A * M + (int64_t)a * M + m;
  double* prec = precision + (int64_t)t * R * KAM + col;
  double* sc = scores + (int64_t)t * R * KAM + col;
  if (np == 0) {
    for (int r = 0; r < R; ++r) prec[r * KAM] = -1.0, sc[r * KAM] = -1.0;
    recall[t * KAM + col] = -1.0;
    return;
  }
  const int32_t e0 = ent_off[k], e1 = ent_off[k + 1], md = max_dets[m];
  const uint8_t* f = flags + (int64_t)(a * T + t) * NL;
  int32_t nd = 0, tp = 0, fp = 0;
  for (int32_t e = e0; e < e1; ++e) {
    if (ent_rank[e] >= md) continue;
    ++nd;
    const uint8_t v = f[ent_idx[e]];
    if (!(v & 1)) (v & 2) ? ++tp : ++fp;
  }
  recall[t * KAM + col] = nd ? (double)tp / (double)np : 0.0;
  int r = R - 1;
  // thresholds past the last detection: the reference's try/except leaves them 0
  while (r >= 0 && (nd == 0 || recall_count(rec_thrs[r], np) > tp)) prec[r * KAM] = 0.0, sc[r * KAM] = 0.0, --r;
  if (r < 0) return;
  const double eps = 2.220446049250313e-16;   // np.spacing(1)
  double smax = 0.0, first_score = 0.0;
  bool any = false;
  for (int32_t e = e1 - 1; e >= e0; --e) {
    if (ent_rank[e] >= md) continue;
    const uint8_t v = f[ent_idx[e]];
    const double pr = (double)tp / ((double)fp + (double)tp + eps);
    if (!any || pr > smax) smax = pr;
    any = true;
    first_score = ent_score[e];
    if (!(v & 1)) {
      if (v & 2) {
        while (r >= 0 && recall_count(rec_thrs[r], np) == tp) prec[r * KAM] = smax, sc[r * KAM] = ent_score[e], --r;
        --tp;
      } else {
        --fp;
      }
    }
  }
  for (; r >= 0; --r) prec[r * KAM] = smax, sc[r * KAM] = first_score;   // target 0: the first detection
}

}  // namespace

extern "C" size_t c3d_eval_match_workspace_bytes(int64_t n_gt, int32_t A, int32_t T) {
  if (n_gt < 0 || A < 1 || T < 1) return 0;
  return (size_t)n_gt * A * T;
}

extern "C" int32_t c3d_eval_match(int32_t mode3d, int32_t eval_prox, int32_t num_groups, int32_t A, int32_t T,
                                  const int32_t* dt_off, const int32_t* gt_off, const double* dt_box, const double* dt_rng,
                                  const double* gt_box, const double* gt_rng, const uint8_t* gt_ignore,
                                  const int64_t* gt_id, const float* iou3d, const int64_t* pair_off, int64_t n_dt,
                                  int64_t n_gt, const double* iou_start_host, const double* ranges_host,
                                  double prox_thresh, int32_t* match, uint8_t* flags, int32_t* npig, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  using c3d::set_error;
  if (num_groups < 0 || n_dt < 0 || n_gt < 0) return set_error(C3D_EINVAL, "eval_match: negative sizes");
  if (A < 1 || A > kMaxA || T < 1 || T > kMaxT) return set_error(C3D_EINVAL, "eval_match: need 1 <= A <= %d, 1 <= T <= %d", kMaxA, kMaxT);
  if (n_dt > INT32_MAX || n_gt > INT32_MAX) return set_error(C3D_EINVAL, "eval_match: more than 2^31 boxes");
  if (!iou_start_host || !ranges_host) return set_error(C3D_EINVAL, "eval_match: null threshold / range array");
  if (num_groups == 0) return C3D_OK;
  if (!dt_off || !gt_off || !dt_box || !dt_rng || !gt_box || !gt_rng || !gt_ignore || !gt_id || !match || !flags || !npig)
    return set_error(C3D_EINVAL, "eval_match: null pointer");
  if (mode3d && (!iou3d || !pair_off)) return set_error(C3D_EINVAL, "eval_match: 3D mode needs iou3d and pair_off");
  if (workspace_bytes < c3d_eval_match_workspace_bytes(n_gt, A, T) || (n_gt > 0 && !workspace))
    return set_error(C3D_EWORKSPACE, "eval_match: workspace %zu < required %zu", workspace_bytes,
                     c3d_eval_match_workspace_bytes(n_gt, A, T));
  MatchParams P{};
  for (int t = 0; t < T; ++t) P.iou_start[t] = iou_start_host[t];
  for (int a = 0; a < A; ++a) P.lo[a] = ranges_host[2 * a], P.hi[a] = ranges_host[2 * a + 1];
  P.prox_thresh = prox_thresh;
  P.A = A, P.T = T, P.mode3d = mode3d != 0, P.eval_prox = eval_prox != 0;
  const int blocks = (num_groups + kMatchWarps - 1) / kMatchWarps;
  eval_match_kernel<<<blocks, kMatchWarps * 32, 0, static_cast<cudaStream_t>(stream)>>>(
      P, num_groups, dt_off, gt_off, dt_box, dt_rng, gt_box, gt_rng, gt_ignore, gt_id, iou3d, pair_off, n_dt, n_gt, match,
      flags, npig, static_cast<uint8_t*>(workspace));
  return c3d::check_launch("eval_match");
}

extern "C" int32_t c3d_eval_accumulate(int32_t K, int32_t A, int32_t T, int32_t M, int32_t R, const int32_t* grp_off,
                                       const int32_t* npig, const int32_t* ent_off, const int32_t* ent_idx,
                                       const int32_t* ent_rank, const double* ent_score, const uint8_t* flags, int64_t n_dt,
                                       const double* rec_thrs, const int32_t* max_dets, double* precision,
                                       double* recall, double* scores, void* stream) {
  using c3d::set_error;
  if (K < 0 || A < 1 || T < 1 || M < 1 || R < 1 || n_dt < 0) return set_error(C3D_EINVAL, "eval_accumulate: bad sizes");
  if (A > 65535 || T * M > kAccThreads) return set_error(C3D_EINVAL, "eval_accumulate: need A <= 65535, T * M <= %d", kAccThreads);
  if (K == 0) return C3D_OK;
  if (!grp_off || !npig || !ent_off || !rec_thrs || !max_dets || !precision || !recall || !scores)
    return set_error(C3D_EINVAL, "eval_accumulate: null pointer");
  if (n_dt > 0 && (!ent_idx || !ent_rank || !ent_score || !flags)) return set_error(C3D_EINVAL, "eval_accumulate: null pointer");
  eval_accumulate_kernel<<<dim3(K, A), kAccThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      K, A, T, M, R, grp_off, npig, ent_off, ent_idx, ent_rank, ent_score, flags, n_dt, rec_thrs, max_dets, precision,
      recall, scores);
  return c3d::check_launch("eval_accumulate");
}
