// Landmark-side kernels of the solver round (sm_100a):
//   k_linearize ("A1"): one thread per (landmark, frame).  Reprojection residuals + Jacobian factors of
//       the frame's cameras, Cauchy weighting, per-frame M_f = sum rho' A^T A and m_f = sum rho' A^T r
//       (stored tile-major, see lm_M_index), plus the pose-block contributions H_pp,f = G^T M_f G and
//       g_p,f = G^T m_f reduced per CTA.  All global loads are issued up front; CTAs whose landmarks
//       do not see the frame exit immediately (landmarks are sorted by observing-frame range).
//   k_lmblock ("A1b"): one thread per landmark: H_ll = sum_f M_f, (H_ll + mu E)^-1 by 3x3 Cholesky.
//   k_schur ("A2"): one CTA per (landmark chunk, window), tiles of 32 landmarks staged by TMA bulk copies:
//       Y_f = W_f L^-T into a tile-local shared-memory tile, then the Schur complement as a SYRK S += Y Y^T
//       over 8x8 blocks on the FP64 tensor cores (details at the kernel).
//   k_quality: post-solve landmark quality (Estimator.cpp:880-894), one thread per landmark.
#pragma once
#include "okb_estimator.cuh"

namespace okb {

constexpr int L1_THREADS = 128;          // k_linearize block = landmarks per CTA (x one frame)
constexpr int A2_THREADS = 256;          // k_schur block (8 warps, two CTAs per SM)
constexpr int A2_TILE = 32;              // landmarks per Y tile
constexpr int kPartH = 32;               // doubles per (cx, frame) record: 27 H_pp/g_p + cost + stepnorm2 + pad

struct SlotCtx {
  SlotXf xf;
  CamIntr cam;
  int frame;
  int valid;
};
static_assert(sizeof(SlotCtx) % 8 == 0, "SlotCtx is copied as doubles");

// (frame, camera) contexts at the candidate poses: computed once per round by the kernel that writes the
// candidate (k_reset / k_solve) instead of by every k_linearize CTA.
__device__ inline void build_slot_ctx(const WinDev& W, int tid, int nthr) {
  for (int s = tid; s < W.NS; s += nthr) {
    const SlotInfo si = W.slots[s];
    SlotCtx sc;
    sc.valid = si.valid; sc.frame = s / W.CP;
    if (si.valid) { make_slot_xf(W.pose_c + 7 * si.pose_idx, W.ext + 7 * si.ext_idx, sc.xf); cam_load(W.cams[si.cam_idx], sc.cam); }
    else { for (int k = 0; k < 9; ++k) sc.xf.R[k] = 0; for (int k = 0; k < 3; ++k) sc.xf.t[k] = 0; cam_load(W.cams[0], sc.cam); }
    W.slot_ctx[s] = sc;
  }
}

// ------------------------------------------------------------------------------------------------
// A1
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(L1_THREADS) k_linearize(const WinDev* __restrict__ wins, int win_first) {
  const WinDev& W = wins[win_first + blockIdx.z];
  const SolverState* st = W.st;
  if (st->done) return;
  const int f = blockIdx.y;
  const int cx = blockIdx.x;
  if (f >= W.K || cx * L1_THREADS >= W.L) return;
  const int tid = threadIdx.x;
  const int L = W.L, CP = W.CP;

  __shared__ SlotCtx slots[32];                 // the frame's cameras (CP <= 32)
  __shared__ double sred[kPartH][L1_THREADS + 1];
  __shared__ double s_tw[3];

  // Landmarks are sorted by observing-frame range: a CTA whose 4 tiles are not seen by frame f has nothing
  // to do except publishing zeros (frame 0 also carries the candidate landmark update).
  if (f != 0) {
    bool any = false;
#pragma unroll
    for (int t = 0; t < L1_THREADS / 32; ++t) {
      const int tile = cx * (L1_THREADS / 32) + t;
      if (tile * 32 < L) {
        const uint32_t tr = W.tile_range[tile];
        any = any || ((int)(tr & 0xffu) <= f && f <= (int)(tr >> 8));
      }
    }
    if (!any) {
      if (tid < 29) W.partH[((size_t)cx * W.K + f) * kPartH + tid] = 0.0;
      return;
    }
  }
  // All global loads of this thread are issued before anything waits on them (one memory round trip instead
  // of a chain visibility -> landmark -> observations): the visibility mask, the landmark, the observations of
  // the first two cameras and, in STEP mode, the stored step.  Speculative for unobserved pairs; with
  // sorted landmarks those are few inside a CTA that is not skipped.
  const int mode = st->mode, cur = st->cur;
  const bool cauchy = W.use_cauchy != 0;
  const int l = cx * L1_THREADS + tid;
  const int lc = min(l, L - 1);
  const uint32_t vmask = W.lm_vis[lc];
  const double4 x4 = *reinterpret_cast<const double4*>(W.lm + 4 * (size_t)lc);
  const size_t gi0 = (size_t)(f * CP) * L + lc;
  double w0 = W.obs_w[gi0], w1 = 0.0;
  double2 z0 = W.obs_z[gi0], z1 = make_double2(0, 0);
  if (CP > 1) { w1 = W.obs_w[gi0 + L]; z1 = W.obs_z[gi0 + L]; }
  double sg[3] = {0, 0, 0}, sE[3] = {1, 1, 1}, sgn[3] = {0, 0, 0};
  if (mode == MODE_STEP) {
    const double* g = W.lm_g[cur] + 3 * (size_t)lc;
    const double* E = W.lm_E[cur] + 3 * (size_t)lc;
    const double* gn = W.lm_gn + 3 * (size_t)lc;
#pragma unroll
    for (int c = 0; c < 3; ++c) { sg[c] = g[c]; sE[c] = E[c]; sgn[c] = gn[c]; }
  }
  {
    const double* src = reinterpret_cast<const double*>(W.slot_ctx + f * CP);
    double* dst = reinterpret_cast<double*>(slots);
    const int n = CP * (int)(sizeof(SlotCtx) / sizeof(double));
    for (int i = tid; i < n; i += L1_THREADS) dst[i] = src[i];
  }
  if (tid < 3) s_tw[tid] = W.pose_c[7 * f + tid];
#pragma unroll
  for (int i = 0; i < 29; ++i) sred[i][tid] = 0.0;   // contributions go straight to shared memory (no live registers)
  __syncthreads();

  if (l < L) {
    const bool vis = (vmask >> f) & 1u;
    if (vis || f == 0) {
      double X[4] = {x4.x, x4.y, x4.z, x4.w};
      if (mode == MODE_STEP) {
        const double a = st->a, b = st->b;
        double dn = 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const double dlt = a * sg[c] / sE[c] + b * sgn[c];
          X[c] += dlt;
          dn += dlt * dlt;
        }
        if (f == 0) sred[28][tid] = dn;
      }
      if (f == 0) *reinterpret_cast<double4*>(W.lm_c + 4 * (size_t)l) = make_double4(X[0], X[1], X[2], X[3]);
      if (vis) {
        double M0 = 0, M1 = 0, M2 = 0, M3 = 0, M4 = 0, M5 = 0, m0 = 0, m1 = 0, m2 = 0, cost = 0, lprod = 1.0;
        auto add_obs = [&](const SlotCtx& sc, double wobs, double2 z) {
          if (wobs > 0.0 && sc.valid) {
            double r[2], A[6];
            reproj_slot<true>(sc.xf, sc.cam, X, z.x, z.y, wobs, r, A);
            const double sq = r[0] * r[0] + r[1] * r[1];
            double rho1 = 1.0;
            if (cauchy) {          // 0.5 log(1 + s) per block: the logs of a frame's cameras are taken as one log of the product
              rho1 = 1.0 / (1.0 + sq);
              lprod *= 1.0 + sq;
              if (lprod > 1e250) { cost += 0.5 * log(lprod); lprod = 1.0; }
            } else cost += 0.5 * sq;
            M0 += rho1 * (A[0] * A[0] + A[3] * A[3]);
            M1 += rho1 * (A[0] * A[1] + A[3] * A[4]);
            M2 += rho1 * (A[0] * A[2] + A[3] * A[5]);
            M3 += rho1 * (A[1] * A[1] + A[4] * A[4]);
            M4 += rho1 * (A[1] * A[2] + A[4] * A[5]);
            M5 += rho1 * (A[2] * A[2] + A[5] * A[5]);
            m0 += rho1 * (A[0] * r[0] + A[3] * r[1]);
            m1 += rho1 * (A[1] * r[0] + A[4] * r[1]);
            m2 += rho1 * (A[2] * r[0] + A[5] * r[1]);
          }
        };
        add_obs(slots[0], w0, z0);
        if (CP > 1) add_obs(slots[1], w1, z1);
        for (int c = 2; c < CP; ++c) {
          const size_t gi = gi0 + (size_t)c * L;
          add_obs(slots[c], W.obs_w[gi], W.obs_z[gi]);
        }
        if (cauchy) cost += 0.5 * log(lprod);
        double* Mo = W.lm_M + lm_M_index(l, f, W.K);          // tile-major: a warp stores 256-byte rows
        Mo[0] = M0; Mo[32] = M1; Mo[64] = M2; Mo[96] = M3; Mo[128] = M4; Mo[160] = M5;
        double* mo = W.lm_mf + lm_mf_index(l, f, W.K);
        mo[0] = m0; mo[32] = m1; mo[64] = m2;
        // pose-block contributions: G = [w I, -[p]x], p = X - t_WS w
        const double w = X[3];
        const double p0 = X[0] - s_tw[0] * w, p1 = X[1] - s_tw[1] * w, p2 = X[2] - s_tw[2] * w;
        const double Q00 = M1 * p2 - M2 * p1, Q01 = -M0 * p2 + M2 * p0, Q02 = M0 * p1 - M1 * p0;
        const double Q10 = M3 * p2 - M4 * p1, Q11 = -M1 * p2 + M4 * p0, Q12 = M1 * p1 - M3 * p0;
        const double Q20 = M4 * p2 - M5 * p1, Q21 = -M2 * p2 + M5 * p0, Q22 = M2 * p1 - M4 * p0;
        const double w2 = w * w;
        sred[0][tid] = w2 * M0; sred[1][tid] = w2 * M1; sred[2][tid] = w2 * M2; sred[3][tid] = w2 * M3; sred[4][tid] = w2 * M4; sred[5][tid] = w2 * M5;
        sred[6][tid] = -w * Q00; sred[7][tid] = -w * Q01; sred[8][tid] = -w * Q02;
        sred[9][tid] = -w * Q10; sred[10][tid] = -w * Q11; sred[11][tid] = -w * Q12;
        sred[12][tid] = -w * Q20; sred[13][tid] = -w * Q21; sred[14][tid] = -w * Q22;
        sred[15][tid] = p2 * Q10 - p1 * Q20; sred[16][tid] = p2 * Q11 - p1 * Q21; sred[17][tid] = p2 * Q12 - p1 * Q22;
        sred[18][tid] = -p2 * Q01 + p0 * Q21; sred[19][tid] = -p2 * Q02 + p0 * Q22;
        sred[20][tid] = p1 * Q02 - p0 * Q12;
        sred[21][tid] = w * m0; sred[22][tid] = w * m1; sred[23][tid] = w * m2;
        sred[24][tid] = p1 * m2 - p2 * m1; sred[25][tid] = p2 * m0 - p0 * m2; sred[26][tid] = p0 * m1 - p1 * m0;
        sred[27][tid] = cost;
      }
    }
  }
  // ---- CTA reduction of the 29 used values (fixed order -> deterministic): 4 threads per value, each sums
  // 32 of the 128 columns serially (no shuffles), then two shuffle steps combine the four partials
  __syncthreads();
  {
    const int e = tid >> 2, q = tid & 3;
    double s = 0.0;
    if (e < 29) {
      const double* row = &sred[e][q * 32];
#pragma unroll 8
      for (int i = 0; i < 32; ++i) s += row[(i + 4 * q) & 31];     // rotated start: the four partial sums hit different banks
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    if (e < 29 && q == 0) W.partH[((size_t)cx * W.K + f) * kPartH + e] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// Landmark blocks: one thread per landmark.  H_ll = sum_f M_f, g_l = -sum_f m_f, the metric E_l,
// R = H_ll + mu E and its Cholesky factor: stores R^-1 (back-substitution), L^-1 (Schur tile),
// g_l, E_l and z = L^-1 g_l.  [f][l] layouts make every load/store coalesced.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_lmblock(const WinDev* __restrict__ wins, int win_first) {
  const WinDev& W = wins[win_first + blockIdx.y];
  SolverState* st = W.st;
  if (st->done) return;
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  const int L = W.L, K = W.K;
  if (l >= L) return;
  const int mode = st->mode, cur = st->cur;
  const double mu = (mode == MODE_STEP) ? fmax(kMinMu, 2.0 * st->mu / kMuIncrease) : st->mu;
  double H[6] = {0, 0, 0, 0, 0, 0}, gl[3] = {0, 0, 0};
  uint32_t vis = W.lm_vis[l];
  for (int f = 0; f < K; ++f) {
    if ((vis >> f) & 1u) {
      const double* Mo = W.lm_M + lm_M_index(l, f, K);
      const double* mo = W.lm_mf + lm_mf_index(l, f, K);
#pragma unroll
      for (int i = 0; i < 6; ++i) H[i] += Mo[32 * i];
      gl[0] -= mo[0]; gl[1] -= mo[32]; gl[2] -= mo[64];
    }
  }
  double sc3[3], E[3];
  const double hd[3] = {H[0], H[3], H[5]};
  if (mode == MODE_INIT) {
#pragma unroll
    for (int c = 0; c < 3; ++c) { sc3[c] = 1.0 / (1.0 + sqrt(hd[c])); W.lm_scale[3 * (size_t)l + c] = sc3[c]; }
  } else {
#pragma unroll
    for (int c = 0; c < 3; ++c) sc3[c] = W.lm_scale[3 * (size_t)l + c];
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const double s2 = sc3[c] * sc3[c];
    E[c] = fmin(fmax(s2 * hd[c], kMinDiag), kMaxDiag) / s2;
  }
  const double R[6] = {H[0] + mu * E[0], H[1], H[2], H[3] + mu * E[1], H[4], H[5] + mu * E[2]};
  double Lc[6], Li[6];
  if (chol3(R, Lc)) linv3(Lc, Li);
  else {
#pragma unroll
    for (int i = 0; i < 6; ++i) Li[i] = 0.0;
    st->numeric_fail = 1;
  }
  double* Ro = W.lm_Rinv + 6 * (size_t)l;
  Ro[0] = Li[0] * Li[0] + Li[1] * Li[1] + Li[3] * Li[3];
  Ro[1] = Li[1] * Li[2] + Li[3] * Li[4];
  Ro[2] = Li[3] * Li[5];
  Ro[3] = Li[2] * Li[2] + Li[4] * Li[4];
  Ro[4] = Li[4] * Li[5];
  Ro[5] = Li[5] * Li[5];
  double* gs = W.lm_g[cur ^ 1] + 3 * (size_t)l;
  double* Es = W.lm_E[cur ^ 1] + 3 * (size_t)l;
#pragma unroll
  for (int c = 0; c < 3; ++c) { gs[c] = gl[c]; Es[c] = E[c]; }
  double* Lo = W.lm_Li + 9 * (size_t)l;     // L^-1 (6) | z (3)
#pragma unroll
  for (int i = 0; i < 6; ++i) Lo[i] = Li[i];
  Lo[6] = Li[0] * gl[0];
  Lo[7] = Li[1] * gl[0] + Li[2] * gl[1];
  Lo[8] = Li[3] * gl[0] + Li[4] * gl[1] + Li[5] * gl[2];
}

// ------------------------------------------------------------------------------------------------
// A2: Schur complement of the landmark blocks,  S = sum_l Y_l Y_l^T  with  Y_l = W_l L_l^-T  (6K+1 rows: the
// pose rows of the frames that see landmark l, plus the augmented row z_l = L_l^-1 g_l that yields the
// reduced right-hand side).
//
// Landmarks arrive sorted by (first, last) observing frame, so a tile of 32 consecutive landmarks only
// touches the frames [fa, fb] listed in W.tile_range.  Y is built tile-local in shared memory, k-major (column
// k = 3 * landmark + c): local row 6(f - fa) + i is pose row 6f + i, local row 6u (u = fb - fa + 1) is the
// augmented row, and rows up to the next multiple of 8 are zero (see schur_ldy).  The SYRK runs on the FP64 tensor cores
// (mma.sync.m8n8k4.f64) over the T = ceil((6u+1)/8) block rows: the lower-triangle 8x8 blocks are dealt to the
// warps as contiguous row-major ranges (at most one block above the average; neighbours share a block row, so
// the A fragment is loaded once for both), two blocks interleaved per warp.  The owning lane adds its fragment
// to the chunk's packed accumulator in shared memory (or to the global partial for windows with many frames):
// the local -> global row map is monotone and injective, so there is one writer per element per tile, and
// tiles are separated by the tile loop's barriers => deterministic.
// ------------------------------------------------------------------------------------------------
constexpr int kLiStride = 9;   // L^-1 (6) | z (3), as in global memory (one bulk copy per tile)

// Y row stride (doubles): at least the 6K+1 rows of the widest tile, and 4 (mod 8) so that the DMMA fragment loads
// (lane 4g + t reads t * ldy + g) and the Y-build double2 stores (4 landmarks x 2 frames per quarter warp) hit
// distinct banks.  The padding rows of a full-width tile's last block row may reach beyond the stride: they alias the
// first rows of the next column (or the 8-double pad after the tile) and only feed output entries that are dropped.
__host__ __device__ inline int schur_ldy(int K) { return 6 * K + 1 + ((3 - 6 * K) & 7); }

// acc_smem: 1 = the chunk's Schur accumulator (packed lower triangle of the (dc+1) x (dc+1) matrix) lives in
// shared memory; 0 = accumulate in the chunk's global partial instead (windows with many frames).
__host__ __device__ inline size_t schur_acc_doubles(int K) { return (size_t)(6 * K + 1) * (6 * K + 2) / 2; }
__host__ __device__ inline size_t smemA2_bytes(int K, int acc_smem) {
  size_t b = 16;                                                    // two mbarriers (TMA completion per buffer)
  b += ((size_t)3 * A2_TILE * schur_ldy(K) + 8) * sizeof(double);  // Y tile, k-major (+ pad: the last block row of a full-width tile)
  b += (size_t)2 * K * 6 * A2_TILE * sizeof(double);               // M tiles [f][e][ll] (double buffered)
  b += (size_t)2 * A2_TILE * kLiStride * sizeof(double);           // L^-1 | z
  b += (size_t)2 * A2_TILE * 4 * sizeof(double);                   // X
  b += (size_t)K * 4 * sizeof(double);                             // frame translations
  b += (size_t)acc_smem * schur_acc_doubles(K) * sizeof(double);
  return b;
}

// ---- TMA bulk copies (cp.async.bulk, 1-D) completing on an mbarrier
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
               "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
  } while (!ok);
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// C += A B on the FP64 tensor cores, fragment layout of m8n8k4 f64: lane 4g + t holds A[g][t], B[t][g], C[g][2t..2t+1]
__device__ __forceinline__ void dmma_8x8x4(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(A2_THREADS, 2) k_schur(const WinDev* __restrict__ wins, int win_first, int acc_smem, int max_iterations) {
  const WinDev& W = wins[win_first + blockIdx.y];
  SolverState* st = W.st;
  if (st->done) return;
  // the step being judged in this round is the last one (iteration limit): k_solve will not build another
  // reduced system, so the Schur complement of this linearisation is never used
  if (st->iteration >= max_iterations) return;
  const int chunk = blockIdx.x;
  if (chunk >= W.n_chunks) return;
  const int tid = threadIdx.x;
  const int K = W.K, dc = W.dc, dcp = W.dcp, L = W.L;
  const int ldy = schur_ldy(K);

  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw);            // [2]: TMA completion of tile buffer 0 / 1
  double* Yt = reinterpret_cast<double*>(smem_raw + 16);
  double* sMb = Yt + (size_t)3 * A2_TILE * ldy + 8;
  double* sLib = sMb + (size_t)2 * K * 6 * A2_TILE;
  double* sXb = sLib + 2 * A2_TILE * kLiStride;
  double* tws = sXb + 2 * A2_TILE * 4;
  double* Sp = W.partA + (size_t)chunk * W.partA_stride;
  double* Sacc = acc_smem ? tws + 4 * K : Sp;     // packed lower triangle in shared memory, or the global partial itself
  const int n_acc = acc_smem ? (dc + 1) * (dc + 2) / 2 : dcp * dcp;

  for (int f = tid; f < K; f += A2_THREADS) {
    tws[4 * f] = W.pose_c[7 * f]; tws[4 * f + 1] = W.pose_c[7 * f + 1]; tws[4 * f + 2] = W.pose_c[7 * f + 2];
  }
  for (int i = tid; i < n_acc; i += A2_THREADS) Sacc[i] = 0.0;
  if (tid < 8) Yt[(size_t)3 * A2_TILE * ldy + tid] = 0.0;

  const int lm_begin = chunk * W.lm_per_chunk;     // multiple of A2_TILE
  const int lm_end = min(L, lm_begin + W.lm_per_chunk);

  // Asynchronous staging of one tile by the TMA engine (cp.async.bulk, issued by the last warp, completion on
  // mbar[buf]); frames [fa, fb] only.  Global and shared layouts agree, so every piece is one contiguous copy:
  //   M  [tile][f][6][32] -> sM[f][6][32] : frames [fa, fb] are one contiguous block
  //   Li [l][9] -> sLi[32][9] (2304 B),  X = lm_c [l][4] -> sX[32][4] (1024 B)
  // Rows beyond the chunk's last landmark read allocated padding (Lp) and are never used.
  const int warp = tid >> 5, lane = tid & 31;
  if (tid == 0) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); fence_proxy_async(); }
  __syncthreads();
  uint32_t phase_bits = 0;      // bit b: parity to wait for on mbar[b]
  auto stage = [&](int base, int buf, uint32_t tr) {
    const int fa = tr & 0xffu, fb = tr >> 8;
    if (fa > fb || warp != A2_THREADS / 32 - 1) return;      // the last warp issues the copies
    double* sM = sMb + (size_t)buf * K * 6 * A2_TILE;
    double* sLi = sLib + buf * A2_TILE * kLiStride;
    double* sX = sXb + buf * A2_TILE * 4;
    // three copies per tile: the M block of frames [fa, fb] (contiguous in the tile-major layout), L^-1|z, X
    if (lane == 0) {       // (the buffer's last generic-proxy reads are ordered before this point by the CTA barrier)
      const uint32_t m_bytes = (uint32_t)(fb - fa + 1) * 6 * A2_TILE * 8;
      mbar_arrive_expect_tx(&mbar[buf], m_bytes + A2_TILE * kLiStride * 8 + A2_TILE * 4 * 8);
      bulk_g2s(sM + (size_t)fa * 6 * A2_TILE, W.lm_M + lm_M_index(base, fa, K), m_bytes, &mbar[buf]);
      bulk_g2s(sLi, W.lm_Li + (size_t)kLiStride * base, A2_TILE * kLiStride * 8, &mbar[buf]);
      bulk_g2s(sX, W.lm_c + 4 * (size_t)base, A2_TILE * 4 * 8, &mbar[buf]);
    }
  };

  // Adds the fragment (c0, c1) of local block (bi, bj) to the chunk accumulator: lane 4g + t holds local row
  // 8 bi + g, columns 8 bj + 2t and 8 bj + 2t + 1.  Padding rows, entries above the diagonal and the z z^T corner
  // (not part of S) are dropped.
  const int g = lane >> 2, t4 = lane & 3;
  auto accumulate = [&](int bi, int bj, double c0, double c1, int row0, int nrow) {
    const int i = 8 * bi + g;
    if (i > nrow) return;
    const int gr = i < nrow ? row0 + i : dc;
    double* rp = Sacc + (acc_smem ? (size_t)gr * (gr + 1) / 2 : (size_t)gr * dcp) + row0;
    const int j = 8 * bj + 2 * t4;
    if (j <= i && j < nrow) rp[j] += c0;
    if (j + 1 <= i && j + 1 < nrow) rp[j + 1] += c1;
  };

#ifdef OKB_SCHUR_PROF     // per-phase cycle counters of chunk 0 / thread 0 (diagnostics builds only): phase_ns[8 + i] for
                          // i = 0 TMA wait + barrier, 1 copy issue, 2 Y build, 3 DMMA, 4 accumulate, 5 copy-out
  const bool prof = (tid == 0 && chunk == 0);
  unsigned long long t_ph = 0, ph[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  auto now = []() { return (unsigned long long)clock64(); };
#define SCHUR_MARK(i) do { if (prof) { const unsigned long long n_ = now(); ph[i] += n_ - t_ph; t_ph = n_; } } while (0)
  if (prof) t_ph = now();
#else
#define SCHUR_MARK(i) do { } while (0)
#endif
  int buf = 0;
  // frame ranges are fetched two tiles ahead so that no global-load latency sits on the tile loop
  const int last_tile = (lm_end - 1) >> 5;
  uint32_t tr_cur = (lm_begin < lm_end) ? W.tile_range[lm_begin >> 5] : 1u;
  uint32_t tr_n1 = (lm_begin + A2_TILE < lm_end) ? W.tile_range[(lm_begin >> 5) + 1] : 1u;
  if (lm_begin < lm_end) stage(lm_begin, 0, tr_cur);
  for (int base = lm_begin; base < lm_end; base += A2_TILE) {
    const uint32_t tr_n2 = W.tile_range[min((base >> 5) + 2, last_tile)];
    const int nl = min(A2_TILE, lm_end - base);
    const double* sM = sMb + (size_t)buf * K * 6 * A2_TILE;
    const double* sLi = sLib + buf * A2_TILE * kLiStride;
    const double* sX = sXb + buf * A2_TILE * 4;
    if ((tr_cur & 0xffu) <= (tr_cur >> 8)) {           // this tile was staged: wait for its bytes
      mbar_wait(&mbar[buf], (phase_bits >> buf) & 1u);
      phase_bits ^= 1u << buf;
    }
    __syncthreads();                       // the previous SYRK has finished (Y tile and the other buffer are free)
    SCHUR_MARK(0);
    if (base + A2_TILE < lm_end) stage(base + A2_TILE, buf ^ 1, tr_n1);   // overlaps with this tile's math
    SCHUR_MARK(1);
    const uint32_t tr = tr_cur;
    tr_cur = tr_n1; tr_n1 = tr_n2;
    const int fa = tr & 0xffu, fb = tr >> 8;
    buf ^= 1;
    if (fa > fb) continue;                 // no observed landmark in this tile (CTA-uniform)
    const int u = fb - fa + 1, nrow = 6 * u, row0 = 6 * fa;
    const int T = (nrow + 8) >> 3;         // 8-row blocks covering the pose rows and z
    // ---- augmented row z (local row nrow) and zero rows up to 8T (or the stride)
    for (int i = tid; i < 3 * A2_TILE * (min(8 * T, ldy) - nrow); i += A2_THREADS) {
      const int k = i % (3 * A2_TILE), r = nrow + i / (3 * A2_TILE), ll = k / 3;
      Yt[(size_t)k * ldy + r] = (r == nrow && ll < nl) ? sLi[ll * kLiStride + 6 + k % 3] : 0.0;
    }
    // ---- Y_f = W_f L^-T for every (landmark, frame) pair of the tile, frames [fa, fb].  Pair p: bits 0-1 and 3-5
    // are the landmark, bit 2 and bits 6.. the frame, so a quarter warp stores 4 landmarks x 2 frames
    // (conflict-free double2 stores with ldy = 4 mod 8).
    for (int p = tid; p < A2_TILE * ((u + 1) & ~1); p += A2_THREADS) {
      const int ll = (p & 3) | ((p >> 1) & 28), fl = ((p >> 2) & 1) | ((p >> 5) & ~1);
      if (fl >= u) continue;
      const int f = fa + fl;
      double2* y0 = reinterpret_cast<double2*>(Yt + (size_t)(3 * ll) * ldy + 6 * fl);
      double2* y1 = reinterpret_cast<double2*>(Yt + (size_t)(3 * ll + 1) * ldy + 6 * fl);
      double2* y2 = reinterpret_cast<double2*>(Yt + (size_t)(3 * ll + 2) * ldy + 6 * fl);
      double M0 = 0, M1 = 0, M2 = 0, M3 = 0, M4 = 0, M5 = 0;
      if (ll < nl) {
        const double* sp = sM + (size_t)(f * 6) * A2_TILE + ll;
        M0 = sp[0]; M1 = sp[A2_TILE]; M2 = sp[2 * A2_TILE]; M3 = sp[3 * A2_TILE]; M4 = sp[4 * A2_TILE]; M5 = sp[5 * A2_TILE];
      }
      if (M0 != 0.0 || M3 != 0.0 || M5 != 0.0) {
        const double* Li = sLi + ll * kLiStride;
        const double w = sX[ll * 4 + 3];
        const double p0 = sX[ll * 4] - tws[4 * f] * w, p1 = sX[ll * 4 + 1] - tws[4 * f + 1] * w, p2 = sX[ll * 4 + 2] - tws[4 * f + 2] * w;
        const double N00 = M0 * Li[0], N01 = M0 * Li[1] + M1 * Li[2], N02 = M0 * Li[3] + M1 * Li[4] + M2 * Li[5];
        const double N10 = M1 * Li[0], N11 = M1 * Li[1] + M3 * Li[2], N12 = M1 * Li[3] + M3 * Li[4] + M4 * Li[5];
        const double N20 = M2 * Li[0], N21 = M2 * Li[1] + M4 * Li[2], N22 = M2 * Li[3] + M4 * Li[4] + M5 * Li[5];
        y0[0] = make_double2(-w * N00, -w * N10); y0[1] = make_double2(-w * N20, -(p1 * N20 - p2 * N10));
        y0[2] = make_double2(-(p2 * N00 - p0 * N20), -(p0 * N10 - p1 * N00));
        y1[0] = make_double2(-w * N01, -w * N11); y1[1] = make_double2(-w * N21, -(p1 * N21 - p2 * N11));
        y1[2] = make_double2(-(p2 * N01 - p0 * N21), -(p0 * N11 - p1 * N01));
        y2[0] = make_double2(-w * N02, -w * N12); y2[1] = make_double2(-w * N22, -(p1 * N22 - p2 * N12));
        y2[2] = make_double2(-(p2 * N02 - p0 * N22), -(p0 * N12 - p1 * N02));
      } else {
        const double2 z = make_double2(0.0, 0.0);
#pragma unroll
        for (int i = 0; i < 3; ++i) { y0[i] = z; y1[i] = z; y2[i] = z; }
      }
    }
    __syncthreads();
    SCHUR_MARK(2);
    // ---- SYRK: this warp's range of the T(T+1)/2 lower-triangle blocks (row-major), two at a time, each over
    // ceil(3 nl / 4) k-steps (columns from 3 nl on are zero)
    const int ns = (3 * nl + 3) >> 2;
    const int nb = T * (T + 1) / 2;
    constexpr int NW = A2_THREADS / 32;
    const int b_lo = warp * nb / NW, b_hi = (warp + 1) * nb / NW;
    int bi = (int)((sqrtf(8.0f * (float)b_lo + 1.0f) - 1.0f) * 0.5f);
    while (bi * (bi + 1) / 2 > b_lo) --bi;
    while ((bi + 1) * (bi + 2) / 2 <= b_lo) ++bi;
    int bj = b_lo - bi * (bi + 1) / 2;
    const double* yl = Yt + (size_t)t4 * ldy + g;
    const int kstep = 4 * ldy;
    for (int b = b_lo; b < b_hi; b += 2) {
      int bi1 = bi, bj1 = bj + 1;
      if (bj1 > bi1) { ++bi1; bj1 = 0; }
      double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
      const double* pa0 = yl + 8 * bi;
      const double* pb0 = yl + 8 * bj;
      const bool diag0 = bi == bj;
      if (b + 1 < b_hi) {
        const double* pa1 = yl + 8 * bi1;
        const double* pb1 = yl + 8 * bj1;
        const bool diag1 = bi1 == bj1, same_row = bi1 == bi;
#pragma unroll 4
        for (int s = 0; s < ns; ++s) {
          const int o = s * kstep;
          const double a0 = pa0[o];
          const double b0 = diag0 ? a0 : pb0[o];
          const double a1 = same_row ? a0 : pa1[o];
          const double b1 = diag1 ? a1 : pb1[o];
          dmma_8x8x4(c00, c01, a0, b0);
          dmma_8x8x4(c10, c11, a1, b1);
        }
      } else {
#pragma unroll 4
        for (int s = 0; s < ns; ++s) {
          const int o = s * kstep;
          const double a0 = pa0[o];
          const double b0 = diag0 ? a0 : pb0[o];
          dmma_8x8x4(c00, c01, a0, b0);
        }
      }
      SCHUR_MARK(3);
      accumulate(bi, bj, c00, c01, row0, nrow);
      if (b + 1 < b_hi) accumulate(bi1, bj1, c10, c11, row0, nrow);
      SCHUR_MARK(4);
      bi = bi1; bj = bj1 + 1;
      if (bj > bi) { ++bi; bj = 0; }
    }
  }
  if (acc_smem) {
    __syncthreads();
    for (int i = tid; i < (dc + 1) * dcp; i += A2_THREADS) {
      const int r = i / dcp, cidx = i % dcp;
      if (cidx <= r) Sp[i] = Sacc[r * (r + 1) / 2 + cidx];
    }
  }
  SCHUR_MARK(5);
#ifdef OKB_SCHUR_PROF
  if (prof) for (int i = 0; i < 8; ++i) st->phase_ns[8 + i] += ph[i];
#endif
#undef SCHUR_MARK
}

// Sums the per-chunk Schur accumulators of a window into chunk 0 (fixed order => deterministic), in
// parallel over the matrix elements, so that k_solve reads one partial regardless of the chunk count.
__global__ void __launch_bounds__(256) k_reduce_partials(const WinDev* __restrict__ wins, int win_first) {
  const WinDev& W = wins[win_first + blockIdx.y];
  if (W.st->done || W.n_chunks <= 1) return;
  const int n = W.dcp * W.dcp;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double s = W.partA[i];
    for (int c = 1; c < W.n_chunks; ++c) s += W.partA[(size_t)c * W.partA_stride + i];
    W.partA[i] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// Landmark-sharded window: k_reduce_partials fused with the push half of the all-reduce.  Every rank sums its
// chunk partials (Schur accumulator) and its per-CTA pose-block records in fixed order and stores the result with
// plain stores into box [parity][rank] of EVERY rank's mailbox (its own included) -- remote stores travel over
// NVLink / NVSwitch and are not waited for.  The last CTA of the window fences at system scope and releases the
// `world` ready flags.  The sum over ranks happens in k_solve's prologue (every rank adds the boxes in rank order
// => bit-identical reduced systems, so the redundant reduced solves stay in lock step).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ double* shard_box(const WinDev& W, int dst, int parity, int src) {
  return reinterpret_cast<double*>(W.shard_mail[dst] + kShardHeaderBytes) + ((size_t)parity * W.shard_world + src) * W.shard_box_cap;
}
__device__ __forceinline__ unsigned long long* shard_flag(const WinDev& W, int dst, size_t which, int parity, int src) {
  return reinterpret_cast<unsigned long long*>(W.shard_mail[dst] + which) + parity * kMaxShard + src;
}

__global__ void __launch_bounds__(256) k_shard_push(const WinDev* __restrict__ wins, int win_first) {
  const WinDev& W = wins[win_first + blockIdx.y];
  SolverState* st = W.st;
  if (st->done) return;
  const int world = W.shard_world, me = W.shard_rank;
  const unsigned long long epoch = st->shard_epoch + 1;
  const int par = (int)(epoch & 1ull);
  const int K = W.K, nA = W.dcp * W.dcp, nH = K * kPartH;
  const int n = nA + nH + 8;
  const int n_cx = (W.L + L1_THREADS - 1) / L1_THREADS;
  double* dst[kMaxShard];
#pragma unroll
  for (int r = 0; r < kMaxShard; ++r) dst[r] = (r < world) ? shard_box(W, r, par, me) : nullptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double s = 0.0;
    if (i < nA) {
      s = W.partA[i];
      for (int c = 1; c < W.n_chunks; ++c) s += W.partA[(size_t)c * W.partA_stride + i];
    } else if (i < nA + nH) {
      const int j = i - nA, f = j / kPartH, e = j % kPartH;
      if (e < 29)
        for (int c = 0; c < n_cx; ++c) s += W.partH[((size_t)c * K + f) * kPartH + e];
    } else if (i == nA + nH) {
      s = st->numeric_fail ? 1.0 : 0.0;
    }
#pragma unroll
    for (int r = 0; r < kMaxShard; ++r)
      if (r < world) dst[r][i] = s;
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int* counter = reinterpret_cast<unsigned int*>(W.shard_mail[me] + kShardCounter);
    const unsigned int prev = atomicAdd(counter, 1u);
    if (prev == gridDim.x - 1) {
      *counter = 0u;
      __threadfence_system();
      for (int r = 0; r < world; ++r) st_release_sys_u64(shard_flag(W, r, kShardFlags1, par, me), epoch);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Post-solve landmark quality: H = sum J_lm^T J_lm (sqrt-information weighted, no robust weight)
// at the final estimate; quality = sqrt(lambda_min)/sqrt(lambda_max), 0 if lambda_min < 1e-12.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_quality(const WinDev* __restrict__ wins, int win_first) {
  const WinDev& W = wins[win_first + blockIdx.y];
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SlotCtx* slots = reinterpret_cast<SlotCtx*>(smem_raw);
  const int tid = threadIdx.x;
  for (int s = tid; s < W.NS; s += blockDim.x) {
    const SlotInfo si = W.slots[s];
    SlotCtx& sc = slots[s];
    sc.valid = si.valid; sc.frame = si.valid ? si.pose_idx : 0;
    if (si.valid) { make_slot_xf(W.pose + 7 * si.pose_idx, W.ext + 7 * si.ext_idx, sc.xf); cam_load(W.cams[si.cam_idx], sc.cam); }
  }
  __syncthreads();
  const int L = W.L, CP = W.CP;
  for (int l = blockIdx.x * blockDim.x + tid; l < L; l += gridDim.x * blockDim.x) {
    const double4 x4 = *reinterpret_cast<const double4*>(W.lm + 4 * (size_t)l);
    const double X[4] = {x4.x, x4.y, x4.z, x4.w};
    double H[6] = {0, 0, 0, 0, 0, 0};
    uint32_t vis = W.lm_vis[l];
    while (vis) {
      const int f = __ffs(vis) - 1;
      vis &= vis - 1;
      for (int c = 0; c < CP; ++c) {
        const int s = f * CP + c;
        const double wobs = W.obs_w[(size_t)s * L + l];
        if (wobs > 0.0 && slots[s].valid) {
          const double2 z = W.obs_z[(size_t)s * L + l];
          double r[2], A[6];
          reproj_slot<true>(slots[s].xf, slots[s].cam, X, z.x, z.y, wobs, r, A);
          H[0] += A[0] * A[0] + A[3] * A[3]; H[1] += A[0] * A[1] + A[3] * A[4]; H[2] += A[0] * A[2] + A[3] * A[5];
          H[3] += A[1] * A[1] + A[4] * A[4]; H[4] += A[1] * A[2] + A[4] * A[5]; H[5] += A[2] * A[2] + A[5] * A[5];
        }
      }
    }
    double ev[3];
    eig3sym_closed(H, ev);
    const double q = (ev[0] < 1.0e-12) ? 0.0 : sqrt(ev[0]) / sqrt(ev[2]);
    W.quality[l] = q;
    // write-back in the caller's order: the master copy (next compile) and the packed download block
    const uint32_t lc = W.perm[l];
    *reinterpret_cast<double4*>(W.m_lm + 4 * (size_t)lc) = x4;
    double* o = W.out + out_lm_offset(W.K, W.NSB);
    *reinterpret_cast<double4*>(o + 4 * (size_t)lc) = x4;
    o[4 * (size_t)L + lc] = q;
  }
  if (blockIdx.x == 0) {
    for (int i = tid; i < 7 * W.K; i += blockDim.x) W.out[i] = W.pose[i];
    for (int i = tid; i < 9 * W.NSB; i += blockDim.x) W.out[7 * W.K + i] = W.sb[i];
  }
}

}  // namespace okb
