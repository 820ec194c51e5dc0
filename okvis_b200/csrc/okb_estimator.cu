// Host side of the estimator path of libokvis_b200.so: context, window packing/upload, the solver
// launch sequence, download, and the single-residual-block test hooks.  C-ABI: include/okvis_b200.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "okb_ctx.h"
#include "okb_hostpack.hpp"
#include "okb_graph.cuh"
#include "okb_kernels.cuh"
#include "okb_marg.cuh"

using namespace okb;

static std::string g_create_error;

#define OKB_CUDA(ctx, call)                                                                             \
  do {                                                                                                  \
    cudaError_t e_ = (call);                                                                            \
    if (e_ != cudaSuccess) {                                                                            \
      (ctx)->set_error(std::string(#call) + ": " + cudaGetErrorString(e_));                             \
      return OKB_ERR_CUDA;                                                                              \
    }                                                                                                   \
  } while (0)

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
// The transfer stream gets the highest priority: its small kernels (k_zero / k_prepare) are scheduled as soon
// as CTA slots free up instead of waiting behind the solver kernels of other slots.
static cudaError_t create_transfer_stream(cudaStream_t* s) {
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);
  return cudaStreamCreateWithPriority(s, cudaStreamNonBlocking, hi);
}

extern "C" int okb_ctx_create(int device_id, int max_windows, okb_ctx** out) {
  if (!out || max_windows < 1) return OKB_ERR_INVALID_ARG;
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
    return OKB_ERR_NO_DEVICE;
  }
  if (device_id < 0 || device_id >= n) { g_create_error = "bad device id"; return OKB_ERR_INVALID_ARG; }
  okb_ctx* c = new okb_ctx();
  c->device = device_id;
  c->max_windows = max_windows;
  // the landmark / solve chain is the critical path of a round: it runs at the highest stream priority, the IMU terms
  // (side stream, a long tail of one-warp CTAs) at the lowest, so they fill what the chain leaves idle
  int prio_least = 0, prio_greatest = 0;
  if (cudaSetDevice(device_id) == cudaSuccess) cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest);
  if (cudaSetDevice(device_id) != cudaSuccess || cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_greatest) != cudaSuccess) {
    g_create_error = "cudaSetDevice / cudaStreamCreate failed";
    delete c;
    return OKB_ERR_CUDA;
  }
  if (cudaStreamCreateWithPriority(&c->stream_imu, cudaStreamNonBlocking, prio_least) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_round, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_imu, cudaEventDisableTiming) != cudaSuccess ||
      create_transfer_stream(&c->stream_xfer) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    g_create_error = "cudaStreamCreate / cudaEventCreate failed";
    delete c;
    return OKB_ERR_CUDA;
  }
  for (int k = 0; k < okb_ctx::kDoneRing; ++k) cudaEventCreateWithFlags(&c->done_ring[k], cudaEventDisableTiming);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device_id);
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = (int)prop.sharedMemPerBlockOptin;
  c->smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
  c->wins.resize(max_windows);
  c->host.assign(max_windows, WinDev());
  std::memset(c->host.data(), 0, sizeof(WinDev) * max_windows);
  c->chunk_cap = std::max(1, std::min(kMaxChunks, (2 * c->sm_count) / max_windows));
  if (cudaMalloc(&c->d_wins, sizeof(WinDev) * max_windows) != cudaSuccess ||
      cudaMalloc(&c->d_states, sizeof(SolverState) * max_windows) != cudaSuccess ||
      cudaMallocHost(&c->h_states, sizeof(SolverState) * max_windows) != cudaSuccess) {
    g_create_error = "cudaMalloc failed";
    delete c;
    return OKB_ERR_CUDA;
  }
  cudaMemset(c->d_states, 0, sizeof(SolverState) * max_windows);
  cudaFuncSetAttribute(k_schur, cudaFuncAttributeMaxDynamicSharedMemorySize, c->smem_optin);
  cudaFuncSetAttribute(k_imu, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemI_bytes());
  cudaFuncSetAttribute(k_imu, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(k_solve<S_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, c->smem_optin);
  cudaFuncSetAttribute(k_solve<S_THREADS>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(k_solve<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, c->smem_optin);
  cudaFuncSetAttribute(k_solve<512>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(k_schur, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(k_quality, cudaFuncAttributeMaxDynamicSharedMemorySize, c->smem_optin);
  *out = c;
  return OKB_OK;
}

extern "C" void okb_ctx_destroy(okb_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  if (c->stream_xfer) cudaStreamSynchronize(c->stream_xfer);
  for (auto& w : c->wins) {
    if (w.arena) cudaFree(w.arena);
    if (w.marg_scratch) cudaFree(w.marg_scratch);
    if (w.staging) cudaFreeHost(w.staging);
    if (w.out_staging) cudaFreeHost(w.out_staging);
    if (w.copied) cudaEventDestroy(w.copied);
    if (w.down) cudaEventDestroy(w.down);
  }
  for (int k = 0; k < okb_ctx::kDoneRing; ++k) if (c->done_ring[k]) cudaEventDestroy(c->done_ring[k]);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->stream_xfer) cudaStreamDestroy(c->stream_xfer);
  okb_frontend_release(c);
  for (int r = 0; r < kMaxShard; ++r)
    if (c->shard_peer_ipc[r] && c->shard_peer[r]) cudaIpcCloseMemHandle(c->shard_peer[r]);
  if (c->shard_local) cudaFree(c->shard_local);
  if (c->d_wins) cudaFree(c->d_wins);
  if (c->d_states) cudaFree(c->d_states);
  if (c->h_states) cudaFreeHost(c->h_states);
  if (c->hook_buf) cudaFree(c->hook_buf);
  for (auto& g : c->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
  for (auto e : c->prof_events) cudaEventDestroy(e);
  if (c->ev_round) cudaEventDestroy(c->ev_round);
  if (c->ev_imu) cudaEventDestroy(c->ev_imu);
  if (c->stream_imu) cudaStreamDestroy(c->stream_imu);
  cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" const char* okb_last_error(const okb_ctx* c) { return c ? c->error.c_str() : g_create_error.c_str(); }
extern "C" int64_t okb_kernel_launches(const okb_ctx* c) { return c ? c->launches : 0; }
extern "C" void* okb_stream(const okb_ctx* c) { return c ? (void*)c->stream : nullptr; }

// ---------------------------------------------------------------------------------------------
// window graph: capacities, arena, command staging, commit (device side: okb_graph.cuh)
// ---------------------------------------------------------------------------------------------
namespace {
struct ArenaPlan {
  size_t total = 0;
  size_t take(size_t bytes) {
    const size_t o = total;
    total = align_up(total + bytes, 256);
    return o;
  }
};

// Orders the solver stream after every transfer issued so far.
int join_transfers(okb_ctx* c) {
  if (cudaEventRecord(c->ev_join, c->stream_xfer) != cudaSuccess) return 1;
  return cudaStreamWaitEvent(c->stream, c->ev_join, 0) != cudaSuccess;
}
// Marks solver-stream work on windows [first, first+count): later transfers of these windows wait for it.
void mark_work(okb_ctx* c, int first, int count) {
  const int k = c->done_next;
  c->done_next = (k + 1) % okb_ctx::kDoneRing;
  cudaEventRecord(c->done_ring[k], c->stream);
  for (int i = first; i < first + count; ++i) c->wins[i].done_idx = k;
}

inline bool caps_cover(const WinCaps& a, const WinCaps& b) {
  return a.K >= b.K && a.L >= b.L && a.O >= b.O && a.S >= b.S && a.T >= b.T && a.NE >= b.NE && a.NC >= b.NC && a.PP >= b.PP && a.MN >= b.MN;
}
inline WinCaps caps_max(const WinCaps& a, const WinCaps& b) {
  return WinCaps{std::max(a.K, b.K), std::max(a.L, b.L), std::max(a.O, b.O), std::max(a.S, b.S), std::max(a.T, b.T),
                 std::max(a.NE, b.NE), std::max(a.NC, b.NC), std::max(a.PP, b.PP), std::max(a.MN, b.MN)};
}
inline size_t full_upload_bytes(const WinCaps& q) {      // command stream of a full upload at these sizes
  return 12 * sizeof(CmdHeader) + 8 * ((size_t)7 * q.NE + 16 * (size_t)q.K + 4 * (size_t)q.L + 2 * kMaxMargBlocks + 16 * kMaxMargBlocks +
                                        (size_t)q.MN * q.MN + q.MN) +
         sizeof(okb_camera) * q.NC + sizeof(okb_observation) * (size_t)q.O + sizeof(okb_imu_term) * q.T + sizeof(okb_imu_sample) * (size_t)q.S +
         (sizeof(okb_pose_prior) + sizeof(okb_sb_prior)) * q.PP + 4096;
}

// Dimensions that follow from the current K / L / NC ... of the host mirror.
void derive_dims(WinDev& W) {
  int CP = 1;
  while (CP < W.NC) CP <<= 1;
  W.CP = CP;
  W.NS = W.K * CP; W.NG = (W.NS + 31) / 32; W.NSP = W.NG * 32;
  W.dc = 6 * W.K; W.d = W.dc + 9 * W.NSB; W.dcp = 4 * ((W.dc + 1 + 3) / 4);
  W.Lp = (W.L + 31) & ~31;
  W.partA_stride = W.dcp * W.dcp;
  W.zero_bytes[0] = align_up(sizeof(double2) * (size_t)W.L * W.NS, 256);
  W.zero_bytes[1] = align_up(sizeof(double) * (size_t)W.L * W.NS, 256);
  W.zero_bytes[2] = align_up(sizeof(double) * 6 * (size_t)W.Lp * W.K, 256);
}

// (Re)plans the slot's arena for `q` and points the host mirror at it.  Contents are lost (callers follow up with a
// full upload).
int plan_arena(okb_ctx* c, int win, const WinCaps& q) {
  WinStore& S = c->wins[win];
  ArenaPlan P;
  int CPc = 1;
  while (CPc < q.NC) CPc <<= 1;
  const int Kc = q.K, Lc = q.L, Lpc = (Lc + 31) & ~31;
  const int NSc = Kc * CPc, NSPc = (NSc + 31) / 32 * 32;
  const int dcc = 6 * Kc, dcap = 15 * Kc, dcpc = 4 * ((dcc + 1 + 3) / 4);
  const int MN = std::max(q.MN, 1), MB = kMaxMargBlocks;
  const size_t o_pose = P.take(8 * 7 * Kc), o_sb = P.take(8 * 9 * Kc), o_ext = P.take(8 * 7 * q.NE), o_mlm = P.take(8 * 4 * (size_t)Lpc);
  const size_t o_out = P.take(8 * (16 * (size_t)Kc + 4 + 5 * (size_t)Lc));
  const size_t o_cams = P.take(sizeof(okb_camera) * q.NC), o_obs = P.take(sizeof(okb_observation) * (size_t)std::max(q.O, 1));
  const size_t o_imut = P.take(sizeof(okb_imu_term) * std::max(q.T, 1)), o_samp = P.take(sizeof(okb_imu_sample) * (size_t)std::max(q.S, 1));
  const size_t o_pp = P.take(sizeof(okb_pose_prior) * std::max(q.PP, 1)), o_sbp = P.take(sizeof(okb_sb_prior) * std::max(q.PP, 1));
  const size_t o_mkind = P.take(4 * MB), o_midx = P.take(4 * MB), o_mcol = P.take(4 * MB), o_moff = P.take(4 * MB);
  const size_t o_mx0 = P.take(8 * 9 * MB), o_mJ = P.take(8 * (size_t)MN * MN), o_me0 = P.take(8 * MN), o_mH0 = P.take(8 * (size_t)MN * MN);
  const size_t o_mHs = P.take(8 * (size_t)MN * MN), o_mb0 = P.take(8 * MN);
  const size_t o_mlmi = P.take(8 * 4 * (size_t)Lpc), o_mark = P.take(Lpc), o_mvis = P.take(4 * (size_t)Lpc);
  const size_t o_bitmap = P.take(4 * (((size_t)NSc * Lc + 31) / 32 + 1));
  const size_t o_perm = P.take(4 * (size_t)Lpc), o_inv = P.take(4 * (size_t)Lpc), o_trange = P.take(4 * (size_t)(Lpc / 32 + 1)), o_vis = P.take(4 * (size_t)Lpc);
  const size_t o_slots = P.take(sizeof(SlotInfo) * NSPc);
  const size_t cmd_cap = align_up(full_upload_bytes(q) + 65536, 256);
  const size_t o_cmd = P.take(cmd_cap);
  // working state / scratch
  const size_t o_lm = P.take(8 * 4 * (size_t)Lpc), o_pose_i = P.take(8 * 7 * Kc), o_sb_i = P.take(8 * 9 * Kc);
  const size_t o_pose_c = P.take(8 * 7 * Kc), o_sb_c = P.take(8 * 9 * Kc), o_lm_c = P.take(8 * 4 * (size_t)Lpc);
  size_t o_lmg[2], o_lmE[2], o_gd[2], o_Ed[2];
  for (int b = 0; b < 2; ++b) { o_lmg[b] = P.take(8 * 3 * (size_t)Lc); o_lmE[b] = P.take(8 * 3 * (size_t)Lc); }
  const size_t o_Rinv = P.take(8 * 6 * (size_t)Lc), o_slotctx = P.take(sizeof(SlotCtx) * NSPc), o_mf = P.take(8 * 3 * (size_t)Lpc * Kc);
  const size_t o_gn = P.take(8 * 3 * (size_t)Lc), o_Li = P.take(8 * 9 * (size_t)Lpc), o_scale = P.take(8 * 3 * (size_t)Lc);
  const int n_cx = (Lc + L1_THREADS - 1) / L1_THREADS;
  const size_t o_partH = P.take(8 * (size_t)n_cx * Kc * kPartH), o_part = P.take(8 * (size_t)dcpc * dcpc * c->chunk_cap);
  const size_t o_Hd = P.take(8 * (size_t)dcap * dcap);
  for (int b = 0; b < 2; ++b) { o_gd[b] = P.take(8 * dcap); o_Ed[b] = P.take(8 * dcap); }
  const size_t o_ud = P.take(8 * dcap), o_scd = P.take(8 * dcap), o_chol = P.take(8 * (size_t)(dcap + 1) * (dcap + 1));
  const size_t o_obsz = P.take(sizeof(double2) * (size_t)Lc * NSc), o_obsw = P.take(8 * (size_t)Lc * NSc), o_M = P.take(8 * 6 * (size_t)Lpc * Kc);
  const size_t o_quality = P.take(8 * (size_t)Lc);
  const size_t o_cache = P.take(sizeof(ImuCache) * std::max(q.T, 1)), o_imu_out = P.take(8 * kImuOut * std::max(q.T, 1));

  if (S.arena_bytes < P.total) {
    if (S.arena) cudaFree(S.arena);
    S.arena = nullptr; S.arena_bytes = 0;
    OKB_CUDA(c, cudaMalloc(&S.arena, P.total));
    S.arena_bytes = P.total;
  }
  const size_t out_bytes = 8 * (16 * (size_t)Kc + 4 + 5 * (size_t)Lc);
  if (S.out_bytes < out_bytes) {
    if (S.out_staging) cudaFreeHost(S.out_staging);
    S.out_staging = nullptr; S.out_bytes = 0;
    OKB_CUDA(c, cudaMallocHost(&S.out_staging, out_bytes));
    S.out_bytes = out_bytes;
  }
  if (!S.down) OKB_CUDA(c, cudaEventCreateWithFlags(&S.down, cudaEventDisableTiming));
  if (!S.copied) OKB_CUDA(c, cudaEventCreateWithFlags(&S.copied, cudaEventDisableTiming));
  // the m_mark scratch must be all zero between commands; dead landmark slots must hold finite values
  OKB_CUDA(c, cudaMemsetAsync(S.arena + o_mark, 0, Lpc, c->stream_xfer));
  OKB_CUDA(c, cudaMemsetAsync(S.arena + o_mlm, 0, 8 * 4 * (size_t)Lpc, c->stream_xfer));
  S.caps = q;
  S.cmd_cap_dev = cmd_cap;

  unsigned char* A = S.arena;
  WinDev W;
  std::memset(&W, 0, sizeof W);
  auto dp = [&](size_t o) { return reinterpret_cast<double*>(A + o); };
  auto up = [&](size_t o) { return reinterpret_cast<uint32_t*>(A + o); };
  W.Kcap = q.K; W.Lcap = q.L; W.Ocap = q.O; W.Scap = q.S; W.Tcap = q.T; W.NEcap = q.NE; W.NCcap = q.NC; W.PPcap = q.PP;
  W.pose = dp(o_pose); W.sb = dp(o_sb); W.ext = dp(o_ext); W.m_lm = dp(o_mlm); W.out = dp(o_out);
  W.cams = reinterpret_cast<okb_camera*>(A + o_cams);
  W.m_obs = reinterpret_cast<okb_observation*>(A + o_obs);
  W.imu_terms = reinterpret_cast<okb_imu_term*>(A + o_imut);
  W.samples = reinterpret_cast<okb_imu_sample*>(A + o_samp);
  W.pp = reinterpret_cast<okb_pose_prior*>(A + o_pp);
  W.sbp = reinterpret_cast<okb_sb_prior*>(A + o_sbp);
  W.marg_kind = reinterpret_cast<int32_t*>(A + o_mkind); W.marg_idx = up(o_midx);
  W.marg_col = reinterpret_cast<int32_t*>(A + o_mcol); W.marg_off = reinterpret_cast<int32_t*>(A + o_moff);
  W.marg_x0 = dp(o_mx0); W.marg_J = dp(o_mJ); W.marg_e0 = dp(o_me0); W.marg_H0 = dp(o_mH0); W.marg_Hs = dp(o_mHs); W.marg_b0 = dp(o_mb0);
  W.m_lm_init = dp(o_mlmi); W.m_mark = A + o_mark; W.m_vis = up(o_mvis); W.m_bitmap = up(o_bitmap);
  W.perm = up(o_perm); W.lm_inv = up(o_inv); W.tile_range = up(o_trange); W.lm_vis = up(o_vis);
  W.slots = reinterpret_cast<SlotInfo*>(A + o_slots);
  W.cmd = A + o_cmd;
  W.lm = dp(o_lm); W.pose_init = dp(o_pose_i); W.sb_init = dp(o_sb_i);
  W.pose_c = dp(o_pose_c); W.sb_c = dp(o_sb_c); W.lm_c = dp(o_lm_c);
  for (int b = 0; b < 2; ++b) { W.lm_g[b] = dp(o_lmg[b]); W.lm_E[b] = dp(o_lmE[b]); W.gd[b] = dp(o_gd[b]); W.Ed[b] = dp(o_Ed[b]); }
  W.lm_Rinv = dp(o_Rinv); W.slot_ctx = reinterpret_cast<SlotCtx*>(A + o_slotctx); W.lm_mf = dp(o_mf); W.lm_gn = dp(o_gn);
  W.lm_Li = dp(o_Li); W.lm_scale = dp(o_scale); W.partH = dp(o_partH); W.partA = dp(o_part);
  W.Hd = dp(o_Hd); W.ud = dp(o_ud); W.scale_d = dp(o_scd); W.chol = dp(o_chol);
  W.obs_z = reinterpret_cast<double2*>(A + o_obsz); W.obs_w = dp(o_obsw); W.lm_M = dp(o_M); W.quality = dp(o_quality);
  W.zero_ptr[0] = A + o_obsz; W.zero_ptr[1] = A + o_obsw; W.zero_ptr[2] = A + o_M;
  W.imu_cache = reinterpret_cast<ImuCache*>(A + o_cache); W.imu_out = dp(o_imu_out);
  W.st = c->d_states + win;
  W.n_chunks = 1; W.use_cauchy = 1;
  c->host[win] = W;
  return OKB_OK;
}

// ---- command staging (pinned, per slot)
int cmd_reserve(okb_ctx* c, WinStore& S, size_t extra) {
  if (S.staging_busy) {          // the previous commit's H2D copy reads the buffer: wait before it is rewritten
    OKB_CUDA(c, cudaEventSynchronize(S.copied));
    S.staging_busy = false;
  }
  const size_t need = S.cmd_used + extra;
  if (need <= S.staging_bytes) return OKB_OK;
  const size_t cap = align_up(std::max(need, 2 * S.staging_bytes), 4096);
  unsigned char* nb = nullptr;
  OKB_CUDA(c, cudaMallocHost(&nb, cap));
  if (S.cmd_used) std::memcpy(nb, S.staging, S.cmd_used);
  if (S.staging) cudaFreeHost(S.staging);
  S.staging = nb; S.staging_bytes = cap;
  return OKB_OK;
}
// Appends a command header and returns the payload pointer (8-byte aligned); payload_bytes is rounded up to 8.
unsigned char* cmd_put(WinStore& S, uint32_t op, uint32_t n, uint32_t a, uint32_t b, size_t payload_bytes) {
  payload_bytes = align_up(payload_bytes, 8);
  CmdHeader h{op, n, a, b, payload_bytes};
  std::memcpy(S.staging + S.cmd_used, &h, sizeof h);
  unsigned char* pay = S.staging + S.cmd_used + sizeof h;
  S.cmd_used += sizeof h + payload_bytes;
  return pay;
}
}  // namespace

static const char* graph_error_text(int e) {
  switch (e) {
    case GERR_INDEX: return "window graph: index out of range";
    case GERR_DUPLICATE: return "window graph: duplicate observation of a landmark in one (frame,camera)";
    case GERR_SLOT_EXT: return "window graph: inconsistent extrinsics block for a (frame,camera) slot";
    case GERR_CAPACITY: return "window graph: capacity exceeded (okb_window_reserve)";
    case GERR_SQRT_INFO: return "window graph: observation with non-positive sqrt information";
    case GERR_DIMS: return "window graph: host / device dimension mismatch";
    case GERR_MARG_REF: return "window graph: a removed frame is still referenced by the marginalisation prior";
    default: return "window graph: unknown error";
  }
}
static int graph_error_status(int e) {
  return e == GERR_DUPLICATE ? OKB_ERR_UNSUPPORTED : e == GERR_CAPACITY ? OKB_ERR_CAPACITY : OKB_ERR_INVALID_ARG;
}

extern "C" int okb_window_reserve(okb_ctx* c, int win, int max_frames, int max_landmarks, int max_observations, int max_imu_samples,
                                  int max_marg_dim) {
  if (!c || win < 0 || win >= c->max_windows || max_frames < 0 || max_landmarks < 0 || max_observations < 0 || max_imu_samples < 0 ||
      max_marg_dim < 0) return OKB_ERR_INVALID_ARG;
  if (max_frames > kMaxFrames || max_marg_dim > kMaxMarg) { c->set_error("okb_window_reserve: beyond the compiled-in limits"); return OKB_ERR_CAPACITY; }
  WinCaps& r = c->wins[win].reserve;
  r.K = max_frames; r.L = max_landmarks; r.O = max_observations; r.S = max_imu_samples; r.T = max_frames; r.MN = max_marg_dim;
  r.PP = std::max(r.PP, 4);
  return OKB_OK;
}

// Commits the pending commands of slots [first, first+count): H2D copies + interpreter + compile on the transfer stream.
static int commit_range(okb_ctx* c, int first, int count) {
  cudaSetDevice(c->device);
  cudaStream_t xs = c->stream_xfer;
  bool any = false;
  int max_work = 1;
  for (int i = first; i < first + count; ++i) {
    WinStore& S = c->wins[i];
    WinDev& W = c->host[i];
    W.cmd_bytes = 0; W.dirty = 0; W.full = 0;
    if (!S.cmd_used) continue;
    if (S.cmd_used > S.cmd_cap_dev) { c->set_error("pending window commands exceed the device command buffer (commit more often)"); return OKB_ERR_CAPACITY; }
    any = true;
    if (S.done_idx >= 0) OKB_CUDA(c, cudaStreamWaitEvent(xs, c->done_ring[S.done_idx], 0));   // solver work on this slot finishes first
    OKB_CUDA(c, cudaMemcpyAsync(const_cast<unsigned char*>(W.cmd), S.staging, S.cmd_used, cudaMemcpyHostToDevice, xs));
    OKB_CUDA(c, cudaEventRecord(S.copied, xs));
    S.staging_busy = true;
    S.h2d_bytes = S.cmd_used;
    W.cmd_bytes = (int)S.cmd_used; W.dirty = 1; W.full = S.full_pending ? 1 : 0;
    W.n_obs = S.obs_bound;
    S.cmd_used = 0; S.full_pending = false; S.committed = true;
    max_work = std::max(max_work, std::max(std::max(W.n_obs, 4 * W.L), std::max(7 * W.K, 9 * W.NSB)));
  }
  if (!any) return OKB_OK;
  OKB_CUDA(c, cudaMemcpyAsync(c->d_wins + first, &c->host[first], sizeof(WinDev) * count, cudaMemcpyHostToDevice, xs));
  const int gx = std::max(1, std::min((max_work + 255) / 256, std::max(4, (8 * c->sm_count + count - 1) / count)));
  k_apply_commands<<<count, 1024, 0, xs>>>(c->d_wins, first);
  k_compile_obs<<<count, 1024, 0, xs>>>(c->d_wins, first);
  k_compile_sort<<<count, 1024, 0, xs>>>(c->d_wins, first);
  k_zero<<<dim3(gx, count), 256, 0, xs>>>(c->d_wins, first);
  k_prepare<<<dim3(gx, count), 256, 0, xs>>>(c->d_wins, first);
  c->launches += 5;
  OKB_CUDA(c, cudaGetLastError());
  for (int i = first; i < first + count; ++i) { c->host[i].cmd_bytes = 0; c->host[i].dirty = 0; c->host[i].full = 0; }
  return OKB_OK;
}

extern "C" int okb_window_commit(okb_ctx* c, int first, int count) {
  if (!c || first < 0 || count < 1 || first + count > c->max_windows) return OKB_ERR_INVALID_ARG;
  return commit_range(c, first, count);
}

// Full upload = a command stream that rebuilds the whole graph (host side: validation of what only the host can
// reject synchronously + one pass of memcpy into the pinned command buffer; sorting / slot tables / duplicate
// detection happen on the device).
static int upload_pack(okb_ctx* c, int win, const okb_window_desc* D) {
  if (!c || !D || win < 0 || win >= c->max_windows) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  const int K = D->n_poses, NSB = D->n_speed_bias, NE = D->n_extrinsics, L = D->n_landmarks, NC = D->n_cameras;
  if (K < 1 || L < 1 || NC < 1 || NE < 1) { c->set_error("empty window"); return OKB_ERR_INVALID_ARG; }
  if (K > kMaxFrames || NSB > kMaxFrames) { c->set_error("more than 32 frames per window"); return OKB_ERR_CAPACITY; }
  for (int e = 0; e < NE; ++e)
    if (!D->extrinsics_fixed || !D->extrinsics_fixed[e]) {
      c->set_error("device solver requires fixed extrinsics (sigma_absolute_* = 0 as in the shipped configs)");
      return OKB_ERR_UNSUPPORTED;
    }
  if (D->n_relpose_terms > 0) { c->set_error("relative-pose terms need free extrinsics"); return OKB_ERR_UNSUPPORTED; }
  if (NC > 32) { c->set_error("more than 32 cameras"); return OKB_ERR_CAPACITY; }
  if (6 * K + 9 * NSB > kMaxDense) { c->set_error("reduced system too large"); return OKB_ERR_CAPACITY; }
  int marg_n = 0, marg_nb = 0, marg_xdim = 0;
  if (D->marg && D->marg->n > 0) {
    marg_n = D->marg->n; marg_nb = D->marg->n_blocks;
    if (marg_n > kMaxMarg || marg_nb > kMaxMargBlocks) { c->set_error("marginalisation prior too large"); return OKB_ERR_CAPACITY; }
    int col = 0;
    for (int b = 0; b < marg_nb; ++b) {
      const int kind = D->marg->block_kind[b];
      const uint32_t idx = D->marg->block_idx[b];
      const int lim = kind == OKB_BLOCK_POSE ? K : kind == OKB_BLOCK_SPEED_BIAS ? NSB : kind == OKB_BLOCK_EXTRINSICS ? NE : -1;
      if (lim < 0) { c->set_error("marginalisation prior: unknown block kind"); return OKB_ERR_INVALID_ARG; }
      if ((int)idx >= lim) { c->set_error("marginalisation prior: block index out of range"); return OKB_ERR_INVALID_ARG; }
      if (kind != OKB_BLOCK_EXTRINSICS) col += (kind == OKB_BLOCK_SPEED_BIAS) ? 9 : 6;
      marg_xdim += (kind == OKB_BLOCK_SPEED_BIAS) ? 9 : 7;
    }
    if (col != marg_n) { c->set_error("marginalisation prior dimension mismatch"); return OKB_ERR_INVALID_ARG; }
  }
  for (int i = 0; i < D->n_pose_priors; ++i)
    if ((int)D->pose_priors[i].pose_idx >= K) { c->set_error("pose prior index out of range"); return OKB_ERR_INVALID_ARG; }
  for (int i = 0; i < D->n_sb_priors; ++i)
    if ((int)D->sb_priors[i].sb_idx >= NSB) { c->set_error("speed/bias prior index out of range"); return OKB_ERR_INVALID_ARG; }
  for (int t = 0; t < D->n_imu_terms; ++t) {
    const okb_imu_term& T = D->imu_terms[t];
    if ((int)T.pose0 >= K || (int)T.pose1 >= K || (int)T.sb0 >= NSB || (int)T.sb1 >= NSB ||
        (uint64_t)T.sample_offset + (uint64_t)T.sample_count > (uint64_t)D->n_imu_samples || T.sample_count < 2) {
      c->set_error("IMU term index out of range");
      return OKB_ERR_INVALID_ARG;
    }
  }
  for (int i = 0; i < D->n_obs; ++i) {
    const okb_observation& ob = D->obs[i];
    if ((int)ob.pose_idx >= K || (int)ob.lm_idx >= L || (int)ob.ext_idx >= NE || (int)ob.cam_idx >= NC) {
      c->set_error("observation index out of range");
      return OKB_ERR_INVALID_ARG;
    }
    if (!(ob.sqrt_info > 0.0)) { c->set_error("observation with non-positive sqrt information"); return OKB_ERR_INVALID_ARG; }
  }
  if (smemA2_bytes(K, 0) > (size_t)c->smem_optin) { c->set_error("window does not fit kernel A shared memory"); return OKB_ERR_CAPACITY; }

  WinStore& S = c->wins[win];
  S.uploaded = false;        // true again only when the whole upload has been issued successfully
  WinCaps need{K, L, D->n_obs, D->n_imu_samples, D->n_imu_terms, NE, NC, std::max(D->n_pose_priors, D->n_sb_priors), marg_n};
  need = caps_max(need, S.reserve);
  need.T = std::max(need.T, need.K);
  if (!S.arena || !caps_cover(S.caps, need)) {
    if (S.done_idx >= 0) OKB_CUDA(c, cudaEventSynchronize(c->done_ring[S.done_idx]));    // the old arena may still be in use
    int rc = plan_arena(c, win, S.arena ? caps_max(S.caps, need) : need);
    if (rc) return rc;
  }
  S.cmd_used = 0;            // a full upload supersedes anything still pending
  int rc = cmd_reserve(c, S, full_upload_bytes(need));
  if (rc) return rc;
  unsigned char* q;
  q = cmd_put(S, CMD_RESET_GRAPH, 0, (uint32_t)NE, (uint32_t)NC, 8 * 7 * (size_t)NE + sizeof(okb_camera) * NC);
  std::memcpy(q, D->extrinsics, 8 * 7 * (size_t)NE);
  std::memcpy(q + 8 * 7 * (size_t)NE, D->cameras, sizeof(okb_camera) * NC);
  q = cmd_put(S, CMD_SET_FRAMES, 0, (uint32_t)K, (uint32_t)NSB, 8 * (7 * (size_t)K + 9 * (size_t)NSB));
  std::memcpy(q, D->poses, 8 * 7 * (size_t)K);
  if (NSB) std::memcpy(q + 8 * 7 * (size_t)K, D->speed_bias, 8 * 9 * (size_t)NSB);
  q = cmd_put(S, CMD_SET_LANDMARKS, (uint32_t)L, 0, 1, 8 * 4 * (size_t)L);
  std::memcpy(q, D->landmarks, 8 * 4 * (size_t)L);
  if (D->n_obs) {
    q = cmd_put(S, CMD_ADD_OBS, (uint32_t)D->n_obs, 0, 0, sizeof(okb_observation) * (size_t)D->n_obs);
    std::memcpy(q, D->obs, sizeof(okb_observation) * (size_t)D->n_obs);
  }
  q = cmd_put(S, CMD_SET_IMU, 0, (uint32_t)D->n_imu_terms, (uint32_t)D->n_imu_samples,
              sizeof(okb_imu_term) * D->n_imu_terms + sizeof(okb_imu_sample) * (size_t)D->n_imu_samples);
  if (D->n_imu_terms) std::memcpy(q, D->imu_terms, sizeof(okb_imu_term) * D->n_imu_terms);
  if (D->n_imu_samples) std::memcpy(q + sizeof(okb_imu_term) * D->n_imu_terms, D->imu_samples, sizeof(okb_imu_sample) * (size_t)D->n_imu_samples);
  q = cmd_put(S, CMD_SET_POSE_PRIORS, (uint32_t)D->n_pose_priors, 0, 0, sizeof(okb_pose_prior) * D->n_pose_priors);
  if (D->n_pose_priors) std::memcpy(q, D->pose_priors, sizeof(okb_pose_prior) * D->n_pose_priors);
  q = cmd_put(S, CMD_SET_SB_PRIORS, (uint32_t)D->n_sb_priors, 0, 0, sizeof(okb_sb_prior) * D->n_sb_priors);
  if (D->n_sb_priors) std::memcpy(q, D->sb_priors, sizeof(okb_sb_prior) * D->n_sb_priors);
  if (marg_n) {
    const size_t kb = align_up(4 * (size_t)marg_nb, 8);
    q = cmd_put(S, CMD_SET_MARG, 0, (uint32_t)marg_n, (uint32_t)marg_nb, 2 * kb + 8 * ((size_t)marg_xdim + (size_t)marg_n * marg_n + marg_n));
    std::memset(q, 0, 2 * kb);
    std::memcpy(q, D->marg->block_kind, 4 * (size_t)marg_nb);
    std::memcpy(q + kb, D->marg->block_idx, 4 * (size_t)marg_nb);
    double* x = reinterpret_cast<double*>(q + 2 * kb);
    std::memcpy(x, D->marg->x0, 8 * (size_t)marg_xdim);
    std::memcpy(x + marg_xdim, D->marg->J, 8 * (size_t)marg_n * marg_n);
    std::memcpy(x + marg_xdim + (size_t)marg_n * marg_n, D->marg->e0, 8 * (size_t)marg_n);
  }
  // host mirror of the dimensions
  WinDev& W = c->host[win];
  W.K = K; W.NSB = NSB; W.NE = NE; W.L = L; W.NC = NC;
  W.n_imu = D->n_imu_terms; W.n_samples = D->n_imu_samples; W.n_pp = D->n_pose_priors; W.n_sbp = D->n_sb_priors;
  W.marg_n = marg_n; W.marg_nb = marg_nb; W.marg_xdim = marg_xdim;
  W.imu_params = D->imu_params;
  derive_dims(W);
  W.shard_rank = c->shard_rank; W.shard_world = c->shard_world; W.shard_box_cap = c->shard_box_cap;
  if (c->shard_world > 1) {
    if (shard_box_doubles(K, W.dcp) > (size_t)c->shard_box_cap) { c->set_error("window exceeds the shard mailbox (max_frames of okb_shard_export)"); return OKB_ERR_CAPACITY; }
    for (int r = 0; r < c->shard_world; ++r) {
      if (!c->shard_peer[r]) { c->set_error("landmark sharding: okb_shard_connect has not been called"); return OKB_ERR_INVALID_ARG; }
      W.shard_mail[r] = c->shard_peer[r] + (size_t)win * c->shard_win_bytes;
    }
  }
  S.terms.assign(D->imu_terms, D->imu_terms + D->n_imu_terms);
  S.pp_idx.clear(); S.sbp_idx.clear();
  for (int i = 0; i < D->n_pose_priors; ++i) S.pp_idx.push_back(D->pose_priors[i].pose_idx);
  for (int i = 0; i < D->n_sb_priors; ++i) S.sbp_idx.push_back(D->sb_priors[i].sb_idx);
  S.obs_bound = D->n_obs;
  S.full_pending = true;
  S.K_init = K; S.NSB_init = NSB; S.L_init = L;
  S.uploaded = true;
  return OKB_OK;
}

extern "C" int okb_window_upload(okb_ctx* c, int win, const okb_window_desc* D) {
  int rc = upload_pack(c, win, D);
  if (rc) return rc;
  return commit_range(c, win, 1);
}

extern "C" int okb_window_upload_batch(okb_ctx* c, int first, int count, const okb_window_desc* descs, int host_threads) {
  if (!c || !descs || count < 1 || first < 0 || first + count > c->max_windows) return OKB_ERR_INVALID_ARG;
  int T = host_threads > 0 ? host_threads : 8;
  T = std::max(1, std::min(T, count));
  std::vector<int> rcs(T, OKB_OK);
  if (T == 1) {
    for (int i = 0; i < count && !rcs[0]; ++i) rcs[0] = upload_pack(c, first + i, descs + i);
  } else {
    std::vector<std::thread> th;
    th.reserve(T);
    for (int t = 0; t < T; ++t)
      th.emplace_back([=, &rcs]() {
        for (int i = t; i < count; i += T) {
          const int rc = upload_pack(c, first + i, descs + i);
          if (rc) { rcs[t] = rc; return; }
        }
      });
    for (auto& x : th) x.join();
  }
  for (int t = 0; t < T; ++t)
    if (rcs[t]) return rcs[t];
  return commit_range(c, first, count);
}

// ---------------------------------------------------------------------------------------------
// incremental graph updates (Estimator::addStates / addLandmark / addObservation / removeObservation / set_*,
// okvis_ceres/src/Estimator.cpp:110-413, implementation/Estimator.hpp:43-90): commands appended to the slot's
// pending stream; nothing touches the device until okb_window_commit / okb_optimize*.
// ---------------------------------------------------------------------------------------------
static int delta_begin(okb_ctx* c, int win, size_t extra, WinStore** S, WinDev** W) {
  if (!c || win < 0 || win >= c->max_windows) return OKB_ERR_INVALID_ARG;
  if (!c->wins[win].uploaded) { c->set_error("window slot not uploaded"); return OKB_ERR_INVALID_ARG; }
  cudaSetDevice(c->device);
  *S = &c->wins[win];
  *W = &c->host[win];
  return cmd_reserve(c, **S, extra + sizeof(CmdHeader) + 64);
}

extern "C" int okb_window_add_frame(okb_ctx* c, int win, const double* pose, const double* speed_bias, const okb_imu_term* term,
                                    const okb_imu_sample* samples, int n_samples) {
  WinStore* S; WinDev* W;
  if (!pose || (term && (!samples || n_samples < 2))) return OKB_ERR_INVALID_ARG;
  int rc = delta_begin(c, win, 16 * 8 + sizeof(okb_imu_term) + sizeof(okb_imu_sample) * (size_t)std::max(n_samples, 0) + sizeof(CmdHeader), &S, &W);
  if (rc) return rc;
  const int K1 = W->K + 1, NSB1 = W->NSB + (speed_bias ? 1 : 0);
  if (K1 > S->caps.K || NSB1 > S->caps.K || 6 * K1 + 9 * NSB1 > kMaxDense) { c->set_error("okb_window_add_frame: frame capacity exceeded (okb_window_reserve)"); return OKB_ERR_CAPACITY; }
  if (smemA2_bytes(K1, 0) > (size_t)c->smem_optin) { c->set_error("window does not fit kernel A shared memory"); return OKB_ERR_CAPACITY; }
  if (term) {
    if ((int)term->pose0 >= K1 || (int)term->pose1 >= K1 || (int)term->sb0 >= NSB1 || (int)term->sb1 >= NSB1 ||
        (uint64_t)term->sample_offset + term->sample_count > (uint64_t)n_samples || term->sample_count < 2) {
      c->set_error("IMU term index out of range");
      return OKB_ERR_INVALID_ARG;
    }
    if (W->n_imu + 1 > S->caps.T || W->n_samples + n_samples > S->caps.S) { c->set_error("okb_window_add_frame: IMU capacity exceeded (okb_window_reserve)"); return OKB_ERR_CAPACITY; }
  }
  if (c->shard_world > 1 && shard_box_doubles(K1, 4 * ((6 * K1 + 1 + 3) / 4)) > (size_t)c->shard_box_cap) { c->set_error("window exceeds the shard mailbox"); return OKB_ERR_CAPACITY; }
  unsigned char* q = cmd_put(*S, CMD_ADD_FRAME, 0, 0, speed_bias ? 1u : 0u, 8 * 16);
  std::memcpy(q, pose, 56);
  if (speed_bias) std::memcpy(q + 56, speed_bias, 72); else std::memset(q + 56, 0, 72);
  W->K = K1; W->NSB = NSB1;
  if (term) {
    q = cmd_put(*S, CMD_ADD_IMU_TERM, (uint32_t)n_samples, 0, 0, sizeof(okb_imu_term) + sizeof(okb_imu_sample) * (size_t)n_samples);
    std::memcpy(q, term, sizeof(okb_imu_term));
    std::memcpy(q + sizeof(okb_imu_term), samples, sizeof(okb_imu_sample) * (size_t)n_samples);
    okb_imu_term mirror = *term;
    mirror.sample_offset += (uint32_t)W->n_samples;
    S->terms.push_back(mirror);
    W->n_imu += 1; W->n_samples += n_samples;
  }
  derive_dims(*W);
  return OKB_OK;
}

extern "C" int okb_window_remove_frame(okb_ctx* c, int win, uint32_t pose_idx, uint32_t sb_idx) {
  WinStore* S; WinDev* W;
  int rc = delta_begin(c, win, 0, &S, &W);
  if (rc) return rc;
  const bool has_sb = sb_idx != 0xffffffffu;
  if ((int)pose_idx >= W->K || (has_sb && (int)sb_idx >= W->NSB) || W->K < 2) { c->set_error("okb_window_remove_frame: index out of range"); return OKB_ERR_INVALID_ARG; }
  // the host mirror of the IMU term / prior counts needs the terms that touch the frame: it keeps a light copy
  cmd_put(*S, CMD_REMOVE_FRAME, 0, pose_idx, sb_idx, 0);
  int kept = 0, s_lo = 0x7fffffff, s_hi = 0;
  for (auto& T : S->terms) {
    const bool drop = T.pose0 == pose_idx || T.pose1 == pose_idx || (has_sb && (T.sb0 == sb_idx || T.sb1 == sb_idx));
    if (drop) continue;
    if (T.pose0 > pose_idx) T.pose0--;
    if (T.pose1 > pose_idx) T.pose1--;
    if (has_sb && T.sb0 > sb_idx) T.sb0--;
    if (has_sb && T.sb1 > sb_idx) T.sb1--;
    s_lo = std::min(s_lo, (int)T.sample_offset); s_hi = std::max(s_hi, (int)(T.sample_offset + T.sample_count));
    S->terms[kept++] = T;
  }
  S->terms.resize(kept);
  if (!kept) { s_lo = 0; s_hi = 0; }
  for (auto& T : S->terms) T.sample_offset -= (uint32_t)s_lo;
  W->n_imu = kept; W->n_samples = s_hi - s_lo;
  auto drop_priors = [](std::vector<uint32_t>& v, uint32_t idx) {
    size_t o = 0;
    for (size_t i = 0; i < v.size(); ++i) { if (v[i] == idx) continue; v[o++] = v[i] > idx ? v[i] - 1 : v[i]; }
    v.resize(o);
  };
  drop_priors(S->pp_idx, pose_idx);
  if (has_sb) drop_priors(S->sbp_idx, sb_idx);
  W->n_pp = (int)S->pp_idx.size(); W->n_sbp = (int)S->sbp_idx.size();
  W->K -= 1;
  if (has_sb) W->NSB -= 1;
  derive_dims(*W);
  return OKB_OK;
}

extern "C" int okb_window_set_landmarks(okb_ctx* c, int win, int n, const uint32_t* idx, const double* xyzw) {
  WinStore* S; WinDev* W;
  if (n < 1 || !idx || !xyzw) return OKB_ERR_INVALID_ARG;
  int rc = delta_begin(c, win, align_up(4 * (size_t)n, 8) + 32 * (size_t)n, &S, &W);
  if (rc) return rc;
  int L = W->L;
  for (int i = 0; i < n; ++i) {
    if ((int)idx[i] >= S->caps.L) { c->set_error("okb_window_set_landmarks: landmark capacity exceeded (okb_window_reserve)"); return OKB_ERR_CAPACITY; }
    L = std::max(L, (int)idx[i] + 1);
  }
  const size_t ib = align_up(4 * (size_t)n, 8);
  unsigned char* q = cmd_put(*S, CMD_SET_LANDMARKS, (uint32_t)n, 0, 0, ib + 32 * (size_t)n);
  std::memset(q, 0, ib);
  std::memcpy(q, idx, 4 * (size_t)n);
  std::memcpy(q + ib, xyzw, 32 * (size_t)n);
  W->L = L;
  derive_dims(*W);
  return OKB_OK;
}

extern "C" int okb_window_remove_landmarks(okb_ctx* c, int win, int n, const uint32_t* idx) {
  WinStore* S; WinDev* W;
  if (n < 1 || !idx) return OKB_ERR_INVALID_ARG;
  int rc = delta_begin(c, win, 4 * (size_t)n + 8, &S, &W);
  if (rc) return rc;
  for (int i = 0; i < n; ++i)
    if ((int)idx[i] >= W->L) { c->set_error("okb_window_remove_landmarks: index out of range"); return OKB_ERR_INVALID_ARG; }
  unsigned char* q = cmd_put(*S, CMD_REMOVE_LANDMARKS, (uint32_t)n, 0, 0, 4 * (size_t)n);
  std::memcpy(q, idx, 4 * (size_t)n);
  return OKB_OK;
}

extern "C" int okb_window_add_observations(okb_ctx* c, int win, int n, const okb_observation* obs) {
  WinStore* S; WinDev* W;
  if (n < 1 || !obs) return OKB_ERR_INVALID_ARG;
  int rc = delta_begin(c, win, sizeof(okb_observation) * (size_t)n, &S, &W);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    const okb_observation& ob = obs[i];
    if ((int)ob.pose_idx >= W->K || (int)ob.lm_idx >= W->L || (int)ob.ext_idx >= W->NE || (int)ob.cam_idx >= W->NC) { c->set_error("observation index out of range"); return OKB_ERR_INVALID_ARG; }
    if (!(ob.sqrt_info > 0.0)) { c->set_error("observation with non-positive sqrt information"); return OKB_ERR_INVALID_ARG; }
  }
  if (S->obs_bound + n > S->caps.O) { c->set_error("okb_window_add_observations: observation capacity exceeded (okb_window_reserve)"); return OKB_ERR_CAPACITY; }
  unsigned char* q = cmd_put(*S, CMD_ADD_OBS, (uint32_t)n, 0, 0, sizeof(okb_observation) * (size_t)n);
  std::memcpy(q, obs, sizeof(okb_observation) * (size_t)n);
  S->obs_bound += n;
  return OKB_OK;
}

extern "C" int okb_window_remove_observations(okb_ctx* c, int win, int n, const okb_obs_key* keys) {
  WinStore* S; WinDev* W;
  if (n < 1 || !keys) return OKB_ERR_INVALID_ARG;
  int rc = delta_begin(c, win, sizeof(okb_obs_key) * (size_t)n, &S, &W);
  if (rc) return rc;
  for (int i = 0; i < n; ++i)
    if ((int)keys[i].pose_idx >= W->K || (int)keys[i].lm_idx >= W->L || (int)keys[i].cam_idx >= W->NC) { c->set_error("observation key out of range"); return OKB_ERR_INVALID_ARG; }
  unsigned char* q = cmd_put(*S, CMD_REMOVE_OBS, (uint32_t)n, 0, 0, sizeof(okb_obs_key) * (size_t)n);
  std::memcpy(q, keys, sizeof(okb_obs_key) * (size_t)n);
  return OKB_OK;
}

extern "C" int okb_window_set_states(okb_ctx* c, int win, int n_poses, const uint32_t* pose_idx, const double* poses, int n_sb,
                                     const uint32_t* sb_idx, const double* speed_bias) {
  WinStore* S; WinDev* W;
  if (n_poses < 0 || n_sb < 0 || (n_poses && (!pose_idx || !poses)) || (n_sb && (!sb_idx || !speed_bias))) return OKB_ERR_INVALID_ARG;
  int rc = delta_begin(c, win, (sizeof(CmdHeader) + 72) * (size_t)(n_poses + n_sb), &S, &W);
  if (rc) return rc;
  for (int i = 0; i < n_poses; ++i) if ((int)pose_idx[i] >= W->K) { c->set_error("okb_window_set_states: pose index out of range"); return OKB_ERR_INVALID_ARG; }
  for (int i = 0; i < n_sb; ++i) if ((int)sb_idx[i] >= W->NSB) { c->set_error("okb_window_set_states: speed/bias index out of range"); return OKB_ERR_INVALID_ARG; }
  for (int i = 0; i < n_poses; ++i) std::memcpy(cmd_put(*S, CMD_SET_POSE, 0, pose_idx[i], 0, 56), poses + 7 * (size_t)i, 56);
  for (int i = 0; i < n_sb; ++i) std::memcpy(cmd_put(*S, CMD_SET_SB, 0, sb_idx[i], 0, 72), speed_bias + 9 * (size_t)i, 72);
  return OKB_OK;
}

extern "C" int okb_window_set_priors(okb_ctx* c, int win, int n_pose_priors, const okb_pose_prior* pose_priors, int n_sb_priors,
                                     const okb_sb_prior* sb_priors, const okb_marg_prior* marg) {
  WinStore* S; WinDev* W;
  if (n_pose_priors < 0 || n_sb_priors < 0) return OKB_ERR_INVALID_ARG;
  const int mn = marg ? marg->n : 0, mnb = marg ? marg->n_blocks : 0;
  int rc = delta_begin(c, win, sizeof(okb_pose_prior) * (size_t)n_pose_priors + sizeof(okb_sb_prior) * (size_t)n_sb_priors + 3 * sizeof(CmdHeader) +
                                   8 * ((size_t)mn * mn + mn + 11 * (size_t)mnb + 8), &S, &W);
  if (rc) return rc;
  if (n_pose_priors > S->caps.PP || n_sb_priors > S->caps.PP) { c->set_error("okb_window_set_priors: more priors than reserved"); return OKB_ERR_CAPACITY; }
  for (int i = 0; i < n_pose_priors; ++i) if ((int)pose_priors[i].pose_idx >= W->K) { c->set_error("pose prior index out of range"); return OKB_ERR_INVALID_ARG; }
  for (int i = 0; i < n_sb_priors; ++i) if ((int)sb_priors[i].sb_idx >= W->NSB) { c->set_error("speed/bias prior index out of range"); return OKB_ERR_INVALID_ARG; }
  int xdim = 0;
  if (marg) {
    if (mn > S->caps.MN || mn > kMaxMarg || mnb > kMaxMargBlocks || mn < 0) { c->set_error("okb_window_set_priors: marginalisation prior larger than reserved"); return OKB_ERR_CAPACITY; }
    int col = 0;
    for (int b = 0; b < mnb; ++b) {
      const int kind = marg->block_kind[b];
      const int lim = kind == OKB_BLOCK_POSE ? W->K : kind == OKB_BLOCK_SPEED_BIAS ? W->NSB : kind == OKB_BLOCK_EXTRINSICS ? W->NE : -1;
      if (lim < 0 || (int)marg->block_idx[b] >= lim) { c->set_error("marginalisation prior: bad block"); return OKB_ERR_INVALID_ARG; }
      if (kind != OKB_BLOCK_EXTRINSICS) col += (kind == OKB_BLOCK_SPEED_BIAS) ? 9 : 6;
      xdim += (kind == OKB_BLOCK_SPEED_BIAS) ? 9 : 7;
    }
    if (col != mn) { c->set_error("marginalisation prior dimension mismatch"); return OKB_ERR_INVALID_ARG; }
  }
  unsigned char* q = cmd_put(*S, CMD_SET_POSE_PRIORS, (uint32_t)n_pose_priors, 0, 0, sizeof(okb_pose_prior) * (size_t)n_pose_priors);
  if (n_pose_priors) std::memcpy(q, pose_priors, sizeof(okb_pose_prior) * (size_t)n_pose_priors);
  q = cmd_put(*S, CMD_SET_SB_PRIORS, (uint32_t)n_sb_priors, 0, 0, sizeof(okb_sb_prior) * (size_t)n_sb_priors);
  if (n_sb_priors) std::memcpy(q, sb_priors, sizeof(okb_sb_prior) * (size_t)n_sb_priors);
  S->pp_idx.clear(); S->sbp_idx.clear();
  for (int i = 0; i < n_pose_priors; ++i) S->pp_idx.push_back(pose_priors[i].pose_idx);
  for (int i = 0; i < n_sb_priors; ++i) S->sbp_idx.push_back(sb_priors[i].sb_idx);
  W->n_pp = n_pose_priors; W->n_sbp = n_sb_priors;
  if (marg) {
    const size_t kb = align_up(4 * (size_t)mnb, 8);
    q = cmd_put(*S, CMD_SET_MARG, 0, (uint32_t)mn, (uint32_t)mnb, 2 * kb + 8 * ((size_t)xdim + (size_t)mn * mn + mn));
    std::memset(q, 0, 2 * kb);
    if (mnb) { std::memcpy(q, marg->block_kind, 4 * (size_t)mnb); std::memcpy(q + kb, marg->block_idx, 4 * (size_t)mnb); }
    double* x = reinterpret_cast<double*>(q + 2 * kb);
    if (xdim) std::memcpy(x, marg->x0, 8 * (size_t)xdim);
    if (mn) { std::memcpy(x + xdim, marg->J, 8 * (size_t)mn * mn); std::memcpy(x + xdim + (size_t)mn * mn, marg->e0, 8 * (size_t)mn); }
    W->marg_n = mn; W->marg_nb = mnb; W->marg_xdim = xdim;
  }
  return OKB_OK;
}

extern "C" int okb_window_remove_speed_bias(okb_ctx* c, int win, uint32_t sb_idx) {
  WinStore* S; WinDev* W;
  int rc = delta_begin(c, win, 0, &S, &W);
  if (rc) return rc;
  if ((int)sb_idx >= W->NSB) { c->set_error("okb_window_remove_speed_bias: index out of range"); return OKB_ERR_INVALID_ARG; }
  cmd_put(*S, CMD_REMOVE_SB, 0, sb_idx, 0, 0);
  int kept = 0, s_lo = 0x7fffffff, s_hi = 0;
  for (auto& T : S->terms) {
    if (T.sb0 == sb_idx || T.sb1 == sb_idx) continue;
    if (T.sb0 > sb_idx) T.sb0--;
    if (T.sb1 > sb_idx) T.sb1--;
    s_lo = std::min(s_lo, (int)T.sample_offset); s_hi = std::max(s_hi, (int)(T.sample_offset + T.sample_count));
    S->terms[kept++] = T;
  }
  S->terms.resize(kept);
  if (!kept) { s_lo = 0; s_hi = 0; }
  for (auto& T : S->terms) T.sample_offset -= (uint32_t)s_lo;
  W->n_imu = kept; W->n_samples = s_hi - s_lo;
  size_t o = 0;
  for (size_t i = 0; i < S->sbp_idx.size(); ++i) { if (S->sbp_idx[i] == sb_idx) continue; S->sbp_idx[o++] = S->sbp_idx[i] > sb_idx ? S->sbp_idx[i] - 1 : S->sbp_idx[i]; }
  S->sbp_idx.resize(o);
  W->n_sbp = (int)o;
  W->NSB -= 1;
  derive_dims(*W);
  return OKB_OK;
}

// ---------------------------------------------------------------------------------------------
// device-side marginalisation (okb_marg.cuh): MarginalizationError::addResidualBlock / marginalizeOut /
// updateErrorComputation (okvis_ceres/src/MarginalizationError.cpp:127-435, 507-846)
// ---------------------------------------------------------------------------------------------
static int hook_alloc_fwd(okb_ctx* c, size_t bytes);
static int check_range(okb_ctx* c, int first, int count);
namespace {
constexpr int kMargImuCap = 32, kMargSbpCap = 8;
struct MargLayout { size_t kind, idx, prev, marg, imu, sbp, lms, payload_end, H, b, A, Q, T, Hn, bn, xlin, lmrec, lmV, lmvis, lmslot, clist, status, total; };
MargLayout marg_layout(int lm_cap, int K_cap, int L_cap, int O_cap) {
  MargLayout m;
  size_t o = sizeof(MargJobHeader);
  auto take = [&](size_t bytes) { const size_t r = o; o = align_up(o + bytes, 16); return r; };
  m.kind = take(4 * kMaxMargBlocks); m.idx = take(4 * kMaxMargBlocks); m.prev = take(4 * kMaxMargBlocks); m.marg = take(kMaxMargBlocks);
  m.imu = take(4 * kMargImuCap); m.sbp = take(4 * kMargSbpCap); m.lms = take(4 * (size_t)lm_cap);
  m.payload_end = o;
  const size_t NN = (size_t)kMargWork * kMargWork * 8;
  m.H = take(NN); m.b = take(8 * kMargWork); m.A = take(NN); m.Q = take(NN); m.T = take(NN); m.Hn = take(NN); m.bn = take(8 * kMargWork);
  m.xlin = take(8 * 9 * kMaxMargBlocks);
  m.lmrec = take(8 * (size_t)lm_cap * K_cap * kMargRec); m.lmV = take(8 * 16 * (size_t)lm_cap); m.lmvis = take(4 * (size_t)lm_cap);
  m.lmslot = take(4 * (size_t)std::max(L_cap, 1)); m.clist = take(4 * (size_t)std::max(O_cap, 1)); m.status = take(16);
  m.total = o;
  return m;
}
MargScratch marg_pointers(unsigned char* base, const MargLayout& m) {
  MargScratch sc;
  sc.hdr = reinterpret_cast<MargJobHeader*>(base);
  sc.kind = reinterpret_cast<int32_t*>(base + m.kind); sc.idx = reinterpret_cast<uint32_t*>(base + m.idx);
  sc.prev = reinterpret_cast<int32_t*>(base + m.prev); sc.marg = base + m.marg;
  sc.imu_terms = reinterpret_cast<uint32_t*>(base + m.imu); sc.sb_priors = reinterpret_cast<uint32_t*>(base + m.sbp);
  sc.landmarks = reinterpret_cast<uint32_t*>(base + m.lms);
  auto dp = [&](size_t o) { return reinterpret_cast<double*>(base + o); };
  sc.H = dp(m.H); sc.b = dp(m.b); sc.A = dp(m.A); sc.Q = dp(m.Q); sc.T = dp(m.T); sc.Hn = dp(m.Hn); sc.bn = dp(m.bn); sc.xlin = dp(m.xlin);
  sc.lmrec = dp(m.lmrec); sc.lmV = dp(m.lmV); sc.lmvis = reinterpret_cast<uint32_t*>(base + m.lmvis);
  sc.lmslot = reinterpret_cast<int32_t*>(base + m.lmslot); sc.clist = reinterpret_cast<int32_t*>(base + m.clist);
  sc.status = reinterpret_cast<int32_t*>(base + m.status);
  return sc;
}
}  // namespace

extern "C" int okb_window_marginalize(okb_ctx* c, int win, const okb_marg_job* job) {
  if (!c || !job || win < 0 || win >= c->max_windows) return OKB_ERR_INVALID_ARG;
  if (!c->wins[win].uploaded) { c->set_error("window slot not uploaded"); return OKB_ERR_INVALID_ARG; }
  cudaSetDevice(c->device);
  int rc = commit_range(c, win, 1);            // pending graph edits first: the job indexes the window as it is now
  if (rc) return rc;
  WinStore& S = c->wins[win];
  WinDev& W = c->host[win];
  if (job->n_blocks < 1 || job->n_blocks > kMaxMargBlocks || job->n_imu_terms < 0 || job->n_imu_terms > kMargImuCap || job->n_sb_priors < 0 ||
      job->n_sb_priors > kMargSbpCap || job->n_landmarks < 0 || !job->block_kind || !job->block_idx || !job->block_prev || !job->block_marginalize) {
    c->set_error("okb_window_marginalize: malformed job");
    return OKB_ERR_INVALID_ARG;
  }
  int N = 0, n_keep = 0, nb_keep = 0, xdim = 0;
  for (int b = 0; b < job->n_blocks; ++b) {
    const int kind = job->block_kind[b];
    if (kind != OKB_BLOCK_POSE && kind != OKB_BLOCK_SPEED_BIAS) { c->set_error("okb_window_marginalize: block kind must be pose or speed/bias (extrinsics are fixed)"); return OKB_ERR_UNSUPPORTED; }
    const int lim = kind == OKB_BLOCK_POSE ? W.K : W.NSB;
    if ((int)job->block_idx[b] >= lim || job->block_prev[b] < -1 || job->block_prev[b] >= W.marg_nb) { c->set_error("okb_window_marginalize: block index out of range"); return OKB_ERR_INVALID_ARG; }
    const int dim = kind == OKB_BLOCK_SPEED_BIAS ? 9 : 6;
    N += dim;
    if (!job->block_marginalize[b]) { n_keep += dim; nb_keep += 1; xdim += (kind == OKB_BLOCK_SPEED_BIAS) ? 9 : 7; }
  }
  for (int i = 0; i < job->n_imu_terms; ++i) if ((int)job->imu_terms[i] >= W.n_imu) { c->set_error("okb_window_marginalize: IMU term index out of range"); return OKB_ERR_INVALID_ARG; }
  for (int i = 0; i < job->n_sb_priors; ++i) if ((int)job->sb_priors[i] >= W.n_sbp) { c->set_error("okb_window_marginalize: prior index out of range"); return OKB_ERR_INVALID_ARG; }
  for (int i = 0; i < job->n_landmarks; ++i) if ((int)job->landmarks[i] >= W.L) { c->set_error("okb_window_marginalize: landmark index out of range"); return OKB_ERR_INVALID_ARG; }
  if (N > kMargWork) { c->set_error("okb_window_marginalize: linear system larger than the compiled-in limit"); return OKB_ERR_CAPACITY; }
  if (n_keep > kMaxMarg || n_keep > S.caps.MN) { c->set_error("okb_window_marginalize: resulting prior larger than reserved (okb_window_reserve max_marg_dim)"); return OKB_ERR_CAPACITY; }
  // scratch
  if (!S.marg_scratch || S.marg_lm_cap < job->n_landmarks || S.marg_K_cap < S.caps.K || S.marg_L_cap < S.caps.L || S.marg_O_cap < S.caps.O) {
    if (S.marg_scratch) { OKB_CUDA(c, cudaStreamSynchronize(c->stream_xfer)); cudaFree(S.marg_scratch); S.marg_scratch = nullptr; }
    S.marg_lm_cap = std::max(256, 2 * job->n_landmarks); S.marg_K_cap = S.caps.K; S.marg_L_cap = S.caps.L; S.marg_O_cap = S.caps.O;
    const MargLayout m = marg_layout(S.marg_lm_cap, S.marg_K_cap, S.marg_L_cap, S.marg_O_cap);
    OKB_CUDA(c, cudaMalloc(&S.marg_scratch, m.total));
    S.marg_scratch_bytes = m.total;
    OKB_CUDA(c, cudaMemsetAsync(S.marg_scratch, 0, m.total, c->stream_xfer));
  }
  const MargLayout m = marg_layout(S.marg_lm_cap, S.marg_K_cap, S.marg_L_cap, S.marg_O_cap);
  rc = cmd_reserve(c, S, m.payload_end);
  if (rc) return rc;
  unsigned char* q = S.staging;
  std::memset(q, 0, m.payload_end);
  MargJobHeader h{job->n_blocks, job->n_imu_terms, job->n_sb_priors, job->n_landmarks, N, n_keep, S.marg_lm_cap, 0};
  std::memcpy(q, &h, sizeof h);
  std::memcpy(q + m.kind, job->block_kind, 4 * (size_t)job->n_blocks);
  std::memcpy(q + m.idx, job->block_idx, 4 * (size_t)job->n_blocks);
  std::memcpy(q + m.prev, job->block_prev, 4 * (size_t)job->n_blocks);
  std::memcpy(q + m.marg, job->block_marginalize, (size_t)job->n_blocks);
  if (job->n_imu_terms) std::memcpy(q + m.imu, job->imu_terms, 4 * (size_t)job->n_imu_terms);
  if (job->n_sb_priors) std::memcpy(q + m.sbp, job->sb_priors, 4 * (size_t)job->n_sb_priors);
  if (job->n_landmarks) std::memcpy(q + m.lms, job->landmarks, 4 * (size_t)job->n_landmarks);
  cudaStream_t xs = c->stream_xfer;
  if (S.done_idx >= 0) OKB_CUDA(c, cudaStreamWaitEvent(xs, c->done_ring[S.done_idx], 0));
  OKB_CUDA(c, cudaMemcpyAsync(S.marg_scratch, q, m.payload_end, cudaMemcpyHostToDevice, xs));
  OKB_CUDA(c, cudaEventRecord(S.copied, xs));
  S.staging_busy = true;
  OKB_CUDA(c, cudaMemsetAsync(S.marg_scratch + m.status, 0, 16, xs));
  OKB_CUDA(c, cudaMemcpyAsync(c->d_wins + win, &W, sizeof(WinDev), cudaMemcpyHostToDevice, xs));
  k_marginalize<<<1, M_THREADS, 0, xs>>>(c->d_wins, win, marg_pointers(S.marg_scratch, m));
  c->launches += 1;
  OKB_CUDA(c, cudaGetLastError());
  W.marg_n = n_keep; W.marg_nb = nb_keep; W.marg_xdim = xdim;
  return OKB_OK;
}

extern "C" int okb_window_download_marg(okb_ctx* c, int win, int32_t* n, int32_t* n_blocks, int32_t* block_kind, uint32_t* block_idx, double* x0,
                                        double* J, double* e0, double* H, double* b0, int32_t* status) {
  int rc = check_range(c, win, 1);
  if (rc) return rc;
  cudaSetDevice(c->device);
  rc = commit_range(c, win, 1);
  if (rc) return rc;
  const int cap = 8 + 2 * kMaxMargBlocks + 9 * kMaxMargBlocks + 2 * kMaxMarg * kMaxMarg + 2 * kMaxMarg;
  rc = hook_alloc_fwd(c, sizeof(double) * cap);
  if (rc) return rc;
  WinStore& S = c->wins[win];
  cudaStream_t xs = c->stream_xfer;
  if (S.done_idx >= 0) OKB_CUDA(c, cudaStreamWaitEvent(xs, c->done_ring[S.done_idx], 0));
  k_marg_export<<<1, 256, 0, xs>>>(c->d_wins, win, reinterpret_cast<double*>(c->hook_buf), cap);
  c->launches += 1;
  std::vector<double> host(cap);
  OKB_CUDA(c, cudaMemcpyAsync(host.data(), c->hook_buf, sizeof(double) * cap, cudaMemcpyDeviceToHost, xs));
  int32_t st[4] = {0, 0, 0, 0};
  if (S.marg_scratch) {
    const MargLayout m = marg_layout(S.marg_lm_cap, S.marg_K_cap, S.marg_L_cap, S.marg_O_cap);
    OKB_CUDA(c, cudaMemcpyAsync(st, S.marg_scratch + m.status, 16, cudaMemcpyDeviceToHost, xs));
  }
  OKB_CUDA(c, cudaStreamSynchronize(xs));
  const int nn = (int)host[0], nb = (int)host[1], xd = (int)host[2];
  if (n) *n = nn;
  if (n_blocks) *n_blocks = nb;
  if (status) std::memcpy(status, st, 16);
  if ((int)host[3] > cap) { c->set_error("okb_window_download_marg: prior larger than the export buffer"); return OKB_ERR_CAPACITY; }
  const double* o = host.data() + 8;
  for (int i = 0; i < nb; ++i) { if (block_kind) block_kind[i] = (int32_t)o[i]; if (block_idx) block_idx[i] = (uint32_t)o[nb + i]; }
  o += 2 * nb;
  if (x0) std::memcpy(x0, o, sizeof(double) * xd);
  o += xd;
  if (J) std::memcpy(J, o, sizeof(double) * (size_t)nn * nn);
  if (e0) std::memcpy(e0, o + (size_t)nn * nn, sizeof(double) * nn);
  if (H) std::memcpy(H, o + (size_t)nn * nn + nn, sizeof(double) * (size_t)nn * nn);
  if (b0) std::memcpy(b0, o + 2 * (size_t)nn * nn + nn, sizeof(double) * nn);
  return OKB_OK;
}

// ---------------------------------------------------------------------------------------------
// landmark-sharded single window: mailbox set-up (SURVEY 8e row 2)
// ---------------------------------------------------------------------------------------------
static int shard_alloc(okb_ctx* c, int rank, int world, int max_frames) {
  if (!c || world < 2 || world > kMaxShard || rank < 0 || rank >= world || max_frames < 1 || max_frames > kMaxFrames) return OKB_ERR_INVALID_ARG;
  if (c->shard_local) { c->set_error("landmark sharding is already set up on this context"); return OKB_ERR_INVALID_ARG; }
  cudaSetDevice(c->device);
  const int dcp = 4 * ((6 * max_frames + 1 + 3) / 4);
  c->shard_box_cap = (int)shard_box_doubles(max_frames, dcp);
  c->shard_win_bytes = shard_win_bytes(world, (size_t)c->shard_box_cap);
  const size_t total = c->shard_win_bytes * (size_t)c->max_windows;
  OKB_CUDA(c, cudaMalloc(&c->shard_local, total));
  OKB_CUDA(c, cudaMemset(c->shard_local, 0, total));
  OKB_CUDA(c, cudaDeviceSynchronize());
  c->shard_rank = rank;
  c->shard_world = world;
  c->shard_peer[rank] = c->shard_local;
  return OKB_OK;
}

extern "C" int okb_shard_export(okb_ctx* c, int rank, int world, int max_frames, void* handle_out) {
  if (!handle_out) return OKB_ERR_INVALID_ARG;
  int rc = shard_alloc(c, rank, world, max_frames);
  if (rc) return rc;
  static_assert(sizeof(cudaIpcMemHandle_t) == OKB_SHARD_HANDLE_BYTES, "handle size");
  cudaIpcMemHandle_t h;
  OKB_CUDA(c, cudaIpcGetMemHandle(&h, c->shard_local));
  std::memcpy(handle_out, &h, sizeof h);
  return OKB_OK;
}

extern "C" int okb_shard_connect(okb_ctx* c, const void* handles) {
  if (!c || !handles || c->shard_world < 2 || !c->shard_local) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  for (int r = 0; r < c->shard_world; ++r) {
    if (r == c->shard_rank) continue;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, static_cast<const unsigned char*>(handles) + (size_t)r * sizeof h, sizeof h);
    void* p = nullptr;
    OKB_CUDA(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    c->shard_peer[r] = static_cast<unsigned char*>(p);
    c->shard_peer_ipc[r] = true;
  }
  return OKB_OK;
}

extern "C" int okb_shard_connect_local(okb_ctx* const* ctxs, int world, int max_frames) {
  if (!ctxs || world < 2 || world > kMaxShard) return OKB_ERR_INVALID_ARG;
  for (int r = 0; r < world; ++r) {
    if (!ctxs[r]) return OKB_ERR_INVALID_ARG;
    if (ctxs[r]->max_windows != ctxs[0]->max_windows) { ctxs[r]->set_error("sharded contexts must have the same number of window slots"); return OKB_ERR_INVALID_ARG; }
    const int rc = shard_alloc(ctxs[r], r, world, max_frames);
    if (rc) return rc;
  }
  for (int r = 0; r < world; ++r) {
    okb_ctx* c = ctxs[r];
    cudaSetDevice(c->device);
    for (int q = 0; q < world; ++q) {
      if (q == r) continue;
      if (ctxs[q]->device != c->device) {
        const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[q]->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { c->set_error(std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e)); return OKB_ERR_CUDA; }
        cudaGetLastError();
      }
      c->shard_peer[q] = ctxs[q]->shard_local;
    }
  }
  return OKB_OK;
}

extern "C" int okb_shard_stats(okb_ctx* c, int win, double out[4]) {
  if (!c || win < 0 || win >= c->max_windows || !out) return OKB_ERR_INVALID_ARG;
  const SolverState& s = c->h_states[win];
  out[0] = (double)s.shard_rounds; out[1] = 1e-3 * (double)s.shard_wait_ns; out[2] = (double)s.shard_fault; out[3] = (double)s.shard_epoch;
  return OKB_OK;
}

// ---- optional event timing around solver kernels
static void prof_begin(okb_ctx* c, int kind) {
  if (!c->profile) return;
  if (c->prof_used + 2 > c->prof_events.size()) {
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    c->prof_events.push_back(a); c->prof_events.push_back(b);
  }
  c->prof_kind.push_back(kind);
  cudaEventRecord(c->prof_events[c->prof_used], c->stream);
}
static void prof_end(okb_ctx* c) {
  if (!c->profile) return;
  cudaEventRecord(c->prof_events[c->prof_used + 1], c->stream);
  c->prof_used += 2;
}
extern "C" int okb_profile_enable(okb_ctx* c, int on) {
  if (!c) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  c->profile = on != 0;
  c->prof_used = 0;
  c->prof_kind.clear();
  return OKB_OK;
}
extern "C" int okb_profile_read(okb_ctx* c, double out[6]) {
  if (!c || !out) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  for (int i = 0; i < 6; ++i) out[i] = 0.0;
  for (size_t i = 0; i < c->prof_kind.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->prof_events[2 * i], c->prof_events[2 * i + 1]);
    out[2 * c->prof_kind[i]] += ms;
    out[2 * c->prof_kind[i] + 1] += 1.0;
  }
  c->prof_used = 0;
  c->prof_kind.clear();
  return OKB_OK;
}

static int check_range(okb_ctx* c, int first, int count) {
  if (!c || first < 0 || count < 1 || first + count > c->max_windows) return OKB_ERR_INVALID_ARG;
  for (int i = first; i < first + count; ++i)
    if (!c->wins[i].uploaded) { c->set_error("window slot not uploaded"); return OKB_ERR_INVALID_ARG; }
  return OKB_OK;
}

extern "C" int64_t okb_window_h2d_bytes(const okb_ctx* c, int win) {
  if (!c || win < 0 || win >= c->max_windows || !c->wins[win].uploaded) return 0;
  return (int64_t)(c->wins[win].h2d_bytes + sizeof(WinDev));     // the last commit's command stream + the window descriptor
}

extern "C" int okb_window_reset(okb_ctx* c, int first, int count) {
  int rc = check_range(c, first, count);
  if (rc) return rc;
  cudaSetDevice(c->device);
  for (int i = first; i < first + count; ++i) {
    const WinStore& S = c->wins[i];
    const WinDev& W = c->host[i];
    if (W.K != S.K_init || W.NSB != S.NSB_init || W.L != S.L_init) { c->set_error("okb_window_reset: the window changed shape since its last full upload"); return OKB_ERR_INVALID_ARG; }
  }
  rc = commit_range(c, first, count);
  if (rc) return rc;
  // Runs on the TRANSFER stream (after the solver work already launched on these slots): restoring a slot is part of
  // preparing it, so it overlaps a solve that is running on other slots; the next okb_optimize* of the slot joins the
  // transfer stream as it does for uploads.
  cudaStream_t xs = c->stream_xfer;
  bool waited[okb_ctx::kDoneRing] = {};
  for (int i = first; i < first + count; ++i) {
    const WinStore& S = c->wins[i];
    if (S.done_idx >= 0 && !waited[S.done_idx]) {
      OKB_CUDA(c, cudaStreamWaitEvent(xs, c->done_ring[S.done_idx], 0));
      waited[S.done_idx] = true;
    }
  }
  k_reset<<<count, 128, 0, xs>>>(c->d_wins, first, 1);
  c->launches += 1;
  OKB_CUDA(c, cudaGetLastError());
  return OKB_OK;
}

// ---------------------------------------------------------------------------------------------
// optimize
// ---------------------------------------------------------------------------------------------
// Launch geometry of one optimize of windows [first, first+count): everything a captured CUDA graph depends on
// besides the kernel arguments.
struct RoundPlan {
  int max_chunks = 1, max_imu = 0, max_cx = 1, max_K = 1, acc_smem = 1, chol_smem = 1, solve_threads = S_THREADS, gxQ = 1, shard = 0, push_gx = 1;
  size_t smA = 0, smS = 0, smQ = 0;
};
static int plan_rounds(okb_ctx* c, int first, int count, RoundPlan& P) {
  P = RoundPlan();
  int chol_smem = 1;       // solve_mode of k_solve: 1 system in shared memory, 2 pose system + chain band, 0 chain band only
  // Schur accumulator in shared memory if two CTAs per SM still fit (else one CTA; else accumulate in global memory)
  int acc_smem = 1;
  const size_t sm_two = ((size_t)c->smem_per_sm - 2048) / 2;
  for (int i = first; i < first + count; ++i)
    if (smemA2_bytes(c->host[i].K, 1) > std::min((size_t)c->smem_optin, sm_two) &&
        smemA2_bytes(c->host[i].K, 0) <= sm_two) acc_smem = 0;
  for (int i = first; i < first + count; ++i)
    if (smemA2_bytes(c->host[i].K, acc_smem) > (size_t)c->smem_optin) acc_smem = 0;
  int maxL = 1;
  for (int i = first; i < first + count; ++i) {
    const WinDev& W = c->host[i];
    P.max_chunks = std::max(P.max_chunks, W.n_chunks);
    P.max_imu = std::max(P.max_imu, W.n_imu);
    P.smA = std::max(P.smA, smemA2_bytes(W.K, acc_smem));
    P.max_cx = std::max(P.max_cx, (W.L + L1_THREADS - 1) / L1_THREADS);
    P.max_K = std::max(P.max_K, W.K);
    {      // the roomiest mode this window fits; the range runs in the most modest one (1 > 2 > 0)
      const int wm = smemS_bytes(W.d, W.dc, W.K, W.marg_n, W.n_imu, 1) <= (size_t)c->smem_optin ? 1
                   : smemS_bytes(W.d, W.dc, W.K, W.marg_n, W.n_imu, 2) <= (size_t)c->smem_optin ? 2 : 0;
      if (wm == 0 || chol_smem == 0) chol_smem = 0;
      else if (wm == 2) chol_smem = 2;
    }
    P.smQ = std::max(P.smQ, (size_t)W.NS * sizeof(SlotCtx));
    maxL = std::max(maxL, W.L);
  }
  for (int i = first; i < first + count; ++i) {
    const WinDev& W = c->host[i];
    P.smS = std::max(P.smS, smemS_bytes(W.d, W.dc, W.K, W.marg_n, W.n_imu, chol_smem));
  }
  if (P.smS > (size_t)c->smem_optin) { c->set_error("window does not fit kernel S shared memory"); return OKB_ERR_CAPACITY; }
  if (const char* force = getenv("OKB_SOLVE_MODE")) {      // diagnostics / tests: a more modest solve_mode than the windows need (2 or 0)
    const int m = atoi(force);
    if ((m == 0 || m == 2) && chol_smem != 0 && !(chol_smem == 2 && m == 2)) {
      chol_smem = m;
      P.smS = 0;
      for (int i = first; i < first + count; ++i) {
        const WinDev& W = c->host[i];
        P.smS = std::max(P.smS, smemS_bytes(W.d, W.dc, W.K, W.marg_n, W.n_imu, chol_smem));
      }
      if (P.smS > (size_t)c->smem_optin) { c->set_error("window does not fit kernel S shared memory"); return OKB_ERR_CAPACITY; }
    }
  }
  P.acc_smem = acc_smem; P.chol_smem = chol_smem;
  P.solve_threads = (2 * count <= c->sm_count) ? 512 : S_THREADS;      // few windows: one wide CTA per SM (all ranks of a sharded window choose alike)
  P.gxQ = std::max(1, std::min((maxL + 127) / 128, (4 * c->sm_count + count - 1) / count));
  P.shard = c->shard_world > 1 ? 1 : 0;
  P.push_gx = std::max(1, std::min(16, c->sm_count / std::max(1, count)));
  return OKB_OK;
}

static int launch_rounds(okb_ctx* c, int first, int count, const okb_solve_options& opt, int rounds, const RoundPlan& P) {
  for (int r = 0; r < rounds; ++r) {
    const dim3 gridA(P.max_chunks, count);
    static const bool imu_serial = getenv("OKB_IMU_SERIAL") != nullptr;     // diagnostics: k_imu on the main stream, ahead of the landmark kernels
    if (P.max_imu > 0 && imu_serial) {
      k_imu<<<dim3((P.max_imu + 32 / IMU_G - 1) / (32 / IMU_G), count), 32, smemI_bytes(), c->stream>>>(c->d_wins, first);
      c->launches += 1;
    } else if (P.max_imu > 0) {   // IMU terms only depend on the previous round's candidate: run beside the landmark kernels
      cudaEventRecord(c->ev_round, c->stream);
      cudaStreamWaitEvent(c->stream_imu, c->ev_round, 0);
      k_imu<<<dim3((P.max_imu + 32 / IMU_G - 1) / (32 / IMU_G), count), 32, smemI_bytes(), c->stream_imu>>>(c->d_wins, first);
      cudaEventRecord(c->ev_imu, c->stream_imu);
      c->launches += 1;
    }
    prof_begin(c, 0);
    k_linearize<<<dim3(P.max_cx, P.max_K, count), L1_THREADS, 0, c->stream>>>(c->d_wins, first);
    k_lmblock<<<dim3(P.max_cx, count), 128, 0, c->stream>>>(c->d_wins, first);
    k_schur<<<gridA, A2_THREADS, P.smA, c->stream>>>(c->d_wins, first, P.acc_smem, opt.max_iterations);
    if (P.shard) {    // chunk reduction fused with the push half of the all-reduce over peer memory
      k_shard_push<<<dim3(P.push_gx, count), 256, 0, c->stream>>>(c->d_wins, first);
      c->launches += 1;
    } else if (P.max_chunks > 1) { k_reduce_partials<<<dim3(8, count), 256, 0, c->stream>>>(c->d_wins, first); c->launches += 1; }
    prof_end(c);
    c->launches += 3;
    if (P.max_imu > 0 && !imu_serial) cudaStreamWaitEvent(c->stream, c->ev_imu, 0);
    prof_begin(c, 1);
    if (P.solve_threads == 512) k_solve<512><<<count, 512, P.smS, c->stream>>>(c->d_wins, first, opt, P.chol_smem);
    else k_solve<S_THREADS><<<count, S_THREADS, P.smS, c->stream>>>(c->d_wins, first, opt, P.chol_smem);
    prof_end(c);
    c->launches += 1;
  }
  OKB_CUDA(c, cudaGetLastError());
  return OKB_OK;
}

// post-solve landmark quality (Estimator.cpp:880-894)
static int launch_quality(okb_ctx* c, int first, int count, const RoundPlan& P) {
  prof_begin(c, 2);
  k_quality<<<dim3(P.gxQ, count), 128, P.smQ, c->stream>>>(c->d_wins, first);
  prof_end(c);
  c->launches += 1;
  OKB_CUDA(c, cudaGetLastError());
  return OKB_OK;
}

// The fixed launch sequence of one optimize (rounds + quality pass) as a CUDA graph: captured once per launch
// geometry / option set and replayed -- one host call instead of ~70 launches and ~40 event operations, which is
// what bounds the latency of a single window (SURVEY 8d "B = 1").  OKB_NO_GRAPH=1 disables it (diagnostics).
static int run_rounds(okb_ctx* c, int first, int count, const okb_solve_options& opt, int rounds, bool with_quality) {
  RoundPlan P;
  int rc = plan_rounds(c, first, count, P);
  if (rc) return rc;
  static const bool no_graph = getenv("OKB_NO_GRAPH") != nullptr;
  // landmark-sharded windows spin on their peers inside k_solve: their kernels must reach the device in stream order,
  // not behind whatever hardware queue a graph's internal branches were mapped to
  if (c->profile || no_graph || c->shard_world > 1) {
    rc = launch_rounds(c, first, count, opt, rounds, P);
    if (!rc && with_quality) rc = launch_quality(c, first, count, P);
    return rc;
  }
  okb_ctx::GraphEntry key;
  std::memset(&key, 0, sizeof key);
  key.first = first; key.count = count; key.rounds = rounds; key.with_quality = with_quality ? 1 : 0;
  key.opt_iter = opt.max_iterations; key.opt_min = opt.min_iterations; key.opt_cauchy = opt.use_cauchy_loss; key.opt_time = opt.time_limit_s;
  static_assert(sizeof(RoundPlan) <= sizeof(key.plan), "plan blob");
  std::memcpy(key.plan, &P, sizeof P);
  for (auto& e : c->graphs)
    if (e.exec && !std::memcmp(&e, &key, offsetof(okb_ctx::GraphEntry, exec))) {
      e.stamp = ++c->graph_clock;
      OKB_CUDA(c, cudaGraphLaunch(e.exec, c->stream));
      c->launches += e.launches;
      return OKB_OK;
    }
  const int64_t l0 = c->launches;
  cudaGraph_t graph = nullptr;
  OKB_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
  rc = launch_rounds(c, first, count, opt, rounds, P);
  if (!rc && with_quality) rc = launch_quality(c, first, count, P);
  const cudaError_t ce = cudaStreamEndCapture(c->stream, &graph);
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  OKB_CUDA(c, ce);
  key.launches = c->launches - l0;
  c->launches = l0;
  OKB_CUDA(c, cudaGraphInstantiate(&key.exec, graph, 0));
  cudaGraphDestroy(graph);
  okb_ctx::GraphEntry* slot = nullptr;
  for (auto& e : c->graphs) if (!e.exec) { slot = &e; break; }
  if (!slot && c->graphs.size() < 16) { c->graphs.emplace_back(); slot = &c->graphs.back(); }
  if (!slot) {     // evict the least recently used
    slot = &c->graphs[0];
    for (auto& e : c->graphs) if (e.stamp < slot->stamp) slot = &e;
    cudaGraphExecDestroy(slot->exec);
  }
  key.stamp = ++c->graph_clock;
  *slot = key;
  OKB_CUDA(c, cudaGraphLaunch(slot->exec, c->stream));
  c->launches += slot->launches;
  return OKB_OK;
}

extern "C" int okb_optimize_async(okb_ctx* c, int first, int count, const okb_solve_options* opt) {
  int rc = check_range(c, first, count);
  if (rc) return rc;
  if (!opt || opt->max_iterations < 0) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  rc = commit_range(c, first, count);       // pending graph commands of these slots (no-op when there are none)
  if (rc) return rc;
  // chunking: enough CTAs for ~2 waves when the batch is small
  for (int i = first; i < first + count; ++i) {
    WinDev& W = c->host[i];
    int chunks = (2 * c->sm_count + count - 1) / count;
    chunks = std::max(1, std::min(chunks, c->chunk_cap));
    chunks = std::min(chunks, std::max(1, W.L / (2 * A2_TILE)));
    W.lm_per_chunk = (((W.L + chunks - 1) / chunks) + A2_TILE - 1) / A2_TILE * A2_TILE;   // whole tiles per chunk
    W.n_chunks = (W.L + W.lm_per_chunk - 1) / W.lm_per_chunk;
    W.use_cauchy = opt->use_cauchy_loss ? 1 : 0;
  }
  if (join_transfers(c)) { c->set_error("stream ordering failed"); return OKB_ERR_CUDA; }
  OKB_CUDA(c, cudaMemcpyAsync(c->d_wins + first, &c->host[first], sizeof(WinDev) * count, cudaMemcpyHostToDevice, c->stream));
  k_reset<<<count, 128, 0, c->stream>>>(c->d_wins, first, 0);
  c->launches += 1;
  for (int i = first; i < first + count; ++i) c->wins[i].opt = *opt;     // okb_optimize_finish relaunches with the range's own options
  // round 0 linearises at the initial state; each later round judges one step and proposes the next
  rc = run_rounds(c, first, count, *opt, opt->max_iterations + 1, true);
  if (rc) return rc;
  OKB_CUDA(c, cudaMemcpyAsync(c->h_states + first, c->d_states + first, sizeof(SolverState) * count, cudaMemcpyDeviceToHost, c->stream));
  mark_work(c, first, count);
  return rc;
}

extern "C" int okb_optimize_finish(okb_ctx* c, int first, int count, okb_summary* out) {
  int rc = check_range(c, first, count);
  if (rc) return rc;
  cudaSetDevice(c->device);
  // optimize_async already queued the landmark-quality pass and the copy of the solver states.  Rebuild
  // rounds (linear-solver failures) consume rounds without advancing the iteration count: keep launching
  // until every window reports done (bounded).
  for (int guard = 0; guard < 64; ++guard) {
    OKB_CUDA(c, cudaStreamSynchronize(c->stream));
    bool all_done = true;
    for (int i = first; i < first + count; ++i) all_done = all_done && c->h_states[i].done;
    if (all_done) break;
    rc = run_rounds(c, first, count, c->wins[first].opt, 2, true);
    if (rc) return rc;
    OKB_CUDA(c, cudaMemcpyAsync(c->h_states + first, c->d_states + first, sizeof(SolverState) * count, cudaMemcpyDeviceToHost, c->stream));
    mark_work(c, first, count);
  }
  for (int i = first; i < first + count; ++i) {
    const SolverState& s = c->h_states[i];
    if (s.g.err) { c->set_error(graph_error_text(s.g.err)); return graph_error_status(s.g.err); }
    WinStore& S = c->wins[i];
    if (!S.cmd_used) S.obs_bound = s.g.n_obs;      // exact length of the compacted observation list
  }
  if (out) {
    for (int i = 0; i < count; ++i) {
      const SolverState& s = c->h_states[first + i];
      okb_summary& o = out[i];
      o.initial_cost = s.initial_cost; o.final_cost = s.cost; o.iterations = s.iteration;
      o.num_successful_steps = s.num_successful; o.termination = s.done ? s.termination : OKB_TERM_FAILURE;
      o.imu_redo_count = s.imu_redo_final; o.final_radius = s.radius; o.solve_time_s = s.solve_time_s;
    }
  }
  return OKB_OK;
}

// diagnostics: the ImuError cache of term `term` (reference bias of the preintegration, valid flag, redo counter)
extern "C" int okb_debug_imu_cache(okb_ctx* c, int win, int term, double sb_ref[9], int32_t* valid, int32_t* redo_count) {
  int rc = check_range(c, win, 1);
  if (rc) return rc;
  cudaSetDevice(c->device);
  rc = commit_range(c, win, 1);
  if (rc) return rc;
  const WinDev& W = c->host[win];
  if (term < 0 || term >= W.n_imu) return OKB_ERR_INVALID_ARG;
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream_xfer));
  ImuCache h;
  OKB_CUDA(c, cudaMemcpy(&h, W.imu_cache + term, sizeof(ImuCache), cudaMemcpyDeviceToHost));
  if (sb_ref) std::memcpy(sb_ref, h.sb_ref, sizeof(double) * 9);
  if (valid) *valid = h.valid;
  if (redo_count) *redo_count = h.redo_count;
  return OKB_OK;
}

// diagnostics: accumulated k_solve phase times (ns) of the last optimize of `win`
extern "C" int okb_debug_phase_ns(okb_ctx* c, int win, double out[16]) {
  if (!c || win < 0 || win >= c->max_windows || !out) return OKB_ERR_INVALID_ARG;
  for (int i = 0; i < 16; ++i) out[i] = (double)c->h_states[win].phase_ns[i];
  return OKB_OK;
}

extern "C" int okb_optimize(okb_ctx* c, int first, int count, const okb_solve_options* opt, okb_summary* out) {
  int rc = okb_optimize_async(c, first, count, opt);
  if (rc) return rc;
  return okb_optimize_finish(c, first, count, out);
}

// The estimates come back from the packed output block (pose | speed/bias | landmarks | quality, caller's order) that
// k_quality / k_prepare / k_reset keep current: one D2H copy per window, plain memcpy on the host.
static size_t out_doubles(const WinDev& W) { return out_lm_offset(W.K, W.NSB) + 5 * (size_t)W.L; }
static void copy_out_window(const WinDev& W, const WinStore& S, double* poses, double* speed_bias, double* landmarks, double* quality) {
  const double* o = reinterpret_cast<const double*>(S.out_staging);
  if (poses) std::memcpy(poses, o, sizeof(double) * 7 * W.K);
  if (speed_bias && W.NSB) std::memcpy(speed_bias, o + 7 * W.K, sizeof(double) * 9 * W.NSB);
  if (landmarks) std::memcpy(landmarks, o + out_lm_offset(W.K, W.NSB), sizeof(double) * 4 * (size_t)W.L);
  if (quality) std::memcpy(quality, o + out_lm_offset(W.K, W.NSB) + 4 * (size_t)W.L, sizeof(double) * (size_t)W.L);
}

extern "C" int okb_window_download(okb_ctx* c, int win, double* poses, double* speed_bias, double* landmarks, double* quality) {
  int rc = check_range(c, win, 1);
  if (rc) return rc;
  cudaSetDevice(c->device);
  rc = commit_range(c, win, 1);
  if (rc) return rc;
  const WinDev& W = c->host[win];
  WinStore& S = c->wins[win];
  cudaStream_t xs = c->stream_xfer;
  if (S.done_idx >= 0) OKB_CUDA(c, cudaStreamWaitEvent(xs, c->done_ring[S.done_idx], 0));
  OKB_CUDA(c, cudaMemcpyAsync(S.out_staging, W.out, sizeof(double) * out_doubles(W), cudaMemcpyDeviceToHost, xs));
  OKB_CUDA(c, cudaEventRecord(S.down, xs));
  OKB_CUDA(c, cudaEventSynchronize(S.down));
  copy_out_window(W, S, poses, speed_bias, landmarks, quality);
  return OKB_OK;
}

extern "C" int okb_window_download_batch(okb_ctx* c, int first, int count, double* const* poses, double* const* speed_bias,
                                         double* const* landmarks, double* const* quality) {
  int rc = check_range(c, first, count);
  if (rc) return rc;
  cudaSetDevice(c->device);
  rc = commit_range(c, first, count);
  if (rc) return rc;
  cudaStream_t xs = c->stream_xfer;
  bool waited[okb_ctx::kDoneRing] = {};
  for (int i = first; i < first + count; ++i) {
    WinStore& S = c->wins[i];
    if (S.done_idx >= 0 && !waited[S.done_idx]) {
      OKB_CUDA(c, cudaStreamWaitEvent(xs, c->done_ring[S.done_idx], 0));
      waited[S.done_idx] = true;
    }
  }
  for (int i = first; i < first + count; ++i)
    OKB_CUDA(c, cudaMemcpyAsync(c->wins[i].out_staging, c->host[i].out, sizeof(double) * out_doubles(c->host[i]), cudaMemcpyDeviceToHost, xs));
  WinStore& S0 = c->wins[first];
  OKB_CUDA(c, cudaEventRecord(S0.down, xs));
  OKB_CUDA(c, cudaEventSynchronize(S0.down));
  auto copy_out = [&](int i) {
    const int k = i - first;
    copy_out_window(c->host[i], c->wins[i], poses ? poses[k] : nullptr, speed_bias ? speed_bias[k] : nullptr,
                    landmarks ? landmarks[k] : nullptr, quality ? quality[k] : nullptr);
  };
  const int T = std::max(1, std::min(8, count / 32));
  if (T == 1) {
    for (int i = first; i < first + count; ++i) copy_out(i);
  } else {
    std::vector<std::thread> th;
    th.reserve(T);
    for (int t = 0; t < T; ++t)
      th.emplace_back([&, t]() { for (int i = first + t; i < first + count; i += T) copy_out(i); });
    for (auto& x : th) x.join();
  }
  return OKB_OK;
}

// ---------------------------------------------------------------------------------------------
// single-block test hooks (ErrorInterface::EvaluateWithMinimalJacobians mirrors)
// ---------------------------------------------------------------------------------------------
namespace {
__global__ void k_hook_reproj(int n, okb_camera cam, const double* pose, const double* lm, const double* ext, const double* z,
                              const double* sq, double* r, double* J0, double* J1, double* J2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  reproj_full(cam, pose + 7 * i, lm + 4 * i, ext + 7 * i, z + 2 * i, sq[i], r + 2 * i, J0 + 12 * i, J1 + 6 * i, J2 + 12 * i);
}
// one warp
__global__ void k_hook_imu(okb_imu_params prm, const okb_imu_sample* s, int n, int64_t t0, int64_t t1, const double* in /*32*/,
                           const double* sb_ref, int have_ref, ImuCache* cache, double* out /* r15 | SF 450 | sqrt 225 | redo */) {
  __shared__ double buf[3 * 225 + 450 + 450 + 16 + 32 * kImuPre];
  WarpCtx cx;
  ImuWork wk{buf, buf + 225, buf + 450, buf + 1125, buf + 1591};
  double* F01 = buf + 675; double* SF = buf + 1125; double* r15 = buf + 1575;
  if (threadIdx.x == 0) { cache->valid = 0; cache->redo_count = 0; for (int k = 0; k < 9; ++k) cache->sb_ref[k] = 0; }
  __syncwarp();
  if (have_ref) imu_preintegrate(cx, s, n, prm, t0, t1, sb_ref, cache, wk);
  const int before = cache->redo_count;
  __syncwarp();
  imu_evaluate(cx, s, n, prm, t0, t1, in, in + 7, in + 16, in + 23, cache, wk, F01, (double*)nullptr, r15, SF);
  for (int e = threadIdx.x; e < 15; e += 32) out[e] = r15[e];
  for (int e = threadIdx.x; e < 450; e += 32) out[15 + e] = SF[e];
  for (int e = threadIdx.x; e < 225; e += 32) out[465 + e] = cache->sqrt_info[e];
  if (threadIdx.x == 0) out[690] = (double)(cache->redo_count - before);
}
__global__ void k_hook_propagate(okb_imu_params prm, const okb_imu_sample* s, int n, int64_t t0, int64_t t1, double* io /*16*/,
                                 double* cov, double* jac, int want_cov, int want_jac, int* n_used) {
  __shared__ double buf[4 * 225 + 32 * kImuPre];
  WarpCtx cx;
  ImuWork wk{buf, buf + 225, buf + 450, buf + 675, buf + 900};
  const int steps = imu_propagate(cx, s, n, prm, t0, t1, io, io + 7, want_cov ? cov : nullptr, want_jac ? jac : nullptr, wk);
  if (threadIdx.x == 0) *n_used = steps;
}
__global__ void k_hook_pose(const double* in /* meas7 S36 pose7 */, double* out /* r6 J36 */) {
  if (threadIdx.x == 0) pose_error(in, in + 7, in + 43, out, out + 6);
}
__global__ void k_hook_relpose(const double* in /* S36 p0 p1 */, double* out /* r6 J0 J1 */) {
  if (threadIdx.x == 0) relative_pose_error(in, in + 36, in + 43, out, out + 6, out + 42);
}
}  // namespace

static int hook_alloc(okb_ctx* c, size_t bytes);
static int hook_alloc_fwd(okb_ctx* c, size_t bytes) { return hook_alloc(c, bytes); }
static int hook_alloc(okb_ctx* c, size_t bytes) {
  if (c->hook_bytes >= bytes) return OKB_OK;
  if (c->hook_buf) cudaFree(c->hook_buf);
  c->hook_buf = nullptr; c->hook_bytes = 0;
  OKB_CUDA(c, cudaMalloc(&c->hook_buf, bytes));
  c->hook_bytes = bytes;
  return OKB_OK;
}

extern "C" int okb_eval_reprojection(okb_ctx* c, int n, const okb_camera* cam, const double* pose, const double* landmark,
                                     const double* extrinsics, const double* z, const double* sqrt_info, double* r,
                                     double* J_pose, double* J_lm, double* J_ext) {
  if (!c || n < 1 || !cam) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  const size_t nin = (size_t)n * (7 + 4 + 7 + 2 + 1), nout = (size_t)n * (2 + 12 + 6 + 12);
  int rc = hook_alloc(c, (nin + nout) * sizeof(double));
  if (rc) return rc;
  double* d = reinterpret_cast<double*>(c->hook_buf);
  double *dp = d, *dl = dp + 7 * (size_t)n, *de = dl + 4 * (size_t)n, *dz = de + 7 * (size_t)n, *dq = dz + 2 * (size_t)n;
  double *dr = dq + n, *d0 = dr + 2 * (size_t)n, *d1 = d0 + 12 * (size_t)n, *d2 = d1 + 6 * (size_t)n;
  OKB_CUDA(c, cudaMemcpyAsync(dp, pose, sizeof(double) * 7 * n, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dl, landmark, sizeof(double) * 4 * n, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(de, extrinsics, sizeof(double) * 7 * n, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dz, z, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dq, sqrt_info, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
  k_hook_reproj<<<(n + 127) / 128, 128, 0, c->stream>>>(n, *cam, dp, dl, de, dz, dq, dr, d0, d1, d2);
  c->launches += 1;
  OKB_CUDA(c, cudaGetLastError());
  if (r) OKB_CUDA(c, cudaMemcpyAsync(r, dr, sizeof(double) * 2 * n, cudaMemcpyDeviceToHost, c->stream));
  if (J_pose) OKB_CUDA(c, cudaMemcpyAsync(J_pose, d0, sizeof(double) * 12 * n, cudaMemcpyDeviceToHost, c->stream));
  if (J_lm) OKB_CUDA(c, cudaMemcpyAsync(J_lm, d1, sizeof(double) * 6 * n, cudaMemcpyDeviceToHost, c->stream));
  if (J_ext) OKB_CUDA(c, cudaMemcpyAsync(J_ext, d2, sizeof(double) * 12 * n, cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  return OKB_OK;
}

extern "C" int okb_eval_imu(okb_ctx* c, const okb_imu_params* prm, const okb_imu_sample* samples, int n_samples, int64_t t0_ns,
                            int64_t t1_ns, const double* pose0, const double* sb0, const double* pose1, const double* sb1,
                            const double* sb_ref, double* r, double* J0, double* J1, double* J2, double* J3,
                            double* sqrt_info_out) {
  if (!c || !prm || !samples || n_samples < 2) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  const size_t sbytes = align_up(sizeof(okb_imu_sample) * n_samples, 256);
  const size_t total = sbytes + align_up(sizeof(ImuCache), 256) + sizeof(double) * (32 + 9 + 7 + 700);
  int rc = hook_alloc(c, total);
  if (rc) return rc;
  unsigned char* base = reinterpret_cast<unsigned char*>(c->hook_buf);
  okb_imu_sample* ds = reinterpret_cast<okb_imu_sample*>(base);
  ImuCache* dc = reinterpret_cast<ImuCache*>(base + sbytes);
  double* din = reinterpret_cast<double*>(base + sbytes + align_up(sizeof(ImuCache), 256));
  double* dref = din + 32;
  double* dout = dref + 16;
  double hin[32];
  std::memcpy(hin, pose0, 56); std::memcpy(hin + 7, sb0, 72); std::memcpy(hin + 16, pose1, 56); std::memcpy(hin + 23, sb1, 72);
  OKB_CUDA(c, cudaMemcpyAsync(ds, samples, sizeof(okb_imu_sample) * n_samples, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(din, hin, sizeof(hin), cudaMemcpyHostToDevice, c->stream));
  if (sb_ref) OKB_CUDA(c, cudaMemcpyAsync(dref, sb_ref, 72, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  k_hook_imu<<<1, 32, 0, c->stream>>>(*prm, ds, n_samples, t0_ns, t1_ns, din, dref, sb_ref ? 1 : 0, dc, dout);
  c->launches += 1;
  OKB_CUDA(c, cudaGetLastError());
  std::vector<double> h(691);
  OKB_CUDA(c, cudaMemcpyAsync(h.data(), dout, sizeof(double) * 691, cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  if (r) std::memcpy(r, h.data(), 15 * 8);
  const double* SF = h.data() + 15;
  for (int rr = 0; rr < 15; ++rr) {
    for (int cc = 0; cc < 6; ++cc) { if (J0) J0[rr * 6 + cc] = SF[rr * 30 + cc]; if (J2) J2[rr * 6 + cc] = SF[rr * 30 + 15 + cc]; }
    for (int cc = 0; cc < 9; ++cc) { if (J1) J1[rr * 9 + cc] = SF[rr * 30 + 6 + cc]; if (J3) J3[rr * 9 + cc] = SF[rr * 30 + 21 + cc]; }
  }
  if (sqrt_info_out) std::memcpy(sqrt_info_out, h.data() + 465, 225 * 8);
  return (int)h[690] > 0 ? 1 : 0;   // 1 = the evaluation re-preintegrated (not an error)
}

extern "C" int okb_imu_propagate(okb_ctx* c, const okb_imu_params* prm, const okb_imu_sample* samples, int n_samples,
                                 int64_t t0_ns, int64_t t1_ns, double* pose, double* sb, double* covariance, double* jacobian,
                                 int* n_used) {
  if (!c || !prm || !samples || n_samples < 2 || !pose || !sb) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  const size_t sbytes = align_up(sizeof(okb_imu_sample) * n_samples, 256);
  int rc = hook_alloc(c, sbytes + sizeof(double) * (16 + 450 + 2));
  if (rc) return rc;
  unsigned char* base = reinterpret_cast<unsigned char*>(c->hook_buf);
  okb_imu_sample* ds = reinterpret_cast<okb_imu_sample*>(base);
  double* dio = reinterpret_cast<double*>(base + sbytes);
  double* dcov = dio + 16;
  double* djac = dcov + 225;
  int* dn = reinterpret_cast<int*>(djac + 225);
  double hio[16];
  std::memcpy(hio, pose, 56); std::memcpy(hio + 7, sb, 72);
  OKB_CUDA(c, cudaMemcpyAsync(ds, samples, sizeof(okb_imu_sample) * n_samples, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dio, hio, sizeof hio, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  k_hook_propagate<<<1, 32, 0, c->stream>>>(*prm, ds, n_samples, t0_ns, t1_ns, dio, dcov, djac, covariance ? 1 : 0, jacobian ? 1 : 0, dn);
  c->launches += 1;
  OKB_CUDA(c, cudaGetLastError());
  int hn = 0;
  OKB_CUDA(c, cudaMemcpyAsync(hio, dio, sizeof hio, cudaMemcpyDeviceToHost, c->stream));
  if (covariance) OKB_CUDA(c, cudaMemcpyAsync(covariance, dcov, 225 * 8, cudaMemcpyDeviceToHost, c->stream));
  if (jacobian) OKB_CUDA(c, cudaMemcpyAsync(jacobian, djac, 225 * 8, cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(&hn, dn, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  if (hn >= 0) { std::memcpy(pose, hio, 56); std::memcpy(sb, hio + 7, 72); }
  if (n_used) *n_used = hn;
  return OKB_OK;
}

extern "C" int okb_eval_pose_error(okb_ctx* c, const double* meas, const double* sqrt_info, const double* pose, double* r, double* J) {
  if (!c) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  int rc = hook_alloc(c, sizeof(double) * (50 + 42));
  if (rc) return rc;
  double* d = reinterpret_cast<double*>(c->hook_buf);
  double h[50];
  std::memcpy(h, meas, 56); std::memcpy(h + 7, sqrt_info, 288); std::memcpy(h + 43, pose, 56);
  OKB_CUDA(c, cudaMemcpyAsync(d, h, sizeof h, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  k_hook_pose<<<1, 32, 0, c->stream>>>(d, d + 50);
  c->launches += 1;
  double o[42];
  OKB_CUDA(c, cudaMemcpyAsync(o, d + 50, sizeof o, cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  if (r) std::memcpy(r, o, 48);
  if (J) std::memcpy(J, o + 6, 288);
  return OKB_OK;
}

namespace {
__global__ void k_hook_sb(const double* in /* meas9 S81 sb9 */, double* out /* r9 J81 */) {
  const int t = threadIdx.x;
  if (t < 9) {
    double s = 0;
    for (int k = 0; k < 9; ++k) s += in[9 + t * 9 + k] * (in[k] - in[90 + k]);
    out[t] = s;
  }
  for (int e = t; e < 81; e += blockDim.x) out[9 + e] = -in[9 + e];
}
}  // namespace

extern "C" int okb_eval_speed_bias_error(okb_ctx* c, const double* meas, const double* sqrt_info, const double* sb, double* r, double* J) {
  if (!c || !meas || !sqrt_info || !sb) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  int rc = hook_alloc(c, sizeof(double) * (99 + 90));
  if (rc) return rc;
  double* d = reinterpret_cast<double*>(c->hook_buf);
  double h[99];
  std::memcpy(h, meas, 72); std::memcpy(h + 9, sqrt_info, 648); std::memcpy(h + 90, sb, 72);
  OKB_CUDA(c, cudaMemcpyAsync(d, h, sizeof h, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  k_hook_sb<<<1, 96, 0, c->stream>>>(d, d + 99);
  c->launches += 1;
  double o[90];
  OKB_CUDA(c, cudaMemcpyAsync(o, d + 99, sizeof o, cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  if (r) std::memcpy(r, o, 72);
  if (J) std::memcpy(J, o + 9, 648);
  return OKB_OK;
}

extern "C" int okb_eval_relative_pose(okb_ctx* c, const double* sqrt_info, const double* pose0, const double* pose1, double* r,
                                      double* J0, double* J1) {
  if (!c) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  int rc = hook_alloc(c, sizeof(double) * (50 + 78));
  if (rc) return rc;
  double* d = reinterpret_cast<double*>(c->hook_buf);
  double h[50];
  std::memcpy(h, sqrt_info, 288); std::memcpy(h + 36, pose0, 56); std::memcpy(h + 43, pose1, 56);
  OKB_CUDA(c, cudaMemcpyAsync(d, h, sizeof h, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  k_hook_relpose<<<1, 32, 0, c->stream>>>(d, d + 50);
  c->launches += 1;
  double o[78];
  OKB_CUDA(c, cudaMemcpyAsync(o, d + 50, sizeof o, cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  if (r) std::memcpy(r, o, 48);
  if (J0) std::memcpy(J0, o + 6, 288);
  if (J1) std::memcpy(J1, o + 42, 288);
  return OKB_OK;
}

namespace {
__global__ void k_hook_marg(int n, int nb, const int32_t* kind, const int32_t* col, const int32_t* off, const double* x0,
                            const double* x, const double* J, const double* e0, double* r, double* Jeff) {
  extern __shared__ double dchi[];
  const int tid = threadIdx.x;
  for (int b = tid; b < nb; b += blockDim.x) {
    if (kind[b] == OKB_BLOCK_SPEED_BIAS) for (int k = 0; k < 9; ++k) dchi[col[b] + k] = x[off[b] + k] - x0[off[b] + k];
    else pose_minus(x0 + off[b], x + off[b], dchi + col[b]);
  }
  __syncthreads();
  for (int i = tid; i < n; i += blockDim.x) {
    double s = e0[i];
    for (int k = 0; k < n; ++k) s += J[(size_t)i * n + k] * dchi[k];
    r[i] = s;
  }
  for (int b = 0; b < nb; ++b) {
    const int m = (kind[b] == OKB_BLOCK_SPEED_BIAS) ? 9 : 6;
    double B[9];
    if (m == 6) marg_pose_rot_block(x0 + off[b], x + off[b], B);
    for (int e = tid; e < n * m; e += blockDim.x) {
      const int i = e / m, a = e % m;
      double s;
      if (m == 9 || a < 3) s = J[(size_t)i * n + col[b] + a];
      else { s = 0; for (int k = 0; k < 3; ++k) s += J[(size_t)i * n + col[b] + 3 + k] * B[k * 3 + (a - 3)]; }
      Jeff[(size_t)i * n + col[b] + a] = s;
    }
  }
}
}  // namespace

extern "C" int okb_eval_marginalization(okb_ctx* c, const okb_marg_prior* m, const double* x, double* r, double* J_eff) {
  if (!c || !m || m->n < 1 || m->n > kMaxMarg) return OKB_ERR_INVALID_ARG;
  cudaSetDevice(c->device);
  const int n = m->n, nb = m->n_blocks;
  std::vector<int32_t> kind(nb), col(nb), off(nb);
  int cc = 0, xo = 0;
  for (int b = 0; b < nb; ++b) {
    kind[b] = m->block_kind[b]; col[b] = cc; off[b] = xo;
    cc += (kind[b] == OKB_BLOCK_SPEED_BIAS) ? 9 : 6;
    xo += (kind[b] == OKB_BLOCK_SPEED_BIAS) ? 9 : 7;
  }
  if (cc != n) return OKB_ERR_INVALID_ARG;
  const size_t ints = align_up(sizeof(int32_t) * 3 * nb, 256);
  const size_t total = ints + sizeof(double) * (2 * xo + (size_t)2 * n * n + 2 * n);
  int rc = hook_alloc(c, total);
  if (rc) return rc;
  unsigned char* base = reinterpret_cast<unsigned char*>(c->hook_buf);
  int32_t* dk = reinterpret_cast<int32_t*>(base);
  double* dx0 = reinterpret_cast<double*>(base + ints);
  double *dx = dx0 + xo, *dJ = dx + xo, *de0 = dJ + (size_t)n * n, *dr = de0 + n, *dJe = dr + n;
  OKB_CUDA(c, cudaMemcpyAsync(dk, kind.data(), 4 * nb, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dk + nb, col.data(), 4 * nb, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dk + 2 * nb, off.data(), 4 * nb, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dx0, m->x0, 8 * xo, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dx, x, 8 * xo, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(dJ, m->J, 8 * (size_t)n * n, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaMemcpyAsync(de0, m->e0, 8 * n, cudaMemcpyHostToDevice, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  k_hook_marg<<<1, 256, sizeof(double) * n, c->stream>>>(n, nb, dk, dk + nb, dk + 2 * nb, dx0, dx, dJ, de0, dr, dJe);
  c->launches += 1;
  OKB_CUDA(c, cudaGetLastError());
  if (r) OKB_CUDA(c, cudaMemcpyAsync(r, dr, 8 * n, cudaMemcpyDeviceToHost, c->stream));
  if (J_eff) OKB_CUDA(c, cudaMemcpyAsync(J_eff, dJe, 8 * (size_t)n * n, cudaMemcpyDeviceToHost, c->stream));
  OKB_CUDA(c, cudaStreamSynchronize(c->stream));
  return OKB_OK;
}
