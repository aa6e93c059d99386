// One global-optimisation iteration of GLAMR on sm_100a (global_recon/models/global_recon_model.py:547-570):
//   traj_forward    (1 CTA / person: trajectory codec with two block-wide prefix scans)
//   cam_forward     (1 thread / frame)
//   pose_prep + lbs + joints_finalize   (smpl_kernels.cu: the full SMPL evaluation for every frame-person)
//   frame_residuals (1 thread / frame-person: projection, residuals, analytic gradients, warp-shuffle reductions)
//   camera_backward (1 thread / frame), camera_scatter (mode 3)
//   traj_backward   (1 CTA / person: reverse scans, variable gradients, regularisers)
//   reduce          (loss partials, fixed-camera gradient)   [-> optional NCCL allreduce by the caller]
//   adam            (loss terms + torch.optim.Adam update, step count on device => CUDA-graph capturable)
// No atomics: every sum is a fixed-order tree, so iterations are bit-reproducible.
#include <stdlib.h>
#include <string.h>

#include "globalopt_frames.cuh"
#include "smpl_model.cuh"
#include "block_scan.cuh"

namespace glamr {

constexpr int kFrameThreads = 128;

__device__ void block_reduce_terms(const TermAcc& acc, double* out /*[NUM_TERMS]*/, double* smem /*[warps][NUM_TERMS]*/) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int k = 0; k < GLAMR_NUM_TERMS; ++k) {
    const double s = warp_sum(acc.v[k]);
    if (lane == 0) smem[wid * GLAMR_NUM_TERMS + k] = s;
  }
  __syncthreads();
  if (threadIdx.x < GLAMR_NUM_TERMS) {
    double s = 0.0;
    for (int w = 0; w < nw; ++w) s += smem[w * GLAMR_NUM_TERMS + threadIdx.x];
    out[threadIdx.x] = s;
  }
}

// ------------------------------------------------------------------------------------------------ kernels
// last-block-done ticket: returns true in exactly one CTA of the grid, after all CTAs passed this point
__device__ bool grid_last_block(unsigned int* ticket) {
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int old = atomicAdd(ticket, 1u);
    last = (old == gridDim.x - 1);
    if (last) *ticket = 0u;
  }
  __syncthreads();
  if (last) __threadfence();
  return last;
}

// blocks [0,P): trajectory codec of one person; blocks [P, P+cam_blocks): camera of 256 frames each (modes 0-2)
__global__ void __launch_bounds__(kScanThreads) traj_cam_forward_kernel(OptCtx c, int with_cam) {
  __shared__ float sm[kScanThreads / 32 + 1];
  // [grad | term sums] of this iteration start from zero (the previous iteration's apply has consumed them)
  for (int i = blockIdx.x * kScanThreads + threadIdx.x; i < c.pb.n_params + GLAMR_NUM_TERMS; i += gridDim.x * kScanThreads) c.sc.grad[i] = 0.0f;
  if ((int)blockIdx.x >= c.pb.P) {
    const int t = (blockIdx.x - c.pb.P) * kScanThreads + threadIdx.x;
    if (with_cam && t < c.pb.T) cam_forward(c, t);
    return;
  }
  const int p = blockIdx.x;
  const glamr_person_t& ps = c.pb.persons[p];
  const int len = ps.len, T = c.pb.T;
  const size_t n0 = (size_t)p * T + ps.start;
  for (int i = threadIdx.x; i < len; i += kScanThreads) traj_pre(c, p, i);
  __syncthreads();
  block_scan_inplace(c.sc.heading + n0, len, 1, false, sm);
  __syncthreads();
  for (int i = threadIdx.x; i < len; i += kScanThreads) traj_mid(c, p, i);
  __syncthreads();
  block_scan_inplace(c.sc.xy + 2 * n0, len, 2, false, sm);
  block_scan_inplace(c.sc.xy + 2 * n0 + 1, len, 2, false, sm);
  __syncthreads();
  for (int t = threadIdx.x; t < T; t += kScanThreads) traj_post(c, p, t);
}

__global__ void __launch_bounds__(kFrameThreads) cam_forward_kernel(OptCtx c) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < c.pb.T) cam_forward(c, t);
}

// One warp per frame-person: lanes = joints for the SMPL joint assembly (lib/models/smpl.py:299-315, fused here) and the
// reprojection terms, warp-shuffle sums, then lane 0 finishes the per-frame terms.  4 frame-persons per CTA.
__global__ void __launch_bounds__(kFrameThreads) frame_residuals_kernel(OptCtx c, SmplDev m, SmplWorkspace wo, int n_begin, double* partial) {
  __shared__ double sm[(kFrameThreads / 32) * GLAMR_NUM_TERMS];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int n = blockIdx.x * (kFrameThreads / 32) + wid;
  const int N = c.pb.P * c.pb.T, J = c.pb.J;
  GLAMR_STAMP(0);
  TermAcc acc;
  acc.clear();
  if (n < N) {
    const int p = n / c.pb.T, t = n - p * c.pb.T;
    if (n >= c.pb.n_begin && n < c.pb.n_end) {
      const int nl = n - n_begin;
      const float* tw = c.sc.trans_world + (size_t)n * 3;
      const float sc = c.pb.scale_all ? c.pb.scale_all[n] : 1.0f;
      float root[3], Rc[9], tc[3], Rs[9];
      raw_joint(m, wo, nl, m.joint_map[0], root);
      mat34_R(c.sc.cam + (size_t)t * 12, Rc);
      tc[0] = c.sc.cam[(size_t)t * 12 + 3]; tc[1] = c.sc.cam[(size_t)t * 12 + 7]; tc[2] = c.sc.cam[(size_t)t * 12 + 11];
      rodrigues_smplx(c.sc.orient_world + (size_t)n * 3, Rs);
      KpGrad kg;
      kg.clear();
      GLAMR_STAMP(1);
      for (int k = lane; k < J; k += 32) {
        float v[3], jw[3];
        raw_joint(m, wo, nl, m.joint_map[k], v);
        jw[0] = (v[0] - root[0]) * sc + tw[0];
        jw[1] = (v[1] - root[1]) * sc + tw[1];
        jw[2] = (v[2] - root[2]) * sc + tw[2];
        float* o = c.sc.joints_world + ((size_t)n * J + k) * 3;
        o[0] = jw[0]; o[1] = jw[1]; o[2] = jw[2];
        kp_joint_terms(c, p, t, k, jw, Rc, tc, Rs, tw, kg);
      }
      GLAMR_STAMP(2);
#pragma unroll
      for (int k = 0; k < 3; ++k) { kg.g_tc[k] = warp_sum(kg.g_tc[k]); kg.g_tw[k] = warp_sum(kg.g_tw[k]); }
#pragma unroll
      for (int k = 0; k < 9; ++k) { kg.g_Rc[k] = warp_sum(kg.g_Rc[k]); kg.g_Rs[k] = warp_sum(kg.g_Rs[k]); }
      kg.kp = warp_sum(kg.kp);
      kg.dist = warp_sum(kg.dist);
      GLAMR_STAMP(3);
      if (lane == 0) frame_rest(c, p, t, kg, acc);
      GLAMR_STAMP(10);
    } else if (lane == 0) {
      for (int k = 0; k < 3; ++k) { c.sc.g_orient[(size_t)n * 3 + k] = 0.0f; c.sc.g_trans[(size_t)n * 3 + k] = 0.0f; }
      for (int k = 0; k < 12; ++k) c.sc.g_cam[(size_t)n * 12 + k] = 0.0f;
    }
  }
  if (lane == 0)
    for (int k = 0; k < GLAMR_NUM_TERMS; ++k) sm[wid * GLAMR_NUM_TERMS + k] = acc.v[k];
  __syncthreads();
  if (threadIdx.x < GLAMR_NUM_TERMS) {
    double s = 0.0;
    for (int w = 0; w < kFrameThreads / 32; ++w) s += sm[w * GLAMR_NUM_TERMS + threadIdx.x];
    partial[(size_t)blockIdx.x * GLAMR_NUM_TERMS + threadIdx.x] = s;
  }
  GLAMR_STAMP(11);
}

#ifdef GLAMR_EXPERIMENT
extern "C" int glamr_exp_frame_stamps(long long* out32) {     // experiment build only: the section stamps of two CTAs of the last launch
  GLAMR_CUDA_TRY(cudaDeviceSynchronize());
  GLAMR_CUDA_TRY(cudaMemcpyFromSymbol(out32, g_frame_stamps, sizeof(long long) * 32));
  return GLAMR_OK;
}
#endif

__global__ void __launch_bounds__(kFrameThreads) camera_backward_kernel(OptCtx c, double* partial) {
  __shared__ double sm[(kFrameThreads / 32) * GLAMR_NUM_TERMS];
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  TermAcc acc;
  acc.clear();
  if (t < c.pb.T) camera_backward(c, t, acc);
  block_reduce_terms(acc, partial + (size_t)blockIdx.x * GLAMR_NUM_TERMS, sm);
}

__global__ void __launch_bounds__(kFrameThreads) camera_scatter_kernel(OptCtx c) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < c.pb.T) camera_scatter_to_persons(c, s);
}

// ---- cross-GPU reduction over NVLink peer memory (one process per GPU, buffers exchanged as CUDA IPC handles) --------
// Every rank owns one buffer: [64 x u32 header | 2 slots x W sources x slot_elems x u64].  Header words: 0 = epochs
// published by this rank, 1 = epochs consumed, 2 = error.  Flag-in-data protocol (no fences, which cost tens of
// microseconds at system scope): iteration e (1-based, never reset) -- the last CTA of traj_cam_backward_kernel packs every
// element of [grad | term sums] with the epoch into one 8-byte word {value, e} and PUSHES it into slot e & 1, source row
// `rank`, of every rank's buffer (plain 8-byte stores over NVLink: value and tag arrive together); apply_kernel polls its
// OWN memory until the word of each source carries tag e and sums the W values in rank order -- the same bits on every
// rank.  (Both halves live in apply_kernel: every thread pushes the elements it owns, then polls for them.)  Two slots suffice: a rank can be at most one iteration ahead of the slowest reader (its next apply needs that
// reader's next push), so epoch e only ever overwrites epoch e - 2, which every rank has finished reading.
struct PeerCtx {
  int rank, world;
  size_t slot_elems;                       // 8-byte words per (slot, source)
  unsigned long long* bufs[GLAMR_MAX_PEERS];
};
constexpr int kPeerHeaderWords = 64;      // u32 words = 32 u64

__device__ __forceinline__ void st_peer_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_peer_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ size_t peer_row(const PeerCtx& pc, uint32_t e, int src) {
  return kPeerHeaderWords / 2 + ((size_t)(e & 1u) * GLAMR_MAX_PEERS + src) * pc.slot_elems;
}
// value of element i published by rank `src` for epoch e (spins on local memory until it has landed)
__device__ __forceinline__ float peer_take(const PeerCtx& pc, uint32_t e, int src, int i) {
  const unsigned long long* p = pc.bufs[pc.rank] + peer_row(pc, e, src) + i;
  unsigned long long w = ld_peer_u64(p);
  if ((uint32_t)(w >> 32) != e) {
    const long long t0 = clock64();
    do {
      if (clock64() - t0 > 40000000000LL) {          // ~20 s: a rank died or left the loop; fail loudly instead of hanging the GPU
        reinterpret_cast<uint32_t*>(pc.bufs[pc.rank])[2] = 1u;
        __trap();
      }
      w = ld_peer_u64(p);
    } while ((uint32_t)(w >> 32) != e);
  }
  return __uint_as_float((uint32_t)w);
}

// loss partials -> un-normalised term sums (reduce_buf tail); fixed camera: sum the per-frame gradients over T
__device__ void reduce_tail(const OptCtx& c, const double* partial, int n_slots, float* reduce_buf, double* sm /*[8*16]*/) {
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid < GLAMR_NUM_TERMS) {
    double s = 0.0;
    for (int k = 0; k < n_slots; ++k) s += partial[(size_t)k * GLAMR_NUM_TERMS + tid];
    reduce_buf[c.pb.n_params + tid] = (float)s;
  }
  if (c.pb.cam_mode == GLAMR_CAM_FIXED) {
    double a[9];
    for (int k = 0; k < 9; ++k) a[k] = 0.0;
    for (int t = tid; t < c.pb.T; t += blockDim.x)
      for (int k = 0; k < 9; ++k) a[k] += (double)c.sc.g_cam_fix[(size_t)t * 12 + k];
    for (int k = 0; k < 9; ++k) {
      const double s = warp_sum(a[k]);
      if (lane == 0) sm[wid * 16 + k] = s;
    }
    __syncthreads();
    if (tid < 9) {
      double s = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sm[w * 16 + tid];
      const int off = (tid < 6) ? c.pb.off_cam_rot + tid : c.pb.off_cam_trans + (tid - 6);
      reduce_buf[off] = (float)s;
    }
  }
}

// blocks [0,P): reverse trajectory codec of one person; blocks [P, P+cam_blocks): camera backward of 256 frames (modes
// 0-2; mode 3 runs camera_backward/scatter kernels first).  The last CTA to finish folds all partial sums.
__global__ void __launch_bounds__(kScanThreads) traj_cam_backward_kernel(OptCtx c, int with_cam, double* partial_traj, const double* partial_all,
                                                                         int n_slots, float* reduce_buf, unsigned int* ticket, PeerCtx pc) {
  __shared__ float sm[kScanThreads / 32 + 1];
  __shared__ double smd[(kScanThreads / 32) * GLAMR_NUM_TERMS];
  TermAcc acc;
  acc.clear();
  if ((int)blockIdx.x >= c.pb.P) {
    const int t = (blockIdx.x - c.pb.P) * kScanThreads + threadIdx.x;
    if (with_cam && t < c.pb.T) camera_backward(c, t, acc);
  } else {
    const int p = blockIdx.x;
    const glamr_person_t& ps = c.pb.persons[p];
    const int len = ps.len, T = c.pb.T;
    const size_t n0 = (size_t)p * T + ps.start;
    for (int t = threadIdx.x; t < T; t += kScanThreads) traj_back_pre(c, p, t, acc);
    __syncthreads();
    block_scan_inplace(c.sc.g_xy + 2 * n0, len, 2, true, sm);
    block_scan_inplace(c.sc.g_xy + 2 * n0 + 1, len, 2, true, sm);
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += kScanThreads) traj_back_mid(c, p, i, acc);
    __syncthreads();
    block_scan_inplace(c.sc.g_head + n0, len, 1, true, sm);
    __syncthreads();
    for (int i = threadIdx.x; i < len; i += kScanThreads) traj_back_post(c, p, i, acc);
  }
  block_reduce_terms(acc, partial_traj + (size_t)blockIdx.x * GLAMR_NUM_TERMS, smd);
  if (grid_last_block(ticket)) {
    reduce_tail(c, partial_all, n_slots, reduce_buf, smd);
  }
}

// Stand-alone sum all-reduce of `count` floats over the peer buffers (same push-then-poll protocol and epoch counter as the
// reduction inside apply_kernel): buf <- sum over ranks, identical bits on every rank.
__global__ void __launch_bounds__(256) peer_allreduce_kernel(PeerCtx pc, float* __restrict__ buf, int count, unsigned int* ticket) {
  const uint32_t epoch = reinterpret_cast<const uint32_t*>(pc.bufs[pc.rank])[1] + 1u;
  const size_t row = peer_row(pc, epoch, pc.rank);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    const unsigned long long w = ((unsigned long long)epoch << 32) | (unsigned long long)__float_as_uint(buf[i]);
    for (int r = 0; r < pc.world; ++r) st_peer_u64(pc.bufs[r] + row + i, w);
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
    float g = 0.0f;
    for (int r = 0; r < pc.world; ++r) g += peer_take(pc, epoch, r, i);
    buf[i] = g;
  }
  if (grid_last_block(ticket) && threadIdx.x == 0) reinterpret_cast<uint32_t*>(pc.bufs[pc.rank])[1] = epoch;
}

struct AdamState {
  float* m;
  float* v;
  double* beta_pow;   // [0] beta1^t, [1] beta2^t, [2] step count (as a double)
};

__device__ void write_losses(const OptCtx& c, const float* term_sums /*[NUM_TERMS] un-normalised*/, float* loss_terms) {
  double total = 0.0;
  for (int k = 0; k < GLAMR_NUM_TERMS; ++k) {
    float val = 0.0f;
    if (c.pb.term_enabled[k]) {
      val = term_sums[k] / c.pb.term_norm[k];
      if (!c.pb.term_monitor[k]) total += (double)val * (double)c.pb.term_weight[k];
    }
    loss_terms[k] = val;
  }
  loss_terms[GLAMR_NUM_TERMS] = (float)total;
}

__global__ void __launch_bounds__(32) losses_kernel(OptCtx c, const float* __restrict__ reduce_buf, float* __restrict__ loss_terms) {
  if (threadIdx.x == 0) write_losses(c, reduce_buf + c.pb.n_params, loss_terms);
}

// loss terms (block 0) + torch.optim.Adam step; the last CTA to finish advances the step count / beta powers.
// pc.world > 1: the gradient is the rank-ordered sum of every GPU's published slot (peer memory), not reduce_buf.
__global__ void __launch_bounds__(256) apply_kernel(OptCtx c, float* __restrict__ theta, const float* __restrict__ reduce_buf, double lr,
                                                    AdamState ad, float* loss_terms, int hist_stride, unsigned int* ticket, PeerCtx pc) {
  const double b1 = ad.beta_pow[0] * 0.9, b2 = ad.beta_pow[1] * 0.999, step = ad.beta_pow[2];
  const uint32_t epoch = pc.world > 1 ? reinterpret_cast<const uint32_t*>(pc.bufs[pc.rank])[1] + 1u : 0u;
  if (pc.world > 1) {
    // one-shot all-reduce over NVLink, part 1: every thread PUSHES its own elements of this rank's [grad | term sums], tagged
    // with the iteration number in the same 8-byte word, into slot (epoch & 1), source row `rank`, of every rank's buffer.  All
    // pushes of a rank are issued before any of its threads starts polling, so ranks never wait on each other circularly.
    const size_t row = peer_row(pc, epoch, pc.rank);
    const int count = c.pb.n_params + GLAMR_NUM_TERMS;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
      const unsigned long long w = ((unsigned long long)epoch << 32) | (unsigned long long)__float_as_uint(reduce_buf[i]);
      for (int r = 0; r < pc.world; ++r) st_peer_u64(pc.bufs[r] + row + i, w);
    }
  }
  // part 2: a thread polls its OWN memory until the word of each source carries this iteration's tag and sums in rank order
  auto grad_at = [&](int i) -> float {
    if (pc.world <= 1) return reduce_buf[i];
    float g = 0.0f;
    for (int r = 0; r < pc.world; ++r) g += peer_take(pc, epoch, r, i);
    return g;
  };
  if (blockIdx.x == 0 && threadIdx.x == 0 && loss_terms) {
    float sums[GLAMR_NUM_TERMS];
    for (int k = 0; k < GLAMR_NUM_TERMS; ++k) sums[k] = grad_at(c.pb.n_params + k);
    write_losses(c, sums, loss_terms + (hist_stride > 0 ? (size_t)step * hist_stride : 0));
  }
  const float bc2s = (float)sqrt(1.0 - b2);
  const float step_size = (float)(lr / (1.0 - b1));
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < c.pb.n_params; i += gridDim.x * blockDim.x) {
    if (!c.pb.active[i]) continue;
    const float g = grad_at(i);
    float m = ad.m[i], v = ad.v[i];
    m = m + 0.1f * (g - m);
    v = v * 0.999f + 0.001f * g * g;
    const float denom = sqrtf(v) / bc2s + 1e-8f;
    theta[i] = theta[i] - step_size * (m / denom);
    ad.m[i] = m;
    ad.v[i] = v;
  }
  if (grid_last_block(ticket) && threadIdx.x == 0) {
    ad.beta_pow[0] = b1;
    ad.beta_pow[1] = b2;
    ad.beta_pow[2] = step + 1.0;
    if (pc.world > 1) reinterpret_cast<uint32_t*>(pc.bufs[pc.rank])[1] = epoch;
  }
}
}  // namespace glamr

using namespace glamr;

struct glamr_opt {
  SmplDev smpl;
  glamr_problem_t pb;
  OptScratch sc;
  SmplWorkspace ws;
  AdamState adam;
  double* partial;
  int n_slots, slots_res, slots_cam, cam_blocks;   // partial-sum slots: residual CTAs | P + cam_blocks (traj/cam kernel) | slots_cam (mode 3)
  unsigned int* tickets;                           // [0] backward tail, [1] apply, [3] stand-alone peer all-reduce
  void* arena;
  size_t arena_bytes;
  float gs[GLAMR_NUM_TERMS];
  int timing;                 // != 0: bracket the LBS kernel with events (bench / roofline only, not graph-capturable)
  cudaEvent_t ev_lbs0, ev_lbs1, ev_blend0, ev_blend1;
  // tensor-core LBS, software-pipelined: the blend GEMM of the NEXT evaluation runs on `aux` concurrently with the residual /
  // backward kernels of this one (it depends on body pose and betas only); `vpt_ready` says the workspace holds a valid v_posed
  cudaStream_t aux;
  cudaEvent_t ev_fork, ev_join;
  int vpt_ready;
  int join_pending;           // a glamr_opt_backward_for_apply call left the side stream un-joined (the next call on the handle joins)
  int features_early;         // the pipelined blend's feature kernel runs at the top of the evaluation
  cudaEvent_t ev[24];         // timing == 2: one event after every launch of glamr_opt_backward / glamr_opt_apply
  int n_ev;
  // glamr_opt_iterate: one captured iteration (backward + apply), valid for the arguments it was captured with
  cudaStream_t cap_stream;
  cudaGraphExec_t iter_exec;
  const void* cap_theta; const void* cap_reduce; const void* cap_hist;
  double cap_lr; int cap_stride; unsigned long long cap_gen, gen;   // gen advances with every glamr_opt_set_problem
  PeerCtx peer;               // world <= 1: single GPU (or the caller reduces reduce_buf itself between backward and apply)
};

extern "C" size_t glamr_sizeof_person(void) { return sizeof(glamr_person_t); }
extern "C" size_t glamr_sizeof_problem(void) { return sizeof(glamr_problem_t); }

static void compute_gs(glamr_opt* st) {
  for (int k = 0; k < GLAMR_NUM_TERMS; ++k) {
    const glamr_problem_t& pb = st->pb;
    st->gs[k] = (pb.term_enabled[k] && !pb.term_monitor[k] && pb.term_norm[k] != 0.0f) ? pb.term_weight[k] / pb.term_norm[k] : 0.0f;
  }
}
static OptCtx make_ctx(const glamr_opt* st, const float* theta, float* grad) {
  OptCtx c;
  c.pb = st->pb;
  c.sc = st->sc;
  c.sc.grad = grad;
  c.theta = theta;
  for (int k = 0; k < GLAMR_NUM_TERMS; ++k) c.gs[k] = st->gs[k];
  return c;
}

extern "C" int glamr_opt_create(glamr_opt_t** out, const glamr_smpl_t* smpl, const glamr_problem_t* pb) {
  if (!out || !smpl || !pb || pb->P <= 0 || pb->T <= 0 || pb->J <= 0 || pb->n_params <= 0) return GLAMR_EINVAL;
  if (pb->J != smpl->dev.n_map) return GLAMR_EINVAL;
  glamr_opt* st = (glamr_opt*)calloc(1, sizeof(glamr_opt));
  if (!st) return GLAMR_EINVAL;
  st->smpl = smpl->dev;
  st->pb = *pb;
  compute_gs(st);
  const size_t N = (size_t)pb->P * pb->T, T = pb->T, J = pb->J;
  st->slots_res = (int)((N + kFrameThreads / 32 - 1) / (kFrameThreads / 32));
  st->slots_cam = (int)((T + kFrameThreads - 1) / kFrameThreads);
  st->cam_blocks = (int)((T + kScanThreads - 1) / kScanThreads);
  st->n_slots = st->slots_res + pb->P + st->cam_blocks + st->slots_cam;
  // one arena for all scratch (floats), doubles first for alignment
  size_t floats = 0;
  auto take = [&](size_t nfl) { size_t o = floats; floats += (nfl + 63) & ~(size_t)63; return o; };
  const size_t o_partial = take((size_t)st->n_slots * GLAMR_NUM_TERMS * 2);
  const size_t o_beta = take(8);
  const size_t o_ticket = take(8);
  const size_t o_heading = take(N), o_xy = take(2 * N), o_tl = take(11 * N), o_ob = take(3 * N), o_tb = take(3 * N),
               o_ow = take(3 * N), o_tw = take(3 * N), o_cam = take(12 * T), o_caminv = take(12 * T), o_camd6 = take(6 * T),
               o_jw = take(N * J * 3), o_kp = take(N * J * 2), o_ociw = take(3 * N), o_tciw = take(3 * N), o_go = take(3 * N),
               o_gt = take(3 * N), o_gcam = take(12 * N), o_gcf = take(12 * T), o_gxy = take(2 * N), o_gh = take(N),
               o_m = take(pb->n_params), o_v = take(pb->n_params);
  const size_t o_ws = take(smpl_workspace_floats((int)N, smpl->dev.S));
  {
    // the feature kernel of the pipelined blend (its A operand; body pose / betas only) runs at the top of the evaluation on the side
    // stream, so that only the GEMM is left after the skinning -- only while this rank's per-frame kernels have fewer CTAs than the GPU
    // has SMs: measured 102.8 -> 94.8 us per L2-flushed iteration at 1 x 300, but 154 -> 180 us at 4 x 300, where the GEMM then no
    // longer follows a kernel with its own shared-memory split
    int sms = 148, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int frame_ctas = (pb->n_end - pb->n_begin + kFrameThreads / 32 - 1) / (kFrameThreads / 32);
    st->features_early = frame_ctas < sms;
  }
  st->arena_bytes = floats * sizeof(float);
  cudaError_t e = cudaMalloc(&st->arena, st->arena_bytes);
  if (e != cudaSuccess) { free(st); return (int)e; }
  e = cudaMemset(st->arena, 0, st->arena_bytes);
  if (e != cudaSuccess) { cudaFree(st->arena); free(st); return (int)e; }
  float* b = (float*)st->arena;
  st->partial = (double*)(b + o_partial);
  st->adam.beta_pow = (double*)(b + o_beta);
  st->tickets = (unsigned int*)(b + o_ticket);
  st->sc.heading = b + o_heading; st->sc.xy = b + o_xy; st->sc.traj_local = b + o_tl; st->sc.orient_base = b + o_ob;
  st->sc.trans_base = b + o_tb; st->sc.orient_world = b + o_ow; st->sc.trans_world = b + o_tw; st->sc.cam = b + o_cam;
  st->sc.cam_inv = b + o_caminv; st->sc.cam_d6 = b + o_camd6; st->sc.joints_world = b + o_jw; st->sc.kp_pred = b + o_kp;
  st->sc.orient_ciw = b + o_ociw; st->sc.trans_ciw = b + o_tciw; st->sc.g_orient = b + o_go; st->sc.g_trans = b + o_gt;
  st->sc.g_cam = b + o_gcam; st->sc.g_cam_fix = b + o_gcf; st->sc.g_xy = b + o_gxy; st->sc.g_head = b + o_gh;
  st->sc.grad = nullptr;
  st->adam.m = b + o_m; st->adam.v = b + o_v;
  st->ws = smpl_carve_workspace(b + o_ws, (int)N, smpl->dev.S);
  const double one[3] = {1.0, 1.0, 0.0};
  e = cudaMemcpy(st->adam.beta_pow, one, sizeof(one), cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { cudaFree(st->arena); free(st); return (int)e; }
  *out = st;
  return GLAMR_OK;
}

extern "C" int glamr_opt_kernel_timing(glamr_opt_t* st, int enable) {
  if (!st) return GLAMR_EINVAL;
  if (enable && !st->ev_lbs0) {
    GLAMR_CUDA_TRY(cudaEventCreate(&st->ev_lbs0));
    GLAMR_CUDA_TRY(cudaEventCreate(&st->ev_lbs1));
    GLAMR_CUDA_TRY(cudaEventCreate(&st->ev_blend0));
    GLAMR_CUDA_TRY(cudaEventCreate(&st->ev_blend1));
    for (int i = 0; i < 24; ++i) GLAMR_CUDA_TRY(cudaEventCreate(&st->ev[i]));
  }
  st->timing = enable;
  return GLAMR_OK;
}

extern "C" int glamr_opt_last_lbs_ms(glamr_opt_t* st, float* ms) {
  if (!st || !ms || !st->ev_lbs0) return GLAMR_EINVAL;
  GLAMR_CUDA_TRY(cudaEventSynchronize(st->ev_lbs1));
  GLAMR_CUDA_TRY(cudaEventElapsedTime(ms, st->ev_lbs0, st->ev_lbs1));
  if (st->vpt_ready && st->aux) {            // tensor-core path: + the blend GEMM (timed on its own stream) = the whole LBS
    float b = 0.0f;
    GLAMR_CUDA_TRY(cudaEventSynchronize(st->ev_blend1));
    GLAMR_CUDA_TRY(cudaEventElapsedTime(&b, st->ev_blend0, st->ev_blend1));
    *ms += b;
  }
  return GLAMR_OK;
}

// The two parts of the last timed evaluation separately: the kernel on the iteration's critical path (skinning on the tensor-core
// path, the whole LBS kernel on the SIMT path) and the blend on its side stream (0 on the SIMT path).
extern "C" int glamr_opt_last_lbs_parts_ms(glamr_opt_t* st, float* critical_ms, float* blend_ms) {
  if (!st || !critical_ms || !blend_ms || !st->ev_lbs0) return GLAMR_EINVAL;
  GLAMR_CUDA_TRY(cudaEventSynchronize(st->ev_lbs1));
  GLAMR_CUDA_TRY(cudaEventElapsedTime(critical_ms, st->ev_lbs0, st->ev_lbs1));
  *blend_ms = 0.0f;
  if (st->vpt_ready && st->aux) {
    GLAMR_CUDA_TRY(cudaEventSynchronize(st->ev_blend1));
    GLAMR_CUDA_TRY(cudaEventElapsedTime(blend_ms, st->ev_blend0, st->ev_blend1));
  }
  return GLAMR_OK;
}

// Measurement hook: the blend (features + tensor-core GEMM) of this rank's frame-persons ALONE on its side stream, `reps` launches
// bracketed by one event pair -> mean ms per launch.  Synchronises.  (In the iteration the blend overlaps other kernels, so its
// in-situ duration says little about the kernel itself.)
extern "C" int glamr_opt_time_blend(glamr_opt_t* st, int reps, float* ms) {
  if (!st || !ms || reps <= 0) return GLAMR_EINVAL;
  if (lbs_path() < 1 || !st->smpl.tcB || !st->aux) return GLAMR_EUNSUPPORTED;
  const glamr_problem_t& pb = st->pb;
  const int nn = pb.n_end - pb.n_begin;
  if (nn <= 0) return GLAMR_EINVAL;
  cudaEvent_t e0, e1;
  GLAMR_CUDA_TRY(cudaEventCreate(&e0));
  GLAMR_CUDA_TRY(cudaEventCreate(&e1));
  GLAMR_CUDA_TRY(cudaDeviceSynchronize());
  GLAMR_CUDA_TRY(cudaEventRecord(e0, st->aux));
  int rc = GLAMR_OK;
  for (int i = 0; i < reps && rc == GLAMR_OK; ++i)
    rc = launch_blend(st->smpl, nn, pb.smpl_pose_all + (size_t)pb.n_begin * 69, pb.smpl_beta_all + (size_t)pb.n_begin * kNB, st->ws, st->aux);
  cudaEventRecord(e1, st->aux);
  cudaEventSynchronize(e1);
  float t = 0.0f;
  cudaEventElapsedTime(&t, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *ms = t / reps;
  return rc;
}

// timing == 2: durations (ms) between consecutive marks of the last glamr_opt_backward (+ apply) call sequence
extern "C" int glamr_opt_kernel_times(glamr_opt_t* st, float* ms, int* n) {
  if (!st || !ms || !n || !st->ev_lbs0) return GLAMR_EINVAL;
  if (st->n_ev < 2) { *n = 0; return GLAMR_OK; }
  GLAMR_CUDA_TRY(cudaEventSynchronize(st->ev[st->n_ev - 1]));
  for (int i = 0; i + 1 < st->n_ev; ++i) GLAMR_CUDA_TRY(cudaEventElapsedTime(&ms[i], st->ev[i], st->ev[i + 1]));
  *n = st->n_ev - 1;
  return GLAMR_OK;
}

extern "C" int glamr_opt_destroy(glamr_opt_t* st) {
  if (st && st->iter_exec) cudaGraphExecDestroy(st->iter_exec);
  if (st && st->cap_stream) cudaStreamDestroy(st->cap_stream);
  if (!st) return GLAMR_OK;
  if (st->ev_lbs0) { cudaEventDestroy(st->ev_lbs0); cudaEventDestroy(st->ev_lbs1); cudaEventDestroy(st->ev_blend0); cudaEventDestroy(st->ev_blend1); for (int i = 0; i < 24; ++i) cudaEventDestroy(st->ev[i]); }
  if (st->aux) { cudaStreamSynchronize(st->aux); cudaStreamDestroy(st->aux); cudaEventDestroy(st->ev_fork); cudaEventDestroy(st->ev_join); }
  cudaFree(st->arena);
  free(st);
  return GLAMR_OK;
}

static int join_pending(glamr_opt_t* st, cudaStream_t s);

extern "C" int glamr_opt_set_problem(glamr_opt_t* st, const glamr_problem_t* pb, int reset_adam, void* stream) {
  if (!st || !pb) return GLAMR_EINVAL;
  if (pb->P != st->pb.P || pb->T != st->pb.T || pb->J != st->pb.J || pb->n_params != st->pb.n_params) return GLAMR_EINVAL;
  {
    const int rc = join_pending(st, (cudaStream_t)stream);
    if (rc) return rc;
  }
  st->pb = *pb;
  st->gen++;
  compute_gs(st);
  if (reset_adam & 2) {      // handle re-used for a new sequence: scratch (incl. tickets, moments) back to its initial zeros
    if (st->aux) GLAMR_CUDA_TRY(cudaStreamSynchronize(st->aux));
    st->vpt_ready = 0;       // new body poses: the pipelined blend has to be primed again
    GLAMR_CUDA_TRY(cudaMemsetAsync(st->arena, 0, st->arena_bytes, (cudaStream_t)stream));
    reset_adam |= 1;
  }
  if (reset_adam & 1) {
    cudaStream_t s = (cudaStream_t)stream;
    GLAMR_CUDA_TRY(cudaMemsetAsync(st->adam.m, 0, sizeof(float) * pb->n_params, s));
    GLAMR_CUDA_TRY(cudaMemsetAsync(st->adam.v, 0, sizeof(float) * pb->n_params, s));
    static const double one[3] = {1.0, 1.0, 0.0};
    GLAMR_CUDA_TRY(cudaMemcpyAsync(st->adam.beta_pow, one, sizeof(one), cudaMemcpyHostToDevice, s));
  }
  return GLAMR_OK;
}

extern "C" size_t glamr_opt_reduce_count(const glamr_opt_t* st) { return st ? (size_t)st->pb.n_params + GLAMR_NUM_TERMS : 0; }

extern "C" int glamr_opt_launch_count(const glamr_opt_t* st) {
  if (!st) return GLAMR_EINVAL;
  const bool from_persons = st->pb.cam_mode == GLAMR_CAM_FROM_PERSONS;
  const bool has_frames = st->pb.n_end > st->pb.n_begin;
  const int fwd = 1 + (from_persons ? 1 : 0) + (has_frames ? 1 + (lbs_kernel_count(st->smpl) == 2 ? 3 : 1) : 0);     // forward [+ cam_forward] [+ pose_prep + lbs]
  return fwd + 1 + (from_persons ? 2 : 0) + 1 + 1;                       // residuals [+ camera backward + scatter] + traj/cam backward + apply
}

#define GLAMR_MARK() do { if (st->timing == 2 && st->n_ev < 24) GLAMR_CUDA_TRY(cudaEventRecord(st->ev[st->n_ev++], s)); } while (0)

// the side stream's work of an earlier evaluation whose join was left to the next call on the handle
static int join_pending(glamr_opt_t* st, cudaStream_t s) {
  if (st->join_pending) {
    GLAMR_CUDA_TRY(cudaStreamWaitEvent(s, st->ev_join, 0));
    st->join_pending = 0;
  }
  return GLAMR_OK;
}

// defer_join: the caller runs glamr_opt_apply on the same handle next (possibly after an exchange of reduce_buf): the pipelined blend on the
// side stream is joined there, so that the exchange overlaps its tail instead of waiting for it
static int backward_impl(glamr_opt_t* st, const float* theta, float* reduce_buf, void* stream, bool use_peers, bool defer_join = false) {
  if (!st || !theta || !reduce_buf) return GLAMR_EINVAL;
  PeerCtx pc = st->peer;
  if (!use_peers) pc.world = 0;
  cudaStream_t s = (cudaStream_t)stream;
  {
    const int rc = join_pending(st, s);
    if (rc) return rc;
  }
  st->n_ev = 0;
  GLAMR_MARK();
  const glamr_problem_t& pb = st->pb;
  OptCtx c = make_ctx(st, theta, reduce_buf);
  const bool from_persons = pb.cam_mode == GLAMR_CAM_FROM_PERSONS;
  // SMPL for the frame-persons this rank owns (global_recon_model.py:517-524); tile-major scratch (A, pf) is local to the launch
  const int n_begin = pb.n_begin, n_end = pb.n_end;
  SmplWorkspace wo = st->ws;
  wo.jposed += (size_t)n_begin * kNJ * 3;
  wo.vcompact += (size_t)n_begin * st->smpl.S * 3;
  wo.root_raw += (size_t)n_begin * 3;
  const bool tc = lbs_path() >= 1 && st->smpl.tcB != nullptr;
  SmplWorkspace wo_pose = wo;
  if (tc) {
    wo_pose.tcA = nullptr;                   // the features belong to blend_features_kernel (side stream); pose prep must not rewrite them
    if (!st->aux) {
      GLAMR_CUDA_TRY(cudaStreamCreateWithFlags(&st->aux, cudaStreamNonBlocking));
      GLAMR_CUDA_TRY(cudaEventCreateWithFlags(&st->ev_fork, cudaEventDisableTiming));
      GLAMR_CUDA_TRY(cudaEventCreateWithFlags(&st->ev_join, cudaEventDisableTiming));
    }
  }
  bool forked = false;
#ifdef GLAMR_EXPERIMENT
  // experiment build only (tools/iter_skip_exp.py): GLAMR_EXP_SKIP bit 1 = no pipelined blend, 2 = no skinning, 4 = no residual kernel, 8 = no backward kernel
  static const int exp_skip = getenv("GLAMR_EXP_SKIP") ? atoi(getenv("GLAMR_EXP_SKIP")) : 0;
#else
  constexpr int exp_skip = 0;
#endif
  const float* const pose_l = pb.smpl_pose_all + (size_t)n_begin * 69;
  const float* const beta_l = pb.smpl_beta_all + (size_t)n_begin * kNB;
  // the blend of the NEXT evaluation (it depends on body pose / betas only): side stream, concurrent with this evaluation.  With
  // features_early its feature kernel is forked at the top and the GEMM after the skinning (which must have read v_posed first);
  // otherwise both are forked after the skinning.
  const int nn = n_end - n_begin;
  const bool features_early = st->features_early && !st->timing;
  auto fork = [&]() -> int {
    GLAMR_CUDA_TRY(cudaEventRecord(st->ev_fork, s));
    GLAMR_CUDA_TRY(cudaStreamWaitEvent(st->aux, st->ev_fork, 0));
    return GLAMR_OK;
  };
  if (tc && nn > 0) {
    int rc;
    if (!st->vpt_ready) {                 // first evaluation after create / a new sequence: v_posed is filled in order
      if ((rc = launch_blend(st->smpl, nn, pose_l, beta_l, wo, s))) return rc;
      st->vpt_ready = 1;
    }
    if (features_early) {
      if ((rc = fork())) return rc;
      if (!(exp_skip & 1))
        if ((rc = launch_blend_features(nn, pose_l, beta_l, wo, st->aux))) return rc;
    }
  }
  traj_cam_forward_kernel<<<pb.P + st->cam_blocks, kScanThreads, 0, s>>>(c, from_persons ? 0 : 1);   // also zeroes reduce_buf
  GLAMR_LAUNCH_CHECK();
  GLAMR_MARK();
  if (from_persons) {          // the camera is the mean of the persons' world transforms: needs traj_forward of all persons
    cam_forward_kernel<<<st->slots_cam, kFrameThreads, 0, s>>>(c);
    GLAMR_LAUNCH_CHECK();
  }
  GLAMR_MARK();
  if (nn > 0) {
    int rc;
    if ((rc = launch_pose_prep(st->smpl, nn, st->sc.orient_world + (size_t)n_begin * 3, pose_l, beta_l, 1, wo_pose, s))) return rc;
    GLAMR_MARK();
    if (st->timing) GLAMR_CUDA_TRY(cudaEventRecord(st->ev_lbs0, s));
    if (tc) {
      if (!(exp_skip & 2))
        if ((rc = launch_skin(st->smpl, nn, wo, nullptr, s))) return rc;
      if (st->timing) GLAMR_CUDA_TRY(cudaEventRecord(st->ev_lbs1, s));
      if ((rc = fork())) return rc;
      if (st->timing) GLAMR_CUDA_TRY(cudaEventRecord(st->ev_blend0, st->aux));
      if (!(exp_skip & 1)) {
        if (!features_early)
          if ((rc = launch_blend_features(nn, pose_l, beta_l, wo, st->aux))) return rc;
        if ((rc = launch_blend_gemm(st->smpl, nn, wo, st->aux))) return rc;
      }
      if (st->timing) GLAMR_CUDA_TRY(cudaEventRecord(st->ev_blend1, st->aux));
      GLAMR_CUDA_TRY(cudaEventRecord(st->ev_join, st->aux));
      forked = true;
    } else {
      if ((rc = launch_lbs(st->smpl, 0, nn, beta_l, wo, nullptr, s))) return rc;
      if (st->timing) GLAMR_CUDA_TRY(cudaEventRecord(st->ev_lbs1, s));
    }
    GLAMR_MARK();
  }
  double* part_res = st->partial;
  double* part_traj = st->partial + (size_t)st->slots_res * GLAMR_NUM_TERMS;
  double* part_cam3 = part_traj + (size_t)(pb.P + st->cam_blocks) * GLAMR_NUM_TERMS;
  if (!(exp_skip & 4)) {
    frame_residuals_kernel<<<st->slots_res, kFrameThreads, 0, s>>>(c, st->smpl, wo, n_begin, part_res);
    GLAMR_LAUNCH_CHECK();
  }
  GLAMR_MARK();
  if (from_persons) {
    camera_backward_kernel<<<st->slots_cam, kFrameThreads, 0, s>>>(c, part_cam3);
    GLAMR_LAUNCH_CHECK();
    camera_scatter_kernel<<<st->slots_cam, kFrameThreads, 0, s>>>(c);
    GLAMR_LAUNCH_CHECK();
    GLAMR_MARK();
  }
  const int n_slots = st->slots_res + pb.P + st->cam_blocks + (from_persons ? st->slots_cam : 0);
  if (!(exp_skip & 8)) {
    traj_cam_backward_kernel<<<pb.P + st->cam_blocks, kScanThreads, 0, s>>>(c, from_persons ? 0 : 1, part_traj, (const double*)st->partial, n_slots,
                                                                            reduce_buf, st->tickets, pc);
    GLAMR_LAUNCH_CHECK();
  }
  GLAMR_MARK();
  if (forked) {
    if (defer_join) st->join_pending = 1;
    else GLAMR_CUDA_TRY(cudaStreamWaitEvent(s, st->ev_join, 0));      // the side stream rejoins before the evaluation ends
  }
  return GLAMR_OK;
}
extern "C" int glamr_opt_backward(glamr_opt_t* st, const float* theta, float* reduce_buf, void* stream) {
  return backward_impl(st, theta, reduce_buf, stream, false);
}
// The first half of an iteration whose second half is glamr_opt_apply on the same stream (with the caller's exchange of reduce_buf in
// between): same work as glamr_opt_backward, but the side-stream blend of the next evaluation is joined by that apply call (or by the next
// call on the handle), so the exchange runs next to its tail.
extern "C" int glamr_opt_backward_for_apply(glamr_opt_t* st, const float* theta, float* reduce_buf, void* stream) {
  return backward_impl(st, theta, reduce_buf, stream, false, true);
}

extern "C" int glamr_opt_losses(glamr_opt_t* st, const float* reduce_buf, float* loss_terms, void* stream) {
  if (!st || !reduce_buf || !loss_terms) return GLAMR_EINVAL;
  OptCtx c = make_ctx(st, nullptr, nullptr);
  losses_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(c, reduce_buf, loss_terms);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}

static int apply_impl(glamr_opt_t* st, float* theta, const float* reduce_buf, double lr, float* loss_terms, int loss_hist_stride,
                      void* stream, bool use_peers) {
  if (!st || !theta || !reduce_buf) return GLAMR_EINVAL;
  PeerCtx pc = st->peer;
  if (!use_peers) pc.world = 0;
  cudaStream_t s = (cudaStream_t)stream;
  {
    const int rc = join_pending(st, s);
    if (rc) return rc;
  }
  OptCtx c = make_ctx(st, theta, nullptr);
  const int blocks = (st->pb.n_params + 255) / 256;
  apply_kernel<<<blocks < 296 ? blocks : 296, 256, 0, s>>>(c, theta, reduce_buf, lr, st->adam, loss_terms, loss_hist_stride, st->tickets + 1, pc);
  GLAMR_LAUNCH_CHECK();
  GLAMR_MARK();
  return GLAMR_OK;
}
extern "C" int glamr_opt_apply(glamr_opt_t* st, float* theta, const float* reduce_buf, double lr, float* loss_terms,
                               int loss_hist_stride, void* stream) {
  return apply_impl(st, theta, reduce_buf, lr, loss_terms, loss_hist_stride, stream, false);
}

// ---- peer memory (CUDA IPC) ---------------------------------------------------------------------------------------------
extern "C" int glamr_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle64) {
  if (!dev_ptr || !handle64 || bytes == 0) return GLAMR_EINVAL;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  void* p = nullptr;
  GLAMR_CUDA_TRY(cudaMalloc(&p, bytes));
  cudaError_t e = cudaMemset(p, 0, bytes);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return (int)e; }
  memcpy(handle64, &h, 64);
  *dev_ptr = p;
  return GLAMR_OK;
}
extern "C" int glamr_peer_open(const unsigned char* handle64, void** dev_ptr) {
  if (!handle64 || !dev_ptr) return GLAMR_EINVAL;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  GLAMR_CUDA_TRY(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return GLAMR_OK;
}
extern "C" int glamr_peer_close(void* dev_ptr) {
  if (!dev_ptr) return GLAMR_EINVAL;
  GLAMR_CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr));
  return GLAMR_OK;
}
extern "C" int glamr_peer_free(void* dev_ptr) {
  if (!dev_ptr) return GLAMR_EINVAL;
  GLAMR_CUDA_TRY(cudaFree(dev_ptr));
  return GLAMR_OK;
}
extern "C" size_t glamr_opt_peer_bytes(const glamr_opt_t* st) {
  if (!st) return 0;
  const size_t slot = ((size_t)st->pb.n_params + GLAMR_NUM_TERMS + 63) & ~(size_t)63;
  return kPeerHeaderWords * sizeof(uint32_t) + 2 * (size_t)GLAMR_MAX_PEERS * slot * sizeof(unsigned long long);
}
extern "C" int glamr_opt_set_peers(glamr_opt_t* st, int rank, int world, void* const* bufs) {
  if (!st || world < 0 || world > GLAMR_MAX_PEERS || (world > 1 && (!bufs || rank < 0 || rank >= world))) return GLAMR_EINVAL;
  st->gen++;                                   // a captured iteration holds the old peer table
  memset(&st->peer, 0, sizeof(st->peer));
  if (world <= 1) return GLAMR_OK;
  st->peer.rank = rank;
  st->peer.world = world;
  st->peer.slot_elems = ((size_t)st->pb.n_params + GLAMR_NUM_TERMS + 63) & ~(size_t)63;
  for (int r = 0; r < world; ++r) {
    if (!bufs[r]) return GLAMR_EINVAL;
    st->peer.bufs[r] = (unsigned long long*)bufs[r];
  }
  return GLAMR_OK;
}

extern "C" int glamr_allreduce_inplace(glamr_opt_t* st, float* buf, size_t count, void* stream) {
  if (!st || !buf) return GLAMR_EINVAL;
  if (st->peer.world <= 1) return GLAMR_OK;     // single rank: the sum is the input
  if (count > st->peer.slot_elems) return GLAMR_ENOSPACE;
  if (count == 0) return GLAMR_OK;
  const int blocks = (int)((count + 255) / 256);
  peer_allreduce_kernel<<<blocks < 592 ? blocks : 592, 256, 0, (cudaStream_t)stream>>>(st->peer, buf, (int)count, st->tickets + 3);
  GLAMR_LAUNCH_CHECK();
  return GLAMR_OK;
}

extern "C" int glamr_opt_iterate(glamr_opt_t* st, float* theta, float* reduce_buf, double lr, float* loss_terms, int loss_hist_stride,
                                 int n_iters, int use_graph, void* stream) {
  if (!st || !theta || !reduce_buf || n_iters < 0) return GLAMR_EINVAL;
  cudaStream_t s = (cudaStream_t)stream;
  int rc, done = 0;
  const bool peers = st->peer.world > 1;      // W > 1: backward publishes, apply sums the peers' slots (no call in between)
  auto eager = [&](cudaStream_t q) -> int {
    if ((rc = backward_impl(st, theta, reduce_buf, q, peers))) return rc;
    return apply_impl(st, theta, reduce_buf, lr, loss_terms, loss_hist_stride, q, peers);
  };
  if (!use_graph || st->timing) {
    for (; done < n_iters; ++done)
      if ((rc = eager(s))) return rc;
    return GLAMR_OK;
  }
  const bool valid = st->iter_exec && st->cap_gen == st->gen && st->cap_theta == theta && st->cap_reduce == reduce_buf &&
                     st->cap_hist == loss_terms && st->cap_lr == lr && st->cap_stride == loss_hist_stride;
  if (!valid) {
    if (n_iters == 0) return GLAMR_OK;
    if ((rc = eager(s))) return rc;          // first iteration eagerly: module loading / function attributes happen outside capture
    done = 1;
    if (n_iters == 1) return GLAMR_OK;
    if (st->iter_exec) { cudaGraphExecDestroy(st->iter_exec); st->iter_exec = nullptr; }
    if (!st->cap_stream) GLAMR_CUDA_TRY(cudaStreamCreateWithFlags(&st->cap_stream, cudaStreamNonBlocking));
    cudaGraph_t g = nullptr;
    GLAMR_CUDA_TRY(cudaStreamBeginCapture(st->cap_stream, cudaStreamCaptureModeThreadLocal));
    rc = eager(st->cap_stream);
    const cudaError_t ce = cudaStreamEndCapture(st->cap_stream, &g);
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (ce != cudaSuccess) return (int)ce;
    const cudaError_t ie = cudaGraphInstantiate(&st->iter_exec, g, 0);
    cudaGraphDestroy(g);
    if (ie != cudaSuccess) { st->iter_exec = nullptr; return (int)ie; }
    st->cap_gen = st->gen; st->cap_theta = theta; st->cap_reduce = reduce_buf; st->cap_hist = loss_terms; st->cap_lr = lr;
    st->cap_stride = loss_hist_stride;
  }
  for (; done < n_iters; ++done) GLAMR_CUDA_TRY(cudaGraphLaunch(st->iter_exec, s));
  return GLAMR_OK;
}

extern "C" int glamr_opt_read(glamr_opt_t* st, int what, const float** ptr, size_t* count) {
  if (!st || !ptr || !count) return GLAMR_EINVAL;
  const size_t N = (size_t)st->pb.P * st->pb.T, T = st->pb.T, J = st->pb.J;
  switch (what) {
    case GLAMR_R_ORIENT_WORLD: *ptr = st->sc.orient_world; *count = 3 * N; break;
    case GLAMR_R_TRANS_WORLD: *ptr = st->sc.trans_world; *count = 3 * N; break;
    case GLAMR_R_ORIENT_BASE: *ptr = st->sc.orient_base; *count = 3 * N; break;
    case GLAMR_R_TRANS_BASE: *ptr = st->sc.trans_base; *count = 3 * N; break;
    case GLAMR_R_KP_PRED: *ptr = st->sc.kp_pred; *count = N * J * 2; break;
    case GLAMR_R_ORIENT_CAM_IN_WORLD: *ptr = st->sc.orient_ciw; *count = 3 * N; break;
    case GLAMR_R_TRANS_CAM_IN_WORLD: *ptr = st->sc.trans_ciw; *count = 3 * N; break;
    case GLAMR_R_CAM_POSE: *ptr = st->sc.cam; *count = 12 * T; break;
    case GLAMR_R_CAM_POSE_INV: *ptr = st->sc.cam_inv; *count = 12 * T; break;
    case GLAMR_R_JOINTS_WORLD: *ptr = st->sc.joints_world; *count = N * J * 3; break;
    case GLAMR_R_TRAJ_LOCAL: *ptr = st->sc.traj_local; *count = 11 * N; break;
    default: return GLAMR_EINVAL;
  }
  return GLAMR_OK;
}
