// The fused online step: ONE host call enqueues everything `Online_NTF.step` (reference src/ontf.py:117-154) does for a
// minibatch -- dictionary update with the OLD aggregates, FP64 Gram + TF32 split of the new dictionary (side stream);
// covariances, LARS-lasso codes, surrogate partial sums (main stream); blend into A, B (side stream) -- with the
// cross-stream ordering expressed through CUDA events owned by an opaque plan.  No device memory is allocated and
// nothing synchronises the host.  A multi-GPU caller all-reduces P[cur] on the side stream between
// onmf_step_launch() and onmf_step_finish(); a single-GPU caller uses onmf_step().
//
// Ordering (one-step lag of the reference: update_dict at step t reads A_{t-1}, B_{t-1}, src/ontf.py:151):
//   side : wait(code_{t-1}) -> BCD(W[cur] -> W[cur^1]) -> Gram, split -> record(W_t)
//   main : [split X] -> cov(W[cur]) -> [wait(AB_{t-1}) if hold_coder] -> LARS -> [split H] -> partial sums -> record(P_t, code_t)
//   side : wait(P_t) -> (all-reduce by the caller) -> blend -> record(AB_t)
//   main : wait(W_t)                                       -- the next coding needs the new dictionary only
//
// The minibatch comes either as a dense sample-major matrix Xt (n x d) or -- tensor-core path, k <= 256 -- as a DESCRIPTOR
// (onmf_minibatch: stored pool + row indices + storage format): then the fused kernels of gemm_fused.cu read the pool rows
// in place (gather, widening and TF32 split inside the loaders), nothing of the minibatch is ever copied or split in HBM,
// and on a single GPU the blend is the epilogue of the partial-sum reduction:
//   main : cov_fused(pool, idx) -> LARS -> wait(W_t) -> sur_fused(Ht, pool, idx) + reduce + blend -> record(code_t, AB_t)
// A third kind, the patch minibatch (onmf_patch_minibatch: image + corners + indices), takes the same fused schedule with
// the loaders reading the patches out of the image.
#include <new>

#include "common.cuh"

// one instantiated CUDA graph of the whole step for a fixed (minibatch pointer, codes pointer, n, cur, buffers)
struct StepGraph {
  const void* Xt;             // minibatch base pointer (Xt, the pool of a minibatch descriptor, or a patch minibatch's image)
  const void* idx;            // minibatch row indices (descriptor form) or nullptr
  const void* codes;
  long long n;
  int cur;
  unsigned long long sig;     // hash of the buffer descriptor the graph was captured with
  cudaGraphExec_t exec;       // nullptr: key seen once, not captured yet
  long long kernels;          // kernels inside the graph (launch accounting)
  unsigned long long last_use;
};
constexpr int STEP_GRAPHS = 8;
constexpr int W_RING = 4096;

struct onmf_step_plan {
  cudaEvent_t ev_P, ev_W, ev_code, ev_AB;
  cudaEvent_t ev_g0, ev_g1, ev_g2, ev_pre;   // fork / partial-sums / join inside a captured step; pre-launch join
  int tslots;                 // LARS timing ring (0 = off)
  long long tcount;
  cudaEvent_t* t0;
  cudaEvent_t* t1;
  long long launches;         // kernels launched through this plan
  StepGraph graphs[STEP_GRAPHS];
  unsigned long long use_clock;
  cudaStream_t cap;           // capture origin (the caller's main stream may be the legacy default stream, which cannot capture)
  double* w_ring;             // pinned host ring of blend weights (copied to buffers->w_dev before each graph launch)
  unsigned long long w_count;
  long long graph_steps;      // steps that ran as a graph replay
};

using namespace onmf;

extern "C" int onmf_step_plan_create(onmf_step_plan** out, int timing_slots) {
  if (!out || timing_slots < 0 || timing_slots > 4096) return fail(ONMF_E_ARG, "step_plan_create: bad argument");
  onmf_step_plan* p = new (std::nothrow) onmf_step_plan();
  if (!p) return fail(ONMF_E_ARG, "step_plan_create: out of host memory");
  p->tslots = timing_slots; p->tcount = 0; p->t0 = p->t1 = nullptr; p->launches = 0;
  memset(p->graphs, 0, sizeof(p->graphs));
  p->use_clock = 0; p->w_ring = nullptr; p->w_count = 0; p->graph_steps = 0;
  ONMF_CUDA(cudaHostAlloc((void**)&p->w_ring, W_RING * sizeof(double), cudaHostAllocDefault));
  ONMF_CUDA(cudaStreamCreateWithFlags(&p->cap, cudaStreamNonBlocking));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_g0, cudaEventDisableTiming));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_g1, cudaEventDisableTiming));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_g2, cudaEventDisableTiming));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_pre, cudaEventDisableTiming));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_P, cudaEventDisableTiming));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_W, cudaEventDisableTiming));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_code, cudaEventDisableTiming));
  ONMF_CUDA(cudaEventCreateWithFlags(&p->ev_AB, cudaEventDisableTiming));
  if (timing_slots > 0) {
    p->t0 = new (std::nothrow) cudaEvent_t[timing_slots];
    p->t1 = new (std::nothrow) cudaEvent_t[timing_slots];
    if (!p->t0 || !p->t1) return fail(ONMF_E_ARG, "step_plan_create: out of host memory");
    for (int i = 0; i < timing_slots; ++i) {
      ONMF_CUDA(cudaEventCreate(&p->t0[i]));
      ONMF_CUDA(cudaEventCreate(&p->t1[i]));
    }
  }
  *out = p;
  return ONMF_OK;
}

extern "C" int onmf_step_plan_destroy(onmf_step_plan* p) {
  if (!p) return ONMF_OK;
  cudaEventDestroy(p->ev_P); cudaEventDestroy(p->ev_W); cudaEventDestroy(p->ev_code); cudaEventDestroy(p->ev_AB);
  cudaEventDestroy(p->ev_g0); cudaEventDestroy(p->ev_g1); cudaEventDestroy(p->ev_g2); cudaEventDestroy(p->ev_pre);
  for (int i = 0; i < STEP_GRAPHS; ++i)
    if (p->graphs[i].exec) cudaGraphExecDestroy(p->graphs[i].exec);
  if (p->w_ring) cudaFreeHost(p->w_ring);
  if (p->cap) cudaStreamDestroy(p->cap);
  for (int i = 0; i < p->tslots; ++i) { cudaEventDestroy(p->t0[i]); cudaEventDestroy(p->t1[i]); }
  delete[] p->t0;
  delete[] p->t1;
  delete p;
  return ONMF_OK;
}

extern "C" int onmf_step_plan_mark_state(onmf_step_plan* p, void* main_stream) {
  if (!p) return fail(ONMF_E_ARG, "step_plan_mark_state: null plan");
  ONMF_CUDA(cudaEventRecord(p->ev_code, (cudaStream_t)main_stream));
  return ONMF_OK;
}

extern "C" long long onmf_step_plan_launches(const onmf_step_plan* p) { return p ? p->launches : 0; }
extern "C" long long onmf_step_plan_graph_steps(const onmf_step_plan* p) { return p ? p->graph_steps : 0; }

extern "C" int onmf_step_plan_reset_timing(onmf_step_plan* p) {
  if (!p) return fail(ONMF_E_ARG, "step_plan_reset_timing: null plan");
  p->tcount = 0;
  return ONMF_OK;
}

extern "C" int onmf_step_plan_lars_ms(onmf_step_plan* p, float* out, int max_out, int* n_out) {
  if (!p || !out || !n_out) return fail(ONMF_E_ARG, "step_plan_lars_ms: bad argument");
  long long have = p->tcount < p->tslots ? p->tcount : p->tslots;
  int n = (int)(have < max_out ? have : max_out);
  const long long first = p->tcount - have;
  for (int i = 0; i < n; ++i) {
    const int s = (int)((first + i) % p->tslots);
    ONMF_CUDA(cudaEventSynchronize(p->t1[s]));
    ONMF_CUDA(cudaEventElapsedTime(&out[i], p->t0[s], p->t1[s]));
  }
  *n_out = n;
  return ONMF_OK;
}

static int check_buffers(const onmf_step_buffers* b, bool need_code_bufs) {
  if (!b) return fail(ONMF_E_ARG, "step: null buffers");
  if (b->dtype != ONMF_F32 && b->dtype != ONMF_F64) return fail(ONMF_E_ARG, "step: bad dtype");
  if (b->d <= 0 || b->k <= 0) return fail(ONMF_E_ARG, "step: bad shape");
  if (!b->W[0] || !b->W[1] || !b->G[0] || !b->G[1] || !b->A || !b->B || !b->P[0] || !b->P[1] || !b->ws_gram)
    return fail(ONMF_E_ARG, "step: null state buffer");
  if (b->use_tc && (b->dtype != ONMF_F32 || !b->Whi[0] || !b->Whi[1] || !b->Wlo[0] || !b->Wlo[1]))
    return fail(ONMF_E_ARG, "step: tensor-core path needs fp32 and the split dictionary buffers");
  if (need_code_bufs && (!b->Ht || !b->ws_sur)) return fail(ONMF_E_ARG, "step: null minibatch buffer");
  if (b->track_C && (!b->C || !b->P2)) return fail(ONMF_E_ARG, "step: track_C needs C and P2");
  return ONMF_OK;
}

// what one step consumes: a dense minibatch, a pool descriptor or a patch minibatch (at most one of Xt / mb / pm; none on
// the pre-split path)
struct StepIn {
  const void* Xt;              // dense (n x d) in the engine dtype, or nullptr
  const onmf_minibatch* mb;    // descriptor (fused tensor-core path), or nullptr
  const onmf_patch_minibatch* pm;   // patches of a resident image (fused tensor-core path), or nullptr
  const void* codes;           // externally computed codes (n x k) or nullptr
  long long n;
};

// blend request of a step: none (the caller blends after its all-reduce), host weight, or device weight (graph replay)
struct Blend {
  int mode;                    // 0 none, 1 host w, 2 *w_dev
  double w;
};

static bool mb_fused(const onmf_step_buffers* b, const StepIn& in) {
  return (in.mb != nullptr || in.pm != nullptr) && b->use_tc && onmf_fused_tc_supported(b->k, b->d);
}

// the two fused products on whichever by-reference minibatch the step carries
static int fused_cov(const onmf_step_buffers* b, const StepIn& in, int cur, cudaStream_t st) {
  if (in.pm) return onmf_cov_fused_tc_patches(in.pm, b->Whi[cur], b->Wlo[cur], b->k, b->Ct, st);
  return onmf_cov_fused_tc(in.mb->kind, in.mb->base, in.mb->n_pool, in.mb->ld, in.mb->idx, in.n, b->d, in.mb->scale, b->Whi[cur],
                           b->Wlo[cur], b->k, b->Ct, st);
}
static int fused_sur(const onmf_step_buffers* b, const StepIn& in, const void* H, void* P, int blend, double w, const double* w_dev,
                     cudaStream_t st) {
  void* A = blend ? b->A : nullptr;
  void* B = blend ? b->B : nullptr;
  if (in.pm) return onmf_surrogate_fused_tc_patches(H, in.pm, b->k, P, blend, w, w_dev, A, B, b->ws_sur, b->ws_sur_bytes, st);
  return onmf_surrogate_fused_tc(H, in.mb->kind, in.mb->base, in.mb->n_pool, in.mb->ld, in.mb->idx, in.n, b->k, b->d, in.mb->scale, P,
                                 blend, w, w_dev, A, B, b->ws_sur, b->ws_sur_bytes, st);
}

// Enqueue one step.  captured = false: two streams ordered by the plan's events (cross-step overlap);
// captured = true: fork/join on p->cap + side for stream capture (no event recorded outside the capture is waited on).
// On return *blended says whether A, B already hold the blended aggregates (fused epilogue) or P[cur] awaits blending.
static int enqueue_step(onmf_step_plan* p, const onmf_step_buffers* b, const StepIn& in, int cur, const Blend& bl, bool captured,
                        bool* blended, long long* kernels) {
  cudaStream_t main = captured ? p->cap : (cudaStream_t)b->main_stream, side = (cudaStream_t)b->side_stream;
  const int dt = b->dtype, d = b->d, k = b->k, nx = cur ^ 1;
  const size_t esz = dt == ONMF_F64 ? 8 : 4;
  const long long n = in.n;
  const bool fused = mb_fused(b, in);
  const bool presplit = (in.Xt == nullptr && in.mb == nullptr && in.pm == nullptr);
  int rc;
  const long long l0 = g_launches;
  *blended = false;

  // ---- side: dictionary update with the OLD aggregates, then everything the coder derives from the dictionary ----
  if (captured) {
    ONMF_CUDA(cudaEventRecord(p->ev_g0, main));
    ONMF_CUDA(cudaStreamWaitEvent(side, p->ev_g0, 0));                    // fork
  } else {
    ONMF_CUDA(cudaStreamWaitEvent(side, p->ev_code, 0));
  }
  // (the large-dictionary fallback of the update borrows the Gram workspace: same stream, used one after the other)
  if ((rc = onmf_update_dict_ws(dt, b->W[cur], b->A, b->B, d, k, b->W[nx], b->ws_gram, b->ws_gram_bytes, side))) return rc;
  if ((rc = onmf_gram_f64(dt, b->W[nx], d, k, b->G[nx], nullptr, b->ws_gram, b->ws_gram_bytes, side))) return rc;
  if (b->use_tc) {
    if ((rc = onmf_split_tf32(b->W[nx], b->Whi[nx], b->Wlo[nx], (int64_t)d * k, side))) return rc;
  }
  ONMF_CUDA(cudaEventRecord(captured ? p->ev_g2 : p->ev_W, side));

  // ---- main: code this minibatch with W[cur], partial sums ----
  if (b->track_C && !captured) ONMF_CUDA(cudaStreamWaitEvent(main, p->ev_AB, 0));   // P2 is single-buffered (AB is recorded after C's blend)
  // the blend may ride on the partial-sum reduction when this call owns the whole step (single GPU) on the fused path
  const bool fuse_blend = fused && bl.mode != 0 && !b->track_C;
  if (n > 0) {
    const void* Hcodes = in.codes ? in.codes : b->Ht;
    if (b->use_tc && !fused && !presplit) {
      if ((rc = onmf_split_tf32(in.Xt, b->Xhi, b->Xlo, n * d, main))) return rc;
    }
    if (!in.codes) {
      if (!b->Ct || !b->ws_lars) return fail(ONMF_E_ARG, "step: null coder buffer");
      if (fused) rc = fused_cov(b, in, cur, main);
      else if (b->use_tc) rc = onmf_cov_tc(b->Xhi, b->Xlo, n, d, b->Whi[cur], b->Wlo[cur], k, b->Ct, main);
      else rc = onmf_cov(dt, in.Xt, n, d, b->W[cur], k, b->Ct, main);
      if (rc) return rc;
      // the dictionary update is one thread-block cluster: it is only placed while a group of SMs in one GPC is free,
      // i.e. before the persistent coder has spread over the GPU -- hold the coder until the blend it follows is done
      if (b->hold_coder && !captured) ONMF_CUDA(cudaStreamWaitEvent(main, p->ev_AB, 0));
      const int rsv = b->reserve_sms >= 0 ? b->reserve_sms : 0;
      const int saved = g_lars_reserved_sms;
      g_lars_reserved_sms = rsv;
      const bool timed = p->tslots > 0 && !captured;
      if (timed) ONMF_CUDA(cudaEventRecord(p->t0[p->tcount % p->tslots], main));
      if (dt == ONMF_F32)
        rc = onmf_lasso_lars_g64(dt, b->G[cur], b->Ct, n, k, d, b->alpha, b->max_iter, b->Ht, b->ws_lars, b->ws_lars_bytes,
                                 b->stats, -1, main);
      else
        rc = onmf_lasso_lars_ex(dt, b->G[cur], b->Ct, n, k, d, b->alpha, b->max_iter, b->Ht, b->ws_lars, b->ws_lars_bytes,
                                b->stats, -1, main);
      g_lars_reserved_sms = saved;
      if (rc) return rc;
      if (timed) {
        ONMF_CUDA(cudaEventRecord(p->t1[p->tcount % p->tslots], main));
        ++p->tcount;
      }
    }
    if (fused) {
      if (fuse_blend) {
        // the blend overwrites A, B: the dictionary update (side) must have finished reading them
        ONMF_CUDA(cudaStreamWaitEvent(main, captured ? p->ev_g2 : p->ev_W, 0));
        rc = fused_sur(b, in, Hcodes, nullptr, 1, bl.w, bl.mode == 2 ? b->w_dev : nullptr, main);
        *blended = true;
      } else {
        rc = fused_sur(b, in, Hcodes, b->P[cur], 0, 0.0, nullptr, main);
      }
      if (rc) return rc;
    } else if (b->use_tc) {
      if ((rc = onmf_split_tf32(Hcodes, b->Hhi, b->Hlo, n * k, main))) return rc;
      if ((rc = onmf_surrogate_partial_tc(b->Hhi, b->Hlo, b->Xhi, b->Xlo, n, k, d, b->P[cur], b->ws_sur, b->ws_sur_bytes, main)))
        return rc;
    } else {
      if ((rc = onmf_surrogate_partial(dt, Hcodes, in.Xt, n, k, d, b->P[cur], b->ws_sur, b->ws_sur_bytes, main))) return rc;
    }
    if (b->track_C) {
      if ((rc = onmf_xxt_partial(dt, in.Xt, n, d, b->P2, b->ws_sur, b->ws_sur_bytes, main))) return rc;
    }
  } else {
    ONMF_CUDA(cudaMemsetAsync(b->P[cur], 0, (size_t)k * (k + d) * esz, main));
    if (b->track_C) ONMF_CUDA(cudaMemsetAsync(b->P2, 0, (size_t)d * d * esz, main));
  }
  *kernels = g_launches - l0;
  return ONMF_OK;
}

static int check_step_in(const onmf_step_buffers* b, const StepIn& in, int cur, const char* who) {
  int rc = check_buffers(b, in.n > 0);
  if (rc) return rc;
  if (in.n < 0 || (cur != 0 && cur != 1)) return fail(ONMF_E_ARG, who);
  if ((in.Xt != nullptr) + (in.mb != nullptr) + (in.pm != nullptr) > 1)
    return fail(ONMF_E_ARG, "step: pass one of a dense minibatch, a descriptor or a patch minibatch");
  if (in.mb) {
    if (in.mb->n != in.n) return fail(ONMF_E_ARG, "step: descriptor row count differs from n");
    if (!mb_fused(b, in)) return fail(ONMF_E_UNSUPPORTED, "step: a minibatch descriptor needs the fused tensor-core path (fp32, onmf_fused_tc_supported)");
    if (b->track_C) return fail(ONMF_E_UNSUPPORTED, "step: track_C needs a dense minibatch");
  }
  if (in.pm) {
    if (in.pm->n != in.n) return fail(ONMF_E_ARG, "step: patch minibatch size differs from n");
    if ((long long)in.pm->p * in.pm->p * in.pm->C != b->d) return fail(ONMF_E_ARG, "step: patch minibatch p*p*C differs from d");
    if (!mb_fused(b, in)) return fail(ONMF_E_UNSUPPORTED, "step: a patch minibatch needs the fused tensor-core path (fp32, onmf_fused_tc_supported); gather it with onmf_gather_patches_mb otherwise");
    if (b->track_C) return fail(ONMF_E_UNSUPPORTED, "step: track_C needs a dense minibatch");
  }
  const bool presplit = (in.Xt == nullptr && in.mb == nullptr && in.pm == nullptr);
  if (in.n > 0 && presplit && !b->use_tc) return fail(ONMF_E_ARG, "step: Xt = NULL needs the tensor-core path");
  if (in.n > 0 && presplit && b->track_C) return fail(ONMF_E_ARG, "step: track_C needs the unsplit minibatch");
  return ONMF_OK;
}

// ---- stream schedule -------------------------------------------------------------------------------------------------
static int launch_streams(onmf_step_plan* p, const onmf_step_buffers* b, const StepIn& in, int cur, const Blend& bl, bool* blended) {
  cudaStream_t main = (cudaStream_t)b->main_stream, side = (cudaStream_t)b->side_stream;
  long long kn = 0;
  int rc = enqueue_step(p, b, in, cur, bl, false, blended, &kn);
  if (rc) return rc;
  p->launches += kn;
  ONMF_CUDA(cudaEventRecord(p->ev_P, main));
  ONMF_CUDA(cudaEventRecord(p->ev_code, main));
  // ---- side: the blend (and the caller's all-reduce before it) needs this step's partial sums ----
  ONMF_CUDA(cudaStreamWaitEvent(side, p->ev_P, 0));
  return ONMF_OK;
}

static int finish_streams(onmf_step_plan* p, const onmf_step_buffers* b, double w, int cur, bool blended) {
  cudaStream_t main = (cudaStream_t)b->main_stream, side = (cudaStream_t)b->side_stream;
  int rc;
  const long long l0 = g_launches;
  if (!blended) {
    if ((rc = onmf_surrogate_blend(b->dtype, b->P[cur], b->k, b->d, w, b->A, b->B, side))) return rc;
  }
  if (b->track_C) {
    if ((rc = onmf_axpby(b->dtype, (int64_t)b->d * b->d, w, b->P2, 1.0 - w, b->C, side))) return rc;
  }
  p->launches += g_launches - l0;
  ONMF_CUDA(cudaEventRecord(p->ev_AB, side));        // (blended on main: side has waited for ev_P, recorded after that blend)
  ONMF_CUDA(cudaStreamWaitEvent(main, p->ev_W, 0));  // the next coding needs the new dictionary only
  return ONMF_OK;
}

extern "C" int onmf_step_launch(onmf_step_plan* p, const onmf_step_buffers* b, const void* Xt, const void* codes,
                                int64_t n, int cur) {
  if (!p) return fail(ONMF_E_ARG, "step_launch: null plan");
  StepIn in{Xt, nullptr, nullptr, codes, n};
  int rc = check_step_in(b, in, cur, "step_launch: bad argument");
  if (rc) return rc;
  bool blended;
  return launch_streams(p, b, in, cur, Blend{0, 0.0}, &blended);
}

extern "C" int onmf_step_launch_mb(onmf_step_plan* p, const onmf_step_buffers* b, const onmf_minibatch* mb, const void* codes, int cur) {
  if (!p || !mb) return fail(ONMF_E_ARG, "step_launch_mb: null plan / descriptor");
  StepIn in{nullptr, mb, nullptr, codes, mb->n};
  int rc = check_step_in(b, in, cur, "step_launch_mb: bad argument");
  if (rc) return rc;
  bool blended;
  return launch_streams(p, b, in, cur, Blend{0, 0.0}, &blended);
}

extern "C" int onmf_step_finish(onmf_step_plan* p, const onmf_step_buffers* b, double w, int cur) {
  if (!p) return fail(ONMF_E_ARG, "step_finish: null plan");
  int rc = check_buffers(b, false);
  if (rc) return rc;
  return finish_streams(p, b, w, cur, false);
}

static int step_streams(onmf_step_plan* p, const onmf_step_buffers* b, const StepIn& in, double w, int cur) {
  bool blended = false;
  int rc = launch_streams(p, b, in, cur, Blend{1, w}, &blended);
  if (rc) return rc;
  return finish_streams(p, b, w, cur, blended);
}

extern "C" int onmf_step(onmf_step_plan* p, const onmf_step_buffers* b, const void* Xt, const void* codes, int64_t n,
                         double w, int cur) {
  if (!p) return fail(ONMF_E_ARG, "step: null plan");
  StepIn in{Xt, nullptr, nullptr, codes, n};
  int rc = check_step_in(b, in, cur, "step: bad argument");
  if (rc) return rc;
  return step_streams(p, b, in, w, cur);
}

extern "C" int onmf_step_mb(onmf_step_plan* p, const onmf_step_buffers* b, const onmf_minibatch* mb, const void* codes, double w,
                            int cur) {
  if (!p || !mb) return fail(ONMF_E_ARG, "step_mb: null plan / descriptor");
  StepIn in{nullptr, mb, nullptr, codes, mb->n};
  int rc = check_step_in(b, in, cur, "step_mb: bad argument");
  if (rc) return rc;
  return step_streams(p, b, in, w, cur);
}

// ------------------------------------------------------------------------------------------------------------------
// The same step as ONE CUDA graph (single GPU).  A step is a fork-join: [dictionary update, Gram, split] on the side
// branch next to [covariances, coder, partial sums] on the main branch, then the blend that needs both -- and the next
// step's coding needs nothing but the new dictionary, so consecutive steps are consecutive graph launches on the main
// stream.  For the small configurations (BASELINE configs[0..3]: a step is ~15 dependent launches of a few microseconds
// each) this removes the per-launch CPU cost and the inter-kernel gaps.  The blend weight w = t^-beta changes every
// step: it is read from device memory (buffers->w_dev), refreshed by a stream-ordered 8-byte copy before each launch.
// Graphs are cached per (minibatch pointers, codes pointer, n, cur, buffer descriptor); a key is captured the second
// time it is seen, so one-off calls never pay for capture + instantiation.
// ------------------------------------------------------------------------------------------------------------------
static unsigned long long buffers_sig(const onmf_step_buffers* b, const onmf_minibatch* mb, const onmf_patch_minibatch* pm) {
  unsigned long long h = 1469598103934665603ULL;
  const unsigned char* q = reinterpret_cast<const unsigned char*>(b);
  for (size_t i = 0; i < sizeof(*b); ++i) { h ^= q[i]; h *= 1099511628211ULL; }
  if (pm) {
    // everything a replay bakes in besides the image / index pointers of the key: corners, geometry, storage, scale
    double sc = pm->scale;
    unsigned long long scb;
    memcpy(&scb, &sc, 8);
    const unsigned long long v[9] = {0x70617463686573ull, (unsigned long long)(uintptr_t)pm->coords, (unsigned long long)pm->n_coords,
                                     (unsigned long long)pm->kind, (unsigned long long)pm->H, (unsigned long long)pm->W,
                                     (unsigned long long)pm->C, (unsigned long long)pm->p, scb};
    for (int i = 0; i < 9; ++i) { h ^= v[i]; h *= 1099511628211ULL; }
  }
  if (mb) {
    const unsigned long long v[4] = {(unsigned long long)mb->kind, (unsigned long long)mb->n_pool, (unsigned long long)mb->ld, 0ull};
    double sc = mb->scale;
    unsigned long long scb;
    memcpy(&scb, &sc, 8);
    for (int i = 0; i < 3; ++i) { h ^= v[i]; h *= 1099511628211ULL; }
    h ^= scb; h *= 1099511628211ULL;
  }
  return h;
}

static int step_graph_impl(onmf_step_plan* p, const onmf_step_buffers* b, const StepIn& in, double w, int cur) {
  // not expressible as this graph: the d x d aggregate (host-side w in its blend), coder timing events, multi-GPU hold
  if (!b->w_dev || b->track_C || p->tslots > 0 || b->hold_coder) return step_streams(p, b, in, w, cur);
  cudaStream_t main = (cudaStream_t)b->main_stream, side = (cudaStream_t)b->side_stream;
  const void* base = in.pm ? in.pm->img : in.mb ? in.mb->base : in.Xt;
  const void* idx = in.pm ? (const void*)in.pm->idx : in.mb ? (const void*)in.mb->idx : nullptr;
  const unsigned long long sig = buffers_sig(b, in.mb, in.pm);
  StepGraph* e = nullptr;
  for (int i = 0; i < STEP_GRAPHS; ++i) {
    StepGraph& g = p->graphs[i];
    if (g.last_use && g.Xt == base && g.idx == idx && g.codes == in.codes && g.n == in.n && g.cur == cur && g.sig == sig) { e = &g; break; }
  }
  if (!e) {                                       // first sight: remember the key, run the stream schedule
    StepGraph* v = &p->graphs[0];
    for (int i = 1; i < STEP_GRAPHS; ++i)
      if (p->graphs[i].last_use < v->last_use) v = &p->graphs[i];
    if (v->exec) cudaGraphExecDestroy(v->exec);
    v->Xt = base; v->idx = idx; v->codes = in.codes; v->n = in.n; v->cur = cur; v->sig = sig; v->exec = nullptr; v->kernels = 0;
    v->last_use = ++p->use_clock;
    return step_streams(p, b, in, w, cur);
  }
  e->last_use = ++p->use_clock;
  if (!e->exec) {                                 // second sight: capture
    // everything the two streams still have in flight from stream-scheduled steps is ordered before the replay by the
    // pre-launch join below; nothing is captured that waits on an event recorded outside the capture
    ONMF_CUDA(cudaStreamBeginCapture(p->cap, cudaStreamCaptureModeThreadLocal));
    long long kn = 0;
    bool blended = false;
    const long long l0 = g_launches;              // launches recorded into the graph are counted when it is replayed
    int rc = enqueue_step(p, b, in, cur, Blend{2, 0.0}, true, &blended, &kn);
    if (!rc) {
      // join: the side branch (dictionary update ...) and, unless the blend rode on the reduction, the blend after both
      cudaError_t ce = cudaSuccess;
      if (!blended) {
        ce = cudaEventRecord(p->ev_g1, p->cap);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(side, p->ev_g1, 0);
        if (ce == cudaSuccess) {
          rc = onmf_surrogate_blend_dev(b->dtype, b->P[cur], b->k, b->d, b->w_dev, b->A, b->B, side);
        }
        if (ce == cudaSuccess && !rc) ce = cudaEventRecord(p->ev_g2, side);
      }
      if (ce == cudaSuccess && !rc) ce = cudaStreamWaitEvent(p->cap, p->ev_g2, 0);
      if (ce != cudaSuccess && !rc) rc = cuda_fail(ce, "step_graph: capture join");
    }
    kn = g_launches - l0;
    g_launches = l0;
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(p->cap, &graph);
    if (rc || ce != cudaSuccess || !graph) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      if (rc) return rc;
      return cuda_fail(ce, "cudaStreamEndCapture");
    }
    ce = cudaGraphInstantiate(&e->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) { e->exec = nullptr; return cuda_fail(ce, "cudaGraphInstantiate"); }
    e->kernels = kn;
  }
  ONMF_CUDA(cudaEventRecord(p->ev_pre, side));
  ONMF_CUDA(cudaStreamWaitEvent(main, p->ev_pre, 0));
  double* slot = &p->w_ring[p->w_count++ % W_RING];
  *slot = w;
  ONMF_CUDA(cudaMemcpyAsync(b->w_dev, slot, sizeof(double), cudaMemcpyHostToDevice, main));
  ONMF_CUDA(cudaGraphLaunch(e->exec, main));
  // leave the stream-schedule events in a consistent state (a later stream-scheduled step, set_state or flush waits on them)
  ONMF_CUDA(cudaEventRecord(p->ev_P, main));
  ONMF_CUDA(cudaEventRecord(p->ev_code, main));
  ONMF_CUDA(cudaEventRecord(p->ev_W, main));
  ONMF_CUDA(cudaEventRecord(p->ev_AB, main));
  p->launches += e->kernels;
  g_launches += e->kernels;
  ++p->graph_steps;
  return ONMF_OK;
}

extern "C" int onmf_step_graph(onmf_step_plan* p, const onmf_step_buffers* b, const void* Xt, const void* codes, int64_t n,
                               double w, int cur) {
  if (!p) return fail(ONMF_E_ARG, "step_graph: null plan");
  StepIn in{Xt, nullptr, nullptr, codes, n};
  int rc = check_step_in(b, in, cur, "step_graph: bad argument");
  if (rc) return rc;
  return step_graph_impl(p, b, in, w, cur);
}

extern "C" int onmf_step_graph_mb(onmf_step_plan* p, const onmf_step_buffers* b, const onmf_minibatch* mb, const void* codes,
                                  double w, int cur) {
  if (!p || !mb) return fail(ONMF_E_ARG, "step_graph_mb: null plan / descriptor");
  StepIn in{nullptr, mb, nullptr, codes, mb->n};
  int rc = check_step_in(b, in, cur, "step_graph_mb: bad argument");
  if (rc) return rc;
  return step_graph_impl(p, b, in, w, cur);
}

// ---- patch minibatches --------------------------------------------------------------------------------------------
extern "C" int onmf_step_launch_patches(onmf_step_plan* p, const onmf_step_buffers* b, const onmf_patch_minibatch* pm, const void* codes,
                                        int cur) {
  if (!p || !pm) return fail(ONMF_E_ARG, "step_launch_patches: null plan / patch minibatch");
  StepIn in{nullptr, nullptr, pm, codes, pm->n};
  int rc = check_step_in(b, in, cur, "step_launch_patches: bad argument");
  if (rc) return rc;
  bool blended;
  return launch_streams(p, b, in, cur, Blend{0, 0.0}, &blended);
}

extern "C" int onmf_step_patches(onmf_step_plan* p, const onmf_step_buffers* b, const onmf_patch_minibatch* pm, const void* codes, double w,
                                 int cur) {
  if (!p || !pm) return fail(ONMF_E_ARG, "step_patches: null plan / patch minibatch");
  StepIn in{nullptr, nullptr, pm, codes, pm->n};
  int rc = check_step_in(b, in, cur, "step_patches: bad argument");
  if (rc) return rc;
  return step_streams(p, b, in, w, cur);
}

extern "C" int onmf_step_graph_patches(onmf_step_plan* p, const onmf_step_buffers* b, const onmf_patch_minibatch* pm, const void* codes,
                                       double w, int cur) {
  if (!p || !pm) return fail(ONMF_E_ARG, "step_graph_patches: null plan / patch minibatch");
  StepIn in{nullptr, nullptr, pm, codes, pm->n};
  int rc = check_step_in(b, in, cur, "step_graph_patches: bad argument");
  if (rc) return rc;
  return step_graph_impl(p, b, in, w, cur);
}
