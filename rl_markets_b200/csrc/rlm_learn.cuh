// rlm_learn.cuh -- the round-2 learner kernel: ONE warp per ready env, no block barrier anywhere.
//
// Replaces, for Q-learning / SARSA / Double-Q training (independent policies and the two shared-policy stages),
// the three-warp kernel rlm_agent3_kernel.  Same arithmetic, bit for bit (Agent::HandleTransition,
// src/rl/agent.cpp:86-142,268-353; Traces, src/rl/traces.cpp:30-50; tiles, src/rl/tiles.cpp:31-75,130-169);
// what changed is the shape of the step:
//   * lane j owns tiling j of ALL three feature groups: 16 coordinate look-ups + 27 tile indices per lane
//     (the action term of the hash is a constant per (group, action): DevParams::rg);
//   * all 27 (54) theta gathers of a lane are in flight together -- one DRAM round trip per evaluation;
//   * raw weights go to a [action][96] table in shared memory; lanes 0..A-1 (and 16..16+A-1 for table B) run
//     the reference's exact-order sum  Q += w0*th (32), w1*th (32), w2*th (64: the third loop restarts at T,
//     SURVEY Appendix A8)  as 128 multiplies feeding one dependent chain of 128 adds;
//   * argmax with rand() tie-breaks runs warp-wide (prefix maximum by shuffles); the serial scan is only taken
//     when two values tie with the running maximum, which is when the reference draws rand();
//   * the trace pass is the fused decay / clear / set / theta-update sweep of round 1 (one probe of the
//     tile -> last-writer table per entry, RED.ADD.F64 at L2); the second evaluation does not read anything back: it
//     adds this step's updates (kept in a shared-memory table, drained in batches of 512) to the weights the first
//     evaluation gathered; tile indices are never stored (re-derived from the three hash sums a lane keeps in registers);
//   * no occupancy bitmap: tables are dense after the first thousands of steps, which is the regime that counts.
// ~4000 warp-instructions per step instead of ~7700, no __syncthreads, no spills at 128 registers, 17.8 KB of shared
// memory per step: 12 steps in flight per SM.
#pragma once

#ifndef LN_WARPS
#define LN_WARPS 3  // steps (warps) per CTA; resident CTAs per SM follow from the shared memory of a step
#endif
#define LN_MIN_CTAS (15 / LN_WARPS)  // register budget: 15 warps per SM (128 registers)
#ifdef RLM_TIMING
#define LPH(i) do { if (lane == 0 && tp_idx < 4096) g_phase_clk[tp_idx * 16 + (i)] = clock64(); } while (0)
#else
#define LPH(i) do { } while (0)
#endif
#define LN_VROW 98  // doubles per action row (96 used): rows 4 banks apart, 16-byte aligned
#define LN_AG_BYTES 704

__host__ __device__ inline size_t ln_v_bytes(int is_double) { return (size_t)(is_double ? 2 : 1) * RLM_MAX_ACTIONS * LN_VROW * 8; }
// feature -> eligibility of every weight this step's update moved (open addressing): the second evaluation of the step
// adds the update to the weights it already holds instead of reading them back from L2 behind the reductions
#ifndef UT_LOG2
#define UT_LOG2 10  // 1024 slots, 512 entries per batch.  Measured: 256 or 512 slots cost more (longer probe chains in
#endif               // every step's patch pass, extra batches on the launch's slowest warp) than the occupancy they buy
static_assert(UT_LOG2 >= 7, "ut_clear writes UT_SLOTS / 128 int4 per lane: a smaller table would never be cleared");
#define UT_SLOTS (1 << UT_LOG2)
#define UT_MAX_ENTRIES (UT_SLOTS / 2)
// learner scratch of one step: [V][tile table 2048][update table 8 * UT_SLOTS][q_pre 2*9 doubles][dec 6 doubles]
__host__ __device__ inline size_t ln_scratch_bytes(int is_double) {
  return (ln_v_bytes(is_double) + TT_SLOTS * 4 + 2 * UT_SLOTS * 4 + 8 * 2 * RLM_MAX_ACTIONS + 48 + 15) & ~(size_t)15;
}
// per-warp shared memory of rlm_learn_kernel: [AgentD 704][scratch]
__host__ __device__ inline size_t ln_warp_bytes(int is_double) { return (size_t)LN_AG_BYTES + ln_scratch_bytes(is_double); }
static_assert(sizeof(AgentD) <= LN_AG_BYTES, "agent block outgrew its shared-memory slot");

// ---- gathers K0 .. K0+N-1 (k = g*9 + a) of one table in flight together; raw weights -> V[a][g*32 + lane]
template <int K0, int N>
__device__ __forceinline__ void ln_gather_issue(const double* __restrict__ th, const LnSums& h, double* v) {
  const int A = P.n_actions;
  if (P.m_pow2) {
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = (((K0 + k) % RLM_MAX_ACTIONS) < A) ? __ldcg(th + ln_tile<true>(h, K0 + k)) : 0.0;
  } else {
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = (((K0 + k) % RLM_MAX_ACTIONS) < A) ? __ldcg(th + ln_tile<false>(h, K0 + k)) : 0.0;
  }
}
template <int K0, int N>
__device__ __forceinline__ void ln_gather_store(const double* v, int lane, double* V) {
  const int A = P.n_actions;
#pragma unroll
  for (int k = 0; k < N; ++k)
    if (((K0 + k) % RLM_MAX_ACTIONS) < A) V[((K0 + k) % RLM_MAX_ACTIONS) * LN_VROW + ((K0 + k) / RLM_MAX_ACTIONS) * 32 + lane] = v[k];
}
template <bool DBL, int GB>
__device__ __forceinline__ void ln_gather(const double* __restrict__ th_a, const double* __restrict__ th_b, const LnSums& h, int lane, double* V) {
  static_assert(GB == 27 || GB == 9, "gather batch: everything, or one feature group at a time");
  double v[GB];
  if (GB == 27) {
    ln_gather_issue<0, GB>(th_a, h, v); ln_gather_store<0, GB>(v, lane, V);
    if (DBL) { ln_gather_issue<0, GB>(th_b, h, v); ln_gather_store<0, GB>(v, lane, V + RLM_MAX_ACTIONS * LN_VROW); }
  } else {
    ln_gather_issue<0, 9>(th_a, h, v); ln_gather_store<0, 9>(v, lane, V);
    ln_gather_issue<9, 9>(th_a, h, v); ln_gather_store<9, 9>(v, lane, V);
    ln_gather_issue<18, 9>(th_a, h, v); ln_gather_store<18, 9>(v, lane, V);
    if (DBL) {
      double* Vb = V + RLM_MAX_ACTIONS * LN_VROW;
      ln_gather_issue<0, 9>(th_b, h, v); ln_gather_store<0, 9>(v, lane, Vb);
      ln_gather_issue<9, 9>(th_b, h, v); ln_gather_store<9, 9>(v, lane, Vb);
      ln_gather_issue<18, 9>(th_b, h, v); ln_gather_store<18, 9>(v, lane, Vb);
    }
  }
}

// second evaluation of a step (same state, theta after this env's own update): theta_new[f] = theta_old[f] + update[f],
// the one IEEE addition the L2 reduction performs, on the weight the first evaluation gathered -- no read-back
__device__ __forceinline__ unsigned ut_hash(int f) { return ((unsigned)f * 2654435761u) >> (32 - UT_LOG2); }
__device__ __forceinline__ void ut_clear(int* ut, int lane) {
  int4* k4 = (int4*)ut;
#pragma unroll
  for (int i = 0; i < UT_SLOTS / 4 / 32; ++i) k4[lane + 32 * i] = make_int4(HS_EMPTY, HS_EMPTY, HS_EMPTY, HS_EMPTY);
}
__device__ __forceinline__ void ut_insert(int* ut, int f, float ev) {  // every f is inserted once per step
  unsigned slot = ut_hash(f);
  while (atomicCAS(&ut[slot], HS_EMPTY, f) != HS_EMPTY) slot = (slot + 1) & (UT_SLOTS - 1);
  ((float*)(ut + UT_SLOTS))[slot] = ev;
}
// the step's tile indices are re-derived from the hash sums (two instructions each for a power-of-two M): no index table
__device__ __forceinline__ void ln_patch_local(const int* ut, double scaled_update, unsigned long long s0, unsigned long long s1, unsigned long long s2,
                                               bool null_state, int lane, double* V) {
  const int A = P.n_actions;
  const float* uv = (const float*)(ut + UT_SLOTS);
  const bool pow2 = P.m_pow2 != 0;
  const unsigned mask = (unsigned)(P.memory_size - 1);
  // rolled over the actions (this runs once per step: code size is time), the three feature groups of one action side by
  // side: three independent index -> hash -> key chains per iteration instead of one
#pragma unroll 1
  for (int a = 0; a < A; ++a) {
    int f[3], key[3];
    unsigned slot[3];
#pragma unroll
    for (int g = 0; g < 3; ++g) {
      const unsigned r = P.rg[g][a];
      const unsigned long long sg = g == 0 ? s0 : (g == 1 ? s1 : s2);
      f[g] = null_state ? 0 : (pow2 ? (int)(((unsigned)sg + r) & mask) : mod_m(sg + r));
    }
#pragma unroll
    for (int g = 0; g < 3; ++g) { slot[g] = ut_hash(f[g]); key[g] = ut[slot[g]]; }
#pragma unroll
    for (int g = 0; g < 3; ++g) {
      while (key[g] != HS_EMPTY && key[g] != f[g]) { slot[g] = (slot[g] + 1) & (UT_SLOTS - 1); key[g] = ut[slot[g]]; }
      if (key[g] == f[g]) {
        const int at = a * LN_VROW + g * 32 + lane;
        V[at] = V[at] + scaled_update * (double)uv[slot[g]];
      }
    }
  }
}

// (the rare mid-list drain of a full table calls this copy; the step's final batch is patched inline)
__device__ __noinline__ void ln_patch_local_ool(const int* ut, double scaled_update, unsigned long long s0, unsigned long long s1, unsigned long long s2,
                                                bool null_state, int lane, double* V) {
  ASSUME_SHARED(ut); ASSUME_SHARED(V);
  ln_patch_local(ut, scaled_update, s0, s1, s2, null_state, lane, V);
}

// ---- exact-order sum of agent.cpp:117-135 over one action row of raw weights: 16 blocks of 8; block b+1 is loaded
// and multiplied while block b is added (the adds are the only dependent chain)
__device__ __forceinline__ double ln_chain(const double* row) {
  const double w0 = P.gw[0], w1 = P.gw[1], w2 = P.gw[2];
  double acc = 0.0, cur[8], nxt[8];
  {
    const double2* r2 = (const double2*)row;
#pragma unroll
    for (int j = 0; j < 4; ++j) { const double2 t = r2[j]; cur[2 * j] = w0 * t.x; cur[2 * j + 1] = w0 * t.y; }
  }
#pragma unroll 1
  for (int b = 1; b <= 16; ++b) {
    const int nb = (b < 16) ? b : 0;  // (the last iteration reloads block 0; unused)
    const double w = (nb < 4) ? w0 : ((nb < 8) ? w1 : w2);
    const int col = (nb < 8) ? 8 * nb : 8 * (nb - 4);  // blocks 8..15 walk columns 32..95 again with w2
    const double2* r2 = (const double2*)(row + col);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const double2 t = r2[j]; nxt[2 * j] = w * t.x; nxt[2 * j + 1] = w * t.y; }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc += cur[j];
#pragma unroll
    for (int j = 0; j < 8; ++j) cur[j] = nxt[j];
  }
  return acc;
}
// lanes 0..A-1: table A, lanes 16..16+A-1: table B (double agents).  Returns this lane's Q (0 elsewhere).
__device__ __noinline__ double ln_sums(const double* V, bool has_b, int lane) {
  ASSUME_SHARED(V);
  const int a = lane & 15, t = lane >> 4;
  double q = 0.0;
  if (a < P.n_actions && (t == 0 || has_b)) q = ln_chain(V + ((size_t)t * RLM_MAX_ACTIONS + a) * LN_VROW);
  return q;
}

// ---- argmax with rand() tie-breaks (agent.cpp:144-169), warp-wide.  v = this lane's value (lanes < A).  The scan's
// running maximum before element a is max(v[0..a-1]) whatever the tie-breaks did, so "rand() is drawn at a" <=>
// v[a] == that prefix maximum; with no such a (and no NaN) the result is the last strict improvement.  Otherwise
// lane 0 runs the reference's scan on `qs` (the same values in shared memory).
__device__ __forceinline__ int ln_argmax(AgentD& ag, double v, const double* qs, int lane) {
  const int A = P.n_actions;
  const bool in = lane < A;
  double m = in ? v : -1.7976931348623157e308;
#pragma unroll
  for (int d = 1; d < 16; d <<= 1) {
    const double t = __shfl_up_sync(FULL, m, d);
    if (lane >= d) m = fmax(m, t);
  }
  const double excl = __shfl_up_sync(FULL, m, 1);  // prefix maximum of v[0..lane-1]
  const bool odd = in && (v != v || (lane > 0 && v == excl));
  const unsigned strict = __ballot_sync(FULL, in && (lane == 0 || v > excl));
  int index;
  if (__any_sync(FULL, odd)) {
    index = 0;
    if (lane == 0) index = argmax_ties(ag, qs);
    index = __shfl_sync(FULL, index, 0);
  } else {
    index = 31 - __clz(strict);
  }
  return index;
}

// ---- tile -> last-writer table of the one-warp learners, ONE word per slot: (feature << 4) | action, empty = -1
// (features < 2^27, at most 16 actions).  Same open addressing as tt_insert / tt_last_writer (rlm_agent.cuh) at half the
// shared memory: 2 KB instead of 4, which is what lets a fourth CTA of three steps (a sixth staged table) share an SM.
static_assert(RLM_MAX_ACTIONS <= 16, "packed tile table: four bits of action");
__device__ __forceinline__ void ptt_insert(int* tt, int f, int a) {
  const int packed = (f << 4) | a;
  unsigned slot = tt_hash(f);
  while (true) {
    const int old = atomicCAS(&tt[slot], HS_EMPTY, packed);
    if (old == HS_EMPTY) return;
    if ((old >> 4) == f) { atomicMax(&tt[slot], packed); return; }  // same feature: the later (larger) action stays
    slot = (slot + 1) & (TT_SLOTS - 1);
  }
}
__device__ __forceinline__ int ptt_last_writer(const int* tt, int f) {
  unsigned slot = tt_hash(f);
  while (true) {
    const int k = tt[slot];
    if (k == HS_EMPTY) return -1;
    if ((k >> 4) == f) return k & 15;
    slot = (slot + 1) & (TT_SLOTS - 1);
  }
}

// ---- Traces::decay + Traces::update + Agent::updateQ in one sweep (see trace_pass in rlm_agent.cuh for the
// derivation); tt = tile -> last-writer table of the from-state, ut = update table (see ln_patch_local)
__device__ __forceinline__ void ln_tt_build(int* tt, const AgentD& ag, int lane) {
  int4* t4 = (int4*)tt;
#pragma unroll
  for (int i = 0; i < TT_SLOTS / 4 / 32; ++i) t4[lane + 32 * i] = make_int4(HS_EMPTY, HS_EMPTY, HS_EMPTY, HS_EMPTY);
  __syncwarp();
  if (!ag.null_from) {
    const int b0 = ag.from_base0[lane];
    const int M = (int)P.memory_size;
#pragma unroll 1
    for (int a = 0; a < P.n_actions; ++a) {
      int f = b0 + P.ra_m[a];
      if (f >= M) f -= M;
      ptt_insert(tt, f, a);
    }
  }
  __syncwarp();
}

// track: `ut` (cleared by the caller) takes the surviving entries, UT_MAX_ENTRIES at a time: when the table is full its
// updates are added to the weights of the to-state right away (ln_patch_local on Vp; every feature is in the list once,
// so every weight still gets at most one addition) and the table starts over.  The caller patches the last batch.
__device__ __forceinline__ int ln_trace_pass(AgentD& e, const int* tt, int* ut, bool track, int* tf, float* te, double* theta, int action,
                                          float rate, double scaled_update, int lane, const LnSums& h, double* Vp) {
  const bool null_from = e.null_from != 0;
  const int b0 = e.from_base0[lane];
  const float tol = 0.01f;
  int w = 0;
  int ins = 0;  // entries in `ut` (warp-uniform)
#define LN_UT_FLUSH() do { __syncwarp(); ln_patch_local_ool(ut, scaled_update, h.s[0], h.s[1], h.s[2], h.null_state, lane, Vp); __syncwarp(); ut_clear(ut, lane); __syncwarp(); ins = 0; } while (0)
  if (rate != 0.0f) {
    const int n = e.n_traces;
#pragma unroll 1
    for (int base = 0; base < n; base += 32 * TR_AHEAD) {
      int fq[TR_AHEAD];
      float eq[TR_AHEAD];
#pragma unroll
      for (int k = 0; k < TR_AHEAD; ++k) {
        const int i = base + 32 * k + lane;
        fq[k] = (i < n) ? __ldcg(tf + i) : 0;
        eq[k] = (i < n) ? __ldcg(te + i) : 0.0f;
      }
#pragma unroll
      for (int k = 0; k < TR_AHEAD; ++k) {
        if (base + 32 * k < n) {  // warp-uniform
          const int i = base + 32 * k + lane;
          const int f = fq[k];
          const float ev = eq[k] * rate;
          bool keep = (i < n) && !(ev < tol);
          if (keep) keep = (null_from ? (f == 0 ? P.n_actions - 1 : -1) : ptt_last_writer(tt, f)) < 0;
          const unsigned mask = __ballot_sync(FULL, keep);
          const int pos = w + __popc(mask & ((1u << lane) - 1u));
          if (track && ins + __popc(mask) > UT_MAX_ENTRIES) LN_UT_FLUSH();
          if (keep) {
            __stcg(tf + pos, f);
            __stcg(te + pos, ev);
            red_add_f64(theta + f, scaled_update * (double)ev);
            if (track) ut_insert(ut, f, ev);
          }
          w += __popc(mask);
          ins += __popc(mask);
        }
      }
    }
  }
  {  // set(): the taken action's tiles that no later action cleared; one entry per distinct f
    int f = 0;
    if (!null_from) {
      f = b0 + P.ra_m[action];
      if (f >= (int)P.memory_size) f -= (int)P.memory_size;
    }
    bool add = null_from ? (action == P.n_actions - 1) : (ptt_last_writer(tt, f) == action);
    const unsigned same = __match_any_sync(FULL, f);
    add = add && ((__ffs(same) - 1) == lane);
    const unsigned mask = __ballot_sync(FULL, add);
    const int pos = w + __popc(mask & ((1u << lane) - 1u));
    int total = w + __popc(mask);
    if (total > P.trace_cap) {
      if (lane == 0) e.err |= ERR_TRACE_OVERFLOW;
      add = add && (pos < P.trace_cap);
      total = P.trace_cap;
    }
    if (track && ins + __popc(mask) > UT_MAX_ENTRIES) LN_UT_FLUSH();
    if (add) {
      __stcg(tf + pos, f);
      __stcg(te + pos, 1.0f);
      red_add_f64(theta + f, scaled_update * (double)1.0f);
      if (track) ut_insert(ut, f, 1.0f);
    }
    w = total;
  }
#undef LN_UT_FLUSH
  __syncwarp();
  return w;
}

// Q-learning's TD step, warp-wide (QLearn::UpdateTraces / UpdateWeights, agent.cpp:272-292); every lane returns the
// same values.  qpre = this lane's Q(to, lane); q_pre_s = the same values in shared memory.
__device__ __forceinline__ void ln_td_qlearn(AgentD& ag, double qpre, const double* q_pre_s, const DynParams& D, int lane, float& rate,
                                             double& scaled) {
  const int action = ag.cur_action;
  const double qf = (lane < P.n_actions) ? ag.q_from[lane] : 0.0;
  const int amax = ln_argmax(ag, qf, ag.q_from, lane);
  rate = (action != amax) ? 0.0f : P.gl;
  const int am2 = ln_argmax(ag, qpre, q_pre_s, lane);
  const double F_term = P.gamma * 0.0 - 0.0;  // potentials are 0 (base.cpp:239-242)
  const double Q = ag.q_from[action];
  const double delta = ag.last_reward + F_term + P.gamma * q_pre_s[am2] - Q;
  __syncwarp();  // (every lane has read last_delta's neighbours before lane 0 writes)
  if (lane == 0) ag.last_delta = delta;
  scaled = (D.alpha * delta) * (1.0 / (double)RLM_N_TILINGS);
}

// Q of this lane's (table, action) -> Q_A / Q_B(from, .) of the agent block
template <bool DBL>
__device__ __forceinline__ void ln_store_q(AgentD& ag, double q, int lane) {
  const int al = lane & 15;
  if (al < P.n_actions) {
    if (lane < 16) { ag.q_from[al] = q; if (!DBL) ag.qb_from[al] = 0.0; }
    else if (DBL) ag.qb_from[al] = q;
  }
}

// One learner step of env `env` by one warp.  stage 0: whole step (independent policies); 1 / 2: the two halves of a
// shared-policy tick (see agent_process_env).  Written as "up to two evaluations, then the update" so that the hashing,
// gather and sum code exists once (instruction-cache footprint is time here):
//   kind 1 (end of warm-up)      : Q(first from-state, .) -> q_from (null State, or the previous episode's stale State)
//   stage 2, kind 0              : Q(to, .) under theta_{t+1} -> q_from; to-state becomes the from-state
//   stage 1, kind 0              : Q(from, .) under theta_t -> q_from (agent.cpp:274,285 read theta at update time), then
//   stage 0 / 1, kind 0 ("main") : Q(to, .), TD error, trace pass / weight update, [stage 0: Q(to, .) again -> q_from]
// RESIDENT: the env record (and `ag` = its agent block) lives in this warp's shared memory (fused engine): nothing is
// staged or written back, and the parity record is filled from `hdr`; otherwise `hdr` is unused.
// GB: gathers in flight per lane and table (27 = all of them; 9 = one feature group at a time, for kernels compiled
// with a small register budget)
template <bool DBL, bool RESIDENT, int GB>
__device__ __forceinline__ void ln_step(const DevPtrs& ptr, const DynParams& D, int env, AgentD& ag, unsigned char* scr, const EnvHdr* hdr, int lane,
                                        int stage, unsigned long long& steps_done, unsigned long long& sum_z, int tp_idx) {
  LPH(0);
  double* V = (double*)scr;
  int* tt = (int*)(scr + ln_v_bytes(DBL ? 1 : 0));
  int* ut = tt + TT_SLOTS;
  double* q_pre_a = (double*)(ut + 2 * UT_SLOTS);
  double* q_pre_b = q_pre_a + RLM_MAX_ACTIONS;
  double* dec = q_pre_b + RLM_MAX_ACTIONS;
  const unsigned* rnd = rlm_rndseq_table;
  const int A = P.n_actions;
  EnvHdr* g = (EnvHdr*)(ptr.env + (size_t)env * P.env_stride);
  constexpr int N16 = (int)(AG_BYTES / 16);
  static_assert(N16 > 32 && N16 <= 64, "two 16-byte loads per lane cover the agent block");
  if (!RESIDENT) {
    const int4* src = (const int4*)&g->ag;
    int4* dst = (int4*)&ag;
    const int4 t0 = __ldcg(src + lane);
    int4 t1 = make_int4(0, 0, 0, 0);
    if (lane + 32 < N16) t1 = __ldcg(src + lane + 32);
    dst[lane] = t0;
    if (lane + 32 < N16) dst[lane + 32] = t1;
  }
  __syncwarp();
  LPH(1);
  if (ag.kind == 0 && stage != 2) {
    // The trace list (read by the trace pass) and the three words of the Mersenne Twister state the next draw touches are
    // in HBM since the env's previous step: ask L2 for them now, they arrive under the hashing, the gathers and the sums.
    const int n_tr = ag.n_traces;
    const int* tf0 = ptr.trace_f + (size_t)env * P.trace_cap;
    const float* te0 = ptr.trace_e + (size_t)env * P.trace_cap;
    if (lane * 32 < n_tr) {
      asm volatile("prefetch.global.L2 [%0];" ::"l"(tf0 + lane * 32));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(te0 + lane * 32));
    }
    if (P.algorithm != RLM_ALGO_Q_LEARN && lane < 3) {
      int k = ag.mt_pol_idx; if (k >= 312) k -= 312;
      int kk = k + (lane == 0 ? 0 : (lane == 1 ? 1 : 156)); if (kk >= 312) kk -= 312;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr.mt_pol + (size_t)env * 312 + kk));
      if (ptr.mt_agt) {
        int a = ag.mt_agt_idx; if (a >= 312) a -= 312;
        int aa = a + (lane == 0 ? 0 : (lane == 1 ? 1 : 156)); if (aa >= 312) aa -= 312;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr.mt_agt + (size_t)env * 312 + aa));
      }
    }
  }
  const size_t pol = P.shared_policy ? 0 : (size_t)env;
  double* theta_a = ptr.theta + pol * (size_t)P.memory_size;
  double* theta_b = DBL ? ptr.theta_b + pol * (size_t)P.memory_size : nullptr;
#ifdef RLM_TIMING  // what-if switches (results are wrong): 1 = every env gathers from ONE 512 KB table, 2 = no fence,
  //                  4 = no re-read of updated weights before the second evaluation
  if (D.debug_flags & 1) theta_a = ptr.theta;
  const bool dbg_nofence = D.debug_flags & 2, dbg_nopatch = D.debug_flags & 4;
#else
  const bool dbg_nofence = false, dbg_nopatch = false;
#endif
  const int kind = ag.kind;
  const int al = lane & 15;  // action of this lane in the sums (lanes 16.. = table B)
  const bool do_main = (stage != 2) && (kind == 0);
  const bool do_pre = (stage == 2) ? (kind == 0) : (kind == 1 || (kind == 0 && stage == 1));
  const int n_evals = (do_pre ? 1 : 0) + (do_main ? 1 : 0);
  LnSums h;
  h.s[0] = h.s[1] = h.s[2] = 0ull; h.null_state = true;
  double q = 0.0;
#pragma unroll 1
  for (int ev = 0; ev < n_evals; ++ev) {
    const bool is_main = do_main && (ev == n_evals - 1);
    const float* vars = (is_main || stage == 2) ? ag.to_vars : ag.from_vars;
    // (kind 1: the never-populated State in a Learner's first episode, the previous episode's stale State afterwards)
    const bool null_state = is_main ? false : ((kind == 1 || stage == 1) ? ag.null_from != 0 : false);
    if (is_main && ag.hs_valid) {  // the tick kernel hashed the to-state (and prefetched its tiles)
      const unsigned long long* hs = ptr.hsum + (size_t)env * 96;
      h.s[0] = __ldcg(hs + lane); h.s[1] = __ldcg(hs + 32 + lane); h.s[2] = __ldcg(hs + 64 + lane);
      h.null_state = false;
    } else {
      h = ln_hash(rnd, vars, null_state, lane);
    }
    LPH(2);
    if (DBL || GB != 27) {
      if (is_main) ln_tt_build(tt, ag, lane);
      ln_gather<DBL, GB>(theta_a, theta_b, h, lane, V);
    } else {
      double v[3 * RLM_MAX_ACTIONS];
      ln_gather_issue<0, 27>(theta_a, h, v);
      LPH(3);
      if (is_main) ln_tt_build(tt, ag, lane);  // under the gathers' round trip
      LPH(4);
      ln_gather_store<0, 27>(v, lane, V);
    }
    __syncwarp();
    LPH(5);
    q = ln_sums(V, DBL, lane);
    __syncwarp();
    LPH(6);
    if (!is_main) {
      ln_store_q<DBL>(ag, q, lane);
      if (kind == 1) {
        if (!null_state) ag.from_base0[lane] = mod_m(h.s[0]);
        if (lane == 0) { ag.need_begin = 1; ag.kind = 2; }
      } else if (stage == 2) {  // the to-state becomes the from-state
        if (lane < RLM_N_STATE_MAX + 3) { ag.prev_vars[lane] = ag.from_vars[lane]; ag.from_vars[lane] = ag.to_vars[lane]; }
        ag.from_base0[lane] = mod_m(h.s[0]);
        if (lane == 0) { ag.prev_null = ag.null_from; ag.null_from = 0; ag.n_steps++; ag.ep_step++; ag.need_begin = 1; }
        steps_done++;
      }
      __syncwarp();
    }
  }
  if (do_main) {
    const double qpre = q;
    if (al < A) { if (lane < 16) q_pre_a[al] = qpre; else q_pre_b[al] = DBL ? qpre : 0.0; }
    __syncwarp();
    float rate;
    double scaled;
    int table = 0;
    if (!DBL && P.algorithm == RLM_ALGO_Q_LEARN) {
      ln_td_qlearn(ag, qpre, q_pre_a, D, lane, rate, scaled);
    } else {
      if (lane == 0)
        td_decision(ag, q_pre_a, q_pre_b, ptr.mt_pol + (size_t)env * 312, ptr.mt_agt ? ptr.mt_agt + (size_t)env * 312 : nullptr, D, dec);
      __syncwarp();
      rate = (float)dec[0];
      scaled = dec[1];
      table = (DBL && dec[2] != 0.0) ? 1 : 0;
    }
    __syncwarp();
    LPH(7);
    int* tf = ptr.trace_f + (size_t)env * P.trace_cap;
    float* te = ptr.trace_e + (size_t)env * P.trace_cap;
    double* th = table ? theta_b : theta_a;
    if (stage == 1) th = table ? ptr.dtheta + P.memory_size : ptr.dtheta;  // accumulate, apply after the all-reduce
    const bool local_patch = (stage == 0) && !dbg_nopatch;
    if (local_patch) { ut_clear(ut, lane); __syncwarp(); }
    const int nz = ln_trace_pass(ag, tt, ut, local_patch, tf, te, th, ag.cur_action, rate, scaled, lane, h,
                                 V + (table ? RLM_MAX_ACTIONS * LN_VROW : 0));
    if (lane == 0) { ag.n_traces = nz; ag.sum_traces += nz; ag.hs_valid = 0; }
    sum_z += (lane == 0) ? (unsigned long long)nz : 0ull;
    __syncwarp();
    LPH(8);
    // theta updates (L2 reductions) are ordered before re-reads: only the parity record and an overfull update table need them
    if (env < P.record_envs && !dbg_nofence) __threadfence();
    LPH(9);
    if (env < P.record_envs) { if (RESIDENT) emit_record_res(ptr, hdr, env, ag, theta_a, ag.to_vars, lane); else emit_record_ool(ptr, g, env, ag, theta_a, ag.to_vars, lane); }
    if (stage == 0) {
      // the to-state becomes the from-state; Q(from, .) under the UPDATED theta (serial.cpp:55,60)
      if (lane < RLM_N_STATE_MAX + 3) { ag.prev_vars[lane] = ag.from_vars[lane]; ag.from_vars[lane] = ag.to_vars[lane]; }
      ag.from_base0[lane] = mod_m(h.s[0]);
      if (lane == 0) { ag.prev_null = ag.null_from; ag.null_from = 0; ag.n_steps++; ag.ep_step++; ag.need_begin = 1; }
      steps_done++;
      LPH(13);
      if (local_patch) ln_patch_local(ut, scaled, h.s[0], h.s[1], h.s[2], h.null_state, lane, V + (table ? RLM_MAX_ACTIONS * LN_VROW : 0));  // the last batch of updates
      LPH(14);
      __syncwarp();
      LPH(10);
      q = ln_sums(V, DBL, lane);
      ln_store_q<DBL>(ag, q, lane);
      LPH(11);
    }
  }
  __syncwarp();
  if (!RESIDENT) {
    int4* dst = (int4*)&g->ag;
    const int4* src = (const int4*)&ag;
    __stcg(dst + lane, src[lane]);
    if (lane + 32 < N16) __stcg(dst + lane + 32, src[lane + 32]);
    // the env's next tick starts with the action selection (begin_step): its generator draw reads three words of the
    // Mersenne Twister state in HBM -- ask L2 for them now instead of paying a DRAM round trip on lane 0 of the tick kernel
    if (lane < 3 && ag.need_begin) {
      int k = ag.mt_pol_idx; if (k >= 312) k -= 312;
      int kk = k + (lane == 0 ? 0 : (lane == 1 ? 1 : 156)); if (kk >= 312) kk -= 312;
      asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr.mt_pol + (size_t)env * 312 + kk));
    }
  }
  __syncwarp();
  LPH(12);
#ifdef RLM_TIMING
  if (lane == 0 && tp_idx < 4096) { unsigned s_; asm volatile("mov.u32 %0, %%smid;" : "=r"(s_)); g_phase_sm[tp_idx] = s_; }
#endif
}

template <bool DBL>
__global__ void __launch_bounds__(LN_WARPS * 32, LN_MIN_CTAS) rlm_learn_kernel(DevPtrs ptr, DynParams D, int tslot, int stage) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char* wsm = smem + (size_t)warp * ln_warp_bytes(DBL ? 1 : 0);
  // the 8 KB hashing table is read at random through L1, which is cold at launch: pull its 64 lines in now, under the
  // ready-count and agent-block round trips, instead of missing on them one dependent batch at a time while hashing
  for (int i = threadIdx.x; i < 64; i += LN_WARPS * 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(rlm_rndseq_table + i * 32));
  const int n_ready = ptr.ready_count[tslot];
  unsigned long long steps_done = 0, sum_z = 0;
  if (n_ready > (int)blockIdx.x) KLOG_BEGIN(1);
  // ready env k goes to warp (k / gridDim.x) of CTA (k % gridDim.x): a short list spreads evenly over all SMs.  (Measured:
  // packing the list into the fewest CTAs instead -- every working CTA with all its warps at work -- leaves some SMs with
  // 12 steps and others with 8, and the launch waits for the fullest SM: 82 us instead of 75.)
  const int C = gridDim.x;
#pragma unroll 1
  for (int idx = warp * C + blockIdx.x; idx < n_ready; idx += LN_WARPS * C)
    ln_step<DBL, false, 27>(ptr, D, ptr.ready[idx], *(AgentD*)wsm, wsm + LN_AG_BYTES, nullptr, lane, stage, steps_done, sum_z, idx);
  if (steps_done) KLOG_END(1);
  if (lane == 0 && (steps_done | sum_z)) {
    atomicAdd(&ptr.counters[1], steps_done);
    atomicAdd(&ptr.counters[2], sum_z);
  }
}

cudaError_t rlm_launch_learn(const DevPtrs& ptr, const DynParams& D, int n_envs, int is_double, int tslot, int n_sms, int stage, int expected_steps, cudaStream_t st) {
  const size_t smem = LN_WARPS * ln_warp_bytes(is_double);
  static size_t attr_smem[2] = {0, 0};
  if (smem > attr_smem[is_double ? 1 : 0]) {
    cudaError_t e = is_double ? cudaFuncSetAttribute(rlm_learn_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                              : cudaFuncSetAttribute(rlm_learn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (is_double) cudaFuncSetAttribute(rlm_learn_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, RLM_SMEM_CARVEOUT);
    else cudaFuncSetAttribute(rlm_learn_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, RLM_SMEM_CARVEOUT);
    attr_smem[is_double ? 1 : 0] = smem;
  }
  int grid = (n_envs + LN_WARPS - 1) / LN_WARPS;  // worst case: every env is ready
  static int per_sm[2] = {0, 0};                  // resident CTAs per SM (shared memory bound)
  if (!per_sm[is_double ? 1 : 0]) {
    int n = 0;
    cudaError_t e = is_double ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, rlm_learn_kernel<true>, LN_WARPS * 32, smem)
                              : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, rlm_learn_kernel<false>, LN_WARPS * 32, smem);
    per_sm[is_double ? 1 : 0] = (e == cudaSuccess && n > 0) ? n : 1;
  }
  // one resident wave; the grid-stride loop takes the rest.  RLM_LEARN_CTAS_PER_SM leaves room for the tick kernel of
  // another sub-batch on the same SMs (round-paced engine with several streams)
  static int per_sm_cap = -1;
  if (per_sm_cap < 0) { const char* e = getenv("RLM_LEARN_CTAS_PER_SM"); per_sm_cap = e ? atoi(e) : 0; }
  int ps = per_sm[is_double ? 1 : 0];
  if (per_sm_cap > 0 && per_sm_cap < ps) ps = per_sm_cap;
  // no more CTAs per SM than the steps this launch usually finds need (measured at C1, ~1 200 steps per tick: 3 CTAs per
  // SM 74.4 us, 4 CTAs 75.6 us; a round's ~2 300 steps want all four)
  if (expected_steps > 0) ps = std::max(1, std::min(ps, (expected_steps + LN_WARPS * n_sms - 1) / (LN_WARPS * n_sms)));
  const int cap = n_sms * ps;
  if (grid > cap) grid = cap;
  if (is_double) rlm_learn_kernel<true><<<grid, LN_WARPS * 32, smem, st>>>(ptr, D, tslot, stage);
  else rlm_learn_kernel<false><<<grid, LN_WARPS * 32, smem, st>>>(ptr, D, tslot, stage);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Fused persistent engine (the default for independent-policy training): ONE launch per rlm_run_ticks call, one warp
// per env for all `n_ticks` ticks.  The env record stays in shared memory for the whole launch; the warp runs the market
// tick (envw_tick) and, whenever its env's midprice has moved, the learner step (ln_step) and the next action selection
// inline.  Envs never wait for each other -- there is no per-tick barrier, no ready list and no launch per tick -- so the
// DRAM bursts of the gathers of some warps overlap the scalar book logic of the others (measured: the per-tick launch
// pair leaves the memory system idle for the whole env kernel and the SMs idle for the whole gather burst).
// Learner scratch (~12 KB) is not per warp: a CTA shares FU2_SLOTS of them, since only ~1 env in 8 is inside a learner
// step at any time; a warp takes a free slot (shared-memory CAS) for the duration of its step.
#define FU2_WARPS 14
#define FU2_SLOTS 4
__host__ __device__ inline size_t fu2_smem_bytes(int is_double) {
  return (size_t)FU2_WARPS * envw_warp_bytes() + 16 * 4 + (size_t)FU2_SLOTS * ln_scratch_bytes(is_double);
}

template <bool DBL>
__global__ void __launch_bounds__(FU2_WARPS * 32, 2) rlm_fused2_kernel(DevPtrs ptr, DynParams D) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int* slot_busy = (int*)(smem + (size_t)FU2_WARPS * envw_warp_bytes());
  unsigned char* slots = (unsigned char*)(slot_busy + 16);
  if (tid < 16) slot_busy[tid] = 0;
  __syncthreads();  // (the only block barrier: before any warp can exit)
  const int env = blockIdx.x * FU2_WARPS + warp;
  if (env >= P.n_envs) return;
  const EnvWarp w = envw_carve(smem + (size_t)warp * envw_warp_bytes());
  EnvHdr& e = *w.e;
  EnvHdr* g = (EnvHdr*)(ptr.env + (size_t)env * P.env_stride);
  double* ring = (double*)((unsigned char*)g + sizeof(EnvHdr));
  if (g->phase == PH_DONE) return;
  envw_stage_in(&e, g, lane);
  __syncwarp();
  unsigned ticked = 0;
  unsigned long long steps_done = 0, sum_z = 0;
  unsigned long long* mt_pol = ptr.mt_pol + (size_t)env * 312;
#ifdef RLM_TIMING  // per env: [0] cycles in ticks, [1] ticks, [2] cycles waiting for a slot, [3] cycles in learner steps, [4] steps, [5] begin_step cycles
  long long fu_t[6] = {0, 0, 0, 0, 0, 0};
#define FUT(i, ...) do { const long long c0_ = clock64(); __VA_ARGS__; fu_t[i] += clock64() - c0_; } while (0)
#else
#define FUT(i, ...) do { __VA_ARGS__; } while (0)
#endif
  if (e.ag.need_begin) {  // (left pending by the tick-synchronous engine)
    if (lane == 0) { begin_step(e, mt_pol, D); e.ag.need_begin = 0; }
    __syncwarp();
  }
#pragma unroll 1
  for (int t = 0; t < D.n_ticks; ++t) {
    if (e.phase == PH_DONE) break;
    int ready;
    FUT(0, ready = envw_tick(w, ring, ptr, D, env, D.stream_off + t, D.stream_ticks, lane, ticked));
#ifdef RLM_TIMING
    fu_t[1]++;
#endif
    if (P.source == RLM_SOURCE_STREAM && D.stream_off + t >= D.stream_ticks) break;
    if (ready < 0) continue;
    // a learner step (or the end of warm-up): borrow a scratch slot of the CTA
    int slot = -1;
    FUT(2, {
      if (lane == 0) {
        while (true) {
#pragma unroll
          for (int k = 0; k < FU2_SLOTS; ++k) {
            const int s = (warp + k) % FU2_SLOTS;
            if (slot < 0 && atomicCAS(&slot_busy[s], 0, 1) == 0) slot = s;
          }
          if (slot >= 0) break;
          __nanosleep(200);
        }
      }
      slot = __shfl_sync(FULL, slot, 0);
    });
    FUT(3, {
      ln_step<DBL, true, 9>(ptr, D, env, e.ag, slots + (size_t)slot * ln_scratch_bytes(DBL ? 1 : 0), &e, lane, 0, steps_done, sum_z, 4096);
      __syncwarp();
    });
#ifdef RLM_TIMING
    fu_t[4]++;
#endif
    if (lane == 0) atomicExch(&slot_busy[slot], 0);
    FUT(5, {
      if (lane == 0) {
        begin_step(e, mt_pol, D);  // serial.cpp:55-61: the next action, DoAction, first reward term
        e.ag.need_begin = 0;
      }
      __syncwarp();
    });
  }
  __syncwarp();
  envw_stage_out(g, &e, lane);
#ifdef RLM_TIMING
  if (lane == 0 && env < 4096) for (int i = 0; i < 6; ++i) g_phase_clk[env * 16 + i] = fu_t[i];
#endif
  if (lane == 0) {
    if (ticked) atomicAdd(&ptr.counters[0], (unsigned long long)ticked);
    if (steps_done | sum_z) { atomicAdd(&ptr.counters[1], steps_done); atomicAdd(&ptr.counters[2], sum_z); }
    const unsigned errs = (unsigned)(e.err | e.ag.err);
    if (errs) atomicOr(&ptr.counters[4], (unsigned long long)errs);
  }
}

cudaError_t rlm_launch_fused2(const DevPtrs& ptr, const DynParams& D, int n_envs, int is_double, cudaStream_t st) {
  const size_t smem = fu2_smem_bytes(is_double);
  static size_t attr_smem[2] = {0, 0};
  if (smem > attr_smem[is_double ? 1 : 0]) {
    cudaError_t e = is_double ? cudaFuncSetAttribute(rlm_fused2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                              : cudaFuncSetAttribute(rlm_fused2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr_smem[is_double ? 1 : 0] = smem;
  }
  const int grid = (n_envs + FU2_WARPS - 1) / FU2_WARPS;
  if (is_double) rlm_fused2_kernel<true><<<grid, FU2_WARPS * 32, smem, st>>>(ptr, D);
  else rlm_fused2_kernel<false><<<grid, FU2_WARPS * 32, smem, st>>>(ptr, D);
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Learner step with the env's WHOLE weight table staged in shared memory by the bulk-copy engine (TMA, 1-D
// cp.async.bulk + mbarrier): small per-env tables (memory_size * 8 <= 64 KB: BASELINE.json configs[4], 1M LOBs with
// M = 4096).  Measured on B200 (tools/ubench/gather.cu): a coalesced 32 KB window streams at 6.6-7.0 TB/s, while the 864
// random 32-byte sectors the gather form of the step needs inside the same window complete at 2.9 TB/s of sector traffic
// -- and hold the SM's miss tracking hostage.  Here one elected lane issues ONE bulk copy per step; the hashing, the
// tile-index table and the from-state's tile table are built while it is in flight; both evaluations, the trace pass
// and the weight update then run against shared memory: the updated weights are written through to HBM (plain stores of
// the sums the L2 reduction would have produced), and the second evaluation simply walks the updated table -- no
// gathers, no reductions, no fence, no patching.  One warp per CTA, one CTA per ready env at a time.
#define LS_IROW 104  // u16 tile indices per action row (96 used; 16-byte aligned rows)
__host__ __device__ inline size_t ls_fixed_bytes() { return 16 + LN_AG_BYTES + (size_t)RLM_MAX_ACTIONS * LS_IROW * 2 + TT_SLOTS * 4 + 8 * 2 * RLM_MAX_ACTIONS + 48; }
__host__ __device__ inline size_t ls_smem_bytes(long long memory_size) { return ((ls_fixed_bytes() + 15) & ~(size_t)15) + (size_t)memory_size * 8; }

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

// exact-order sum of agent.cpp:117-135 for one action: weights come from the staged table through the index row
__device__ __forceinline__ double ls_chain(const double* tab, const unsigned short* irow) {
  const double w0 = P.gw[0], w1 = P.gw[1], w2 = P.gw[2];
  double acc = 0.0, cur[8], nxt[8];
  {
    const uint4 i8 = *(const uint4*)irow;
    const unsigned short* ii = (const unsigned short*)&i8;
#pragma unroll
    for (int j = 0; j < 8; ++j) cur[j] = w0 * tab[ii[j]];
  }
#pragma unroll 1
  for (int b = 1; b <= 16; ++b) {
    const int nb = (b < 16) ? b : 0;
    const double w = (nb < 4) ? w0 : ((nb < 8) ? w1 : w2);
    const int col = (nb < 8) ? 8 * nb : 8 * (nb - 4);
    const uint4 i8 = *(const uint4*)(irow + col);
    const unsigned short* ii = (const unsigned short*)&i8;
#pragma unroll
    for (int j = 0; j < 8; ++j) nxt[j] = w * tab[ii[j]];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc += cur[j];
#pragma unroll
    for (int j = 0; j < 8; ++j) cur[j] = nxt[j];
  }
  return acc;
}
__device__ __noinline__ double ls_sums(const double* tab, const unsigned short* idx, int lane) {
  ASSUME_SHARED(tab); ASSUME_SHARED(idx);
  return (lane < P.n_actions) ? ls_chain(tab, idx + lane * LS_IROW) : 0.0;
}

__global__ void __launch_bounds__(32, 6) rlm_learn_staged_kernel(DevPtrs ptr, DynParams D, int tslot) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int lane = threadIdx.x;
  unsigned long long* mbar = (unsigned long long*)smem;
  AgentD& ag = *(AgentD*)(smem + 16);
  unsigned short* idx_s = (unsigned short*)(smem + 16 + LN_AG_BYTES);
  int* tt = (int*)(idx_s + RLM_MAX_ACTIONS * LS_IROW);
  double* q_pre_a = (double*)(tt + TT_SLOTS);
  double* q_pre_b = q_pre_a + RLM_MAX_ACTIONS;
  double* dec = q_pre_b + RLM_MAX_ACTIONS;
  double* tab = (double*)(smem + ((ls_fixed_bytes() + 15) & ~(size_t)15));
  const unsigned mbar_a = smem_u32(mbar), tab_a = smem_u32(tab);
  const unsigned table_bytes = (unsigned)(P.memory_size * 8);
  if (lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar_a) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  unsigned parity = 0;
  const int n_ready = ptr.ready_count[tslot];
  const int A = P.n_actions;
  const unsigned* rnd = rlm_rndseq_table;
  unsigned long long steps_done = 0, sum_z = 0;
  constexpr int N16 = (int)(AG_BYTES / 16);
#pragma unroll 1
  for (int idx = blockIdx.x; idx < n_ready; idx += gridDim.x) {
    const int env = ptr.ready[idx];
    EnvHdr* g = (EnvHdr*)(ptr.env + (size_t)env * P.env_stride);
    double* theta = ptr.theta + (size_t)env * (size_t)P.memory_size;
    // every lane is done with the previous env's table and index rows; order those generic-proxy accesses before the
    // bulk copy's async-proxy writes
    __syncwarp();
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar_a), "r"(table_bytes) : "memory");
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(tab_a), "l"(theta),
                   "r"(table_bytes), "r"(mbar_a)
                   : "memory");
    }
    {
      const int4* src = (const int4*)&g->ag;
      int4* dst = (int4*)&ag;
      const int4 t0 = __ldcg(src + lane);
      int4 t1 = make_int4(0, 0, 0, 0);
      if (lane + 32 < N16) t1 = __ldcg(src + lane + 32);
      dst[lane] = t0;
      if (lane + 32 < N16) dst[lane + 32] = t1;
    }
    __syncwarp();
    const int kind = ag.kind;
    const bool main_step = kind == 0;
    if (main_step) {  // (see ln_step: the trace list and the generator words, asked for now)
      const int n_tr = ag.n_traces;
      if (lane * 32 < n_tr) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr.trace_f + (size_t)env * P.trace_cap + lane * 32));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr.trace_e + (size_t)env * P.trace_cap + lane * 32));
      }
    }
    // ---- tile indices of the state to evaluate (to-state; first from-state at the end of warm-up), under the copy
    LnSums h;
    const bool null_state = (kind == 1) && ag.null_from != 0;
    if (main_step && ag.hs_valid) {
      const unsigned long long* hs = ptr.hsum + (size_t)env * 96;
      h.s[0] = __ldcg(hs + lane); h.s[1] = __ldcg(hs + 32 + lane); h.s[2] = __ldcg(hs + 64 + lane);
      h.null_state = false;
    } else {
      h = ln_hash(rnd, main_step ? ag.to_vars : ag.from_vars, null_state, lane);
    }
    if (P.m_pow2) {
#pragma unroll
      for (int k = 0; k < 3 * RLM_MAX_ACTIONS; ++k)
        if ((k % RLM_MAX_ACTIONS) < A) idx_s[(k % RLM_MAX_ACTIONS) * LS_IROW + (k / RLM_MAX_ACTIONS) * 32 + lane] = (unsigned short)ln_tile<true>(h, k);
    } else {
#pragma unroll
      for (int k = 0; k < 3 * RLM_MAX_ACTIONS; ++k)
        if ((k % RLM_MAX_ACTIONS) < A) idx_s[(k % RLM_MAX_ACTIONS) * LS_IROW + (k / RLM_MAX_ACTIONS) * 32 + lane] = (unsigned short)ln_tile<false>(h, k);
    }
    if (main_step) ln_tt_build(tt, ag, lane);
    __syncwarp();
    {  // the table has landed
      unsigned done = 0;
      while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(mbar_a), "r"(parity) : "memory");
      parity ^= 1u;
    }
    double q = ls_sums(tab, idx_s, lane);
    if (kind == 1) {
      if (lane < A) { ag.q_from[lane] = q; ag.qb_from[lane] = 0.0; }
      if (!null_state) ag.from_base0[lane] = mod_m(h.s[0]);
      if (lane == 0) { ag.need_begin = 1; ag.kind = 2; }
    } else if (main_step) {
      if (lane < A) { q_pre_a[lane] = q; q_pre_b[lane] = 0.0; }
      __syncwarp();
      float rate;
      double scaled;
      if (P.algorithm == RLM_ALGO_Q_LEARN) {
        ln_td_qlearn(ag, q, q_pre_a, D, lane, rate, scaled);
      } else {
        if (lane == 0) td_decision(ag, q_pre_a, q_pre_b, ptr.mt_pol + (size_t)env * 312, nullptr, D, dec);
        __syncwarp();
        rate = (float)dec[0];
        scaled = dec[1];
      }
      __syncwarp();
      // ---- Traces::decay + Traces::update + Agent::updateQ (see ln_trace_pass), weights updated in the staged table
      int* tf = ptr.trace_f + (size_t)env * P.trace_cap;
      float* te = ptr.trace_e + (size_t)env * P.trace_cap;
      const bool null_from = ag.null_from != 0;
      const int action = ag.cur_action;
      int w = 0;
      if (rate != 0.0f) {
        const int n = ag.n_traces;
#pragma unroll 1
        for (int base = 0; base < n; base += 32 * TR_AHEAD) {
          int fq[TR_AHEAD];
          float eq[TR_AHEAD];
#pragma unroll
          for (int k = 0; k < TR_AHEAD; ++k) {
            const int i = base + 32 * k + lane;
            fq[k] = (i < n) ? __ldcg(tf + i) : 0;
            eq[k] = (i < n) ? __ldcg(te + i) : 0.0f;
          }
#pragma unroll
          for (int k = 0; k < TR_AHEAD; ++k) {
            if (base + 32 * k < n) {
              const int i = base + 32 * k + lane;
              const int f = fq[k];
              const float ev = eq[k] * rate;
              bool keep = (i < n) && !(ev < 0.01f);
              if (keep) keep = (null_from ? (f == 0 ? A - 1 : -1) : ptt_last_writer(tt, f)) < 0;
              const unsigned mask = __ballot_sync(FULL, keep);
              const int pos = w + __popc(mask & ((1u << lane) - 1u));
              if (keep) {
                __stcg(tf + pos, f);
                __stcg(te + pos, ev);
                const double nv = tab[f] + scaled * (double)ev;  // the addition the L2 reduction performs
                tab[f] = nv;
                __stcg(theta + f, nv);
              }
              w += __popc(mask);
            }
          }
        }
      }
      {
        int f = 0;
        if (!null_from) {
          f = ag.from_base0[lane] + P.ra_m[action];
          if (f >= (int)P.memory_size) f -= (int)P.memory_size;
        }
        bool add = null_from ? (action == A - 1) : (ptt_last_writer(tt, f) == action);
        const unsigned same = __match_any_sync(FULL, f);
        add = add && ((__ffs(same) - 1) == lane);
        const unsigned mask = __ballot_sync(FULL, add);
        const int pos = w + __popc(mask & ((1u << lane) - 1u));
        int total = w + __popc(mask);
        if (total > P.trace_cap) {
          if (lane == 0) ag.err |= ERR_TRACE_OVERFLOW;
          add = add && (pos < P.trace_cap);
          total = P.trace_cap;
        }
        if (add) {
          __stcg(tf + pos, f);
          __stcg(te + pos, 1.0f);
          const double nv = tab[f] + scaled * (double)1.0f;
          tab[f] = nv;
          __stcg(theta + f, nv);
        }
        w = total;
      }
      __syncwarp();
      if (lane == 0) { ag.n_traces = w; ag.sum_traces += w; ag.hs_valid = 0; }
      sum_z += (lane == 0) ? (unsigned long long)w : 0ull;
      if (env < P.record_envs) { __threadfence(); emit_record_ool(ptr, g, env, ag, theta, ag.to_vars, lane); }
      // the to-state becomes the from-state; Q(from, .) under the UPDATED table (serial.cpp:55,60)
      if (lane < RLM_N_STATE_MAX + 3) { ag.prev_vars[lane] = ag.from_vars[lane]; ag.from_vars[lane] = ag.to_vars[lane]; }
      ag.from_base0[lane] = mod_m(h.s[0]);
      if (lane == 0) { ag.prev_null = ag.null_from; ag.null_from = 0; ag.n_steps++; ag.ep_step++; ag.need_begin = 1; }
      steps_done++;
      __syncwarp();
      q = ls_sums(tab, idx_s, lane);
      if (lane < A) { ag.q_from[lane] = q; ag.qb_from[lane] = 0.0; }
    }
    __syncwarp();
    {
      int4* dst = (int4*)&g->ag;
      const int4* src = (const int4*)&ag;
      __stcg(dst + lane, src[lane]);
      if (lane + 32 < N16) __stcg(dst + lane + 32, src[lane + 32]);
      if (lane < 3 && ag.need_begin) {  // (see ln_step: the generator words of the next action selection)
        int k = ag.mt_pol_idx; if (k >= 312) k -= 312;
        int kk = k + (lane == 0 ? 0 : (lane == 1 ? 1 : 156)); if (kk >= 312) kk -= 312;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr.mt_pol + (size_t)env * 312 + kk));
      }
    }
  }
  if (lane == 0 && (steps_done | sum_z)) {
    atomicAdd(&ptr.counters[1], steps_done);
    atomicAdd(&ptr.counters[2], sum_z);
  }
}

// staged form: independent policies, one table per env of at most 64 KB with 16-bit tile indices
__host__ inline bool rlm_learn_staged_ok(long long memory_size, int is_double, int shared_policy) {
  return !is_double && !shared_policy && memory_size * 8 <= 65536 && memory_size <= 65536 && (memory_size % 2) == 0;
}
cudaError_t rlm_launch_learn_staged(const DevPtrs& ptr, const DynParams& D, int n_envs, long long memory_size, int tslot, int n_sms, cudaStream_t st) {
  const size_t smem = ls_smem_bytes(memory_size);
  static size_t attr_smem = 0;
  static int per_sm = 1;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(rlm_learn_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cudaFuncSetAttribute(rlm_learn_staged_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    int n = 0;
    per_sm = (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, rlm_learn_staged_kernel, 32, smem) == cudaSuccess && n > 0) ? n : 1;
    attr_smem = smem;
  }
  int grid = n_envs;
  const int cap = n_sms * per_sm;
  if (grid > cap) grid = cap;
  rlm_learn_staged_kernel<<<grid, 32, smem, st>>>(ptr, D, tslot);
  return cudaGetLastError();
}
