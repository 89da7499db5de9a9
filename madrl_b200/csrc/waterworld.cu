// MAWaterWorld batched engine: persistent warp-per-env rollout kernel for sm_100a.
//
// Reference semantics: madrl_environments/pursuit/waterworld.py (cited as ww:LINE).
//
// Design (see DESIGN.md):
//   * One WARP owns one env for the WHOLE T-step rollout.  The env's state lives in REGISTERS:
//     lane l holds objects l, l+32, ... (position + velocity); objects are ordered pursuers,
//     evaders, poisons.  There is no shared memory and no block barrier anywhere: warps are
//     completely independent, so the SM's schedulers overlap the phases of different envs.
//     HBM sees the state once per launch (a coalesced per-env record) and, per step, only
//     actions in and obs / reward / done / info out.
//   * Per step and pursuer, lanes act first as OBJECTS (relative position, squared distance,
//     collision test and exact conservative range cull, all reduced with __ballot_sync), then as
//     SENSORS (lane k = sensor k) looping over the few surviving candidates, whose geometry is
//     broadcast with __shfl_sync; nearest-object-per-sensor keeps the lowest index among equal
//     minima (np.argmin).  The 7 feature rows of the pursuer are stored as coalesced
//     feature-major runs straight from registers.
//   * sqrt-free thresholds: every `cdist(...) <= thr` of the reference is evaluated as
//     d2 <= thr2 with thr2 the largest representable value whose correctly-rounded sqrt is
//     <= thr (computed on the host), which is exactly equivalent.
//   * fp32 production instantiation and fp64 verification instantiation of the same template.
#include <math.h>
#include <cmath>
#include <new>

#include "common.cuh"
#include "philox.cuh"
#include "host_pipeline.cuh"

namespace madrl {

template <typename real>
struct WWParams {
  int E, env_id_base, Np, Ne, Npo, K, n_coop, D, Nall;
  int reward_global, addid, speed_features, random_obstacle, timestep_limit, max_path_length;
  int T, mode, auto_reset;  // mode 0 = rollout, 1 = reset
  // element strides of one lockstep step in the trajectory tensors (host-computed so that the
  // per-step pointer bumps are plain 64-bit adds on constant-bank operands)
  size_t obs_step, agent_step;   // E*Np*D and E*Np
  real r_p2, range, cull2;                           // sensing thresholds (ww:68-69)
  real range_up;                                     // nextafter(range, +inf): `sv < range_up` <=> `sv <= range`
  real coll2_e, coll2_po;                            // (r_p + r_obj) as exact squared thresholds
  real obst2_p, obst2_e, obst2_po;                   // (r_class + R_obst)       ww:251,259,267
  real resp2_p, resp2_e, resp2_po;                   // (2 r_class + R_obst)     ww:140
  real obst_x, obst_y, ev_speed, poison_speed, action_scale;
  real poison_reward, food_reward, encounter_reward, control_penalty;
  uint64_t seed;
  // state: per-env records
  real* objs;         // [E][4][Nall]  (x, y, vx, vy rows)
  real* obst;         // [E][2]
  int32_t *timestep, *path_len;
  uint64_t* ctr;
  const real* sensors;  // [2][K]
  // trajectory tensors
  const real* actions;
  real* obs;
  real* rew;
  uint8_t* done;
  int32_t* info;
  const uint8_t* mask;
  real* term_obs;   // optional [T][E][A][D]: terminal observations of done steps (see keep_terminal_rows)
  // in-kernel action source (POLICY instantiation, madrl_ww_rollout_heuristic): the reference's hand-written
  // policy (heuristics/waterworld.py:11-53) closes the loop inside the launch -- no action tensor is read
  const real* policy_obs0;   // [E][Np][D] the observation the FIRST action is computed from
  real* actions_out;         // [T][E][Np][2] the actions taken (NULL = not recorded)
  // fused per-rollout exchange (multi-GPU): every rank also stores its reward / done / info rows
  // into slot `peer_rank` of each destination gather buffer through NVLink peer mappings (CUDA
  // IPC).  Rows are staged in registers and written as coalesced runs (rewards every 32/Np steps,
  // done/info every 32 steps) into an ENV-major layout [slot][E][Tmax][...], because thousands of
  // 4-byte remote stores per step cost far more than the bytes they carry.
  int n_peers, peer_rank, peer_tmax;
  real* peer_rew[8];
  uint8_t* peer_done[8];
  int32_t* peer_info[8];
};

template <typename real> struct Vec2;
template <> struct Vec2<float> { typedef float2 type; };
template <> struct Vec2<double> { typedef double2 type; };

template <typename real>
__device__ __forceinline__ real warp_sum(real v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}

// 0 <= sv < best for best > 0, in one comparison for float: non-negative floats order like their bit patterns
// and every negative one has the sign bit set, i.e. compares above any positive `best` as an unsigned integer.
// (-0.0 would be rejected where `sv < 0` is false, but sx * jx + sy * jy in round-to-nearest only yields -0.0
// from two negative-zero terms, and neither a position difference nor a product with one can be -0.0 here.)
__device__ __forceinline__ bool in_zero_to(float sv, float best) { return __float_as_uint(sv) < __float_as_uint(best); }
__device__ __forceinline__ bool in_zero_to(double sv, double best) { return !(sv < 0.0) && sv < best; }

template <typename real>
struct Spawn { real x, y, vx, vy; uint64_t ctr; };

// ww:139-142 + ww:360-374: rejection-sample a position outside the obstacle's keep-out disc,
// then (optionally) a velocity.  Executed warp-uniformly (every lane runs the same stream), so
// no broadcast is needed; rare, hence not inlined into the hot loop.
template <typename real>
__device__ __noinline__ Spawn<real> spawn_object(uint64_t seed, uint32_t env_id, uint64_t ctr,
                                                 real obx, real oby, real thr2, real speed,
                                                 int with_velocity) {
  SeqStream rs;
  rs.init(seed, env_id, 0u, ctr);
  Spawn<real> s;
  s.x = rs.next_unit<real>();
  s.y = rs.next_unit<real>();
  while (true) {
    const real dx = s.x - obx, dy = s.y - oby;
    if (!(dx * dx + dy * dy <= thr2)) break;
    s.x = rs.next_unit<real>();
    s.y = rs.next_unit<real>();
  }
  s.vx = 0; s.vy = 0;
  if (with_velocity) {
    s.vx = (rs.next_unit<real>() - (real)0.5) * speed;
    s.vy = (rs.next_unit<real>() - (real)0.5) * speed;
  }
  s.ctr = rs.counter;
  return s;
}

// OPL = objects per lane (ceil(n_obj / 32)); KCH = sensors per lane (ceil(K / 32));
// KC = compile-time sensor count (0 = runtime p.K): with KC known the 7 feature-row stores of a
// pursuer use immediate offsets from one running pointer instead of 64-bit address arithmetic.
// PEER = compile the fused multi-GPU exchange in (a separate instantiation, so the single-GPU kernel
// carries none of its registers).
// POLICY = the actions come from the in-kernel heuristic policy instead of the action tensor (again a
// separate instantiation: the open-loop kernel carries none of its instructions).
template <typename real, int OPL, int KCH, int KC, bool PEER, bool POLICY = false>
__global__ void __launch_bounds__(32, (OPL <= 4 ? 28 : 16))
ww_kernel(const __grid_constant__ WWParams<real> p) {
  const real INF = real_inf<real>();
  const int K = KC > 0 ? KC : p.K;
  // 32-thread blocks: the env index derives from blockIdx alone, so ptxas can prove every loop and
  // branch on it warp-uniform -- no BRA.DIV guards in front of the warp collectives, loop bookkeeping
  // on the uniform datapath, 72 -> 56 registers (measured +4 % on C2/C4, profiles/r2_ab_variants.log).
  const int lane = threadIdx.x;
  const int warp_global = blockIdx.x;
  const int warp_stride = gridDim.x;
  const int eLo = p.Np, eHi = p.Np + p.Ne, Nall = p.Nall;
  constexpr bool SMEM = OPL >= 2;
  const unsigned lt_mask = lanemask_lt();
  extern __shared__ __align__(16) unsigned char ww_smem[];
  // this warp's candidate slots (32-bit shared address)
  uint32_t slots = SMEM ? smem_addr(ww_smem) : 0u;
  asm volatile("" : "+r"(slots));   // keep it in a register: ptxas otherwise re-derives it from SR_CgaCtaId at every use

  // ---- per-lane constants: this lane as OBJECT (classes, thresholds) and as SENSOR -----------
  real cull2_l[OPL], coll2_l[OPL];
  unsigned mE[OPL], mP[OPL], mU[OPL];  // warp-uniform class masks of each object chunk
#pragma unroll
  for (int c = 0; c < OPL; ++c) {
    const int o = lane + 32 * c;
    const bool isU = o < eLo, isE = o >= eLo && o < eHi, isP = o >= eHi && o < Nall;
    cull2_l[c] = p.cull2;   // uniform: lanes beyond the last object hold a far-away sentinel position instead
    coll2_l[c] = isE ? p.coll2_e : (isP ? p.coll2_po : (real)-1);
    mU[c] = __ballot_sync(FULL_MASK, isU);
    mE[c] = __ballot_sync(FULL_MASK, isE);
    mP[c] = __ballot_sync(FULL_MASK, isP);
  }
  real sx_l[KCH], sy_l[KCH];
#pragma unroll
  for (int kc = 0; kc < KCH; ++kc) {
    const int k = lane + 32 * kc;
    sx_l[kc] = (k < K) ? p.sensors[k] : (real)0;
    sy_l[kc] = (k < K) ? p.sensors[K + k] : (real)0;
  }
  // the compile-time-K instantiation is also the speed_features = True one (the reference's defaults: K = 30, 7 rows
  // per sensor): no layout branch per pursuer; every other combination takes the KC = 0 instantiation
  const bool speed = KC > 0 ? true : (p.speed_features != 0);
  const int n_feat = speed ? 7 : 4;
  typedef typename Vec2<real>::type V2;

  for (int e = warp_global; e < p.E; e += warp_stride) {
    if (p.mode == 1 && p.mask != nullptr && p.mask[e] == 0) continue;
    const uint32_t env_id = (uint32_t)(p.env_id_base + e);
    // ---- state: HBM record -> registers -----------------------------------------------------
    real x[OPL], y[OPL], vx[OPL], vy[OPL];
    unsigned col[OPL];  // per object: bit q set <=> pursuer q collides with it this step
    real* rec = p.objs + (size_t)e * 4 * Nall;
#pragma unroll
    for (int c = 0; c < OPL; ++c) {
      const int o = lane + 32 * c;
      const bool v = o < Nall;
      x[c] = v ? rec[o] : (real)1e18;            // sentinel: never in range of anything, never written back
      y[c] = v ? rec[Nall + o] : (real)1e18;
      vx[c] = v ? rec[2 * Nall + o] : (real)0;
      vy[c] = v ? rec[3 * Nall + o] : (real)0;
      col[c] = 0u;
    }
    real obx = p.obst[2 * (size_t)e], oby = p.obst[2 * (size_t)e + 1];
    int tt = p.timestep[e], ts = p.path_len[e];
    uint64_t ctr = p.ctr[e];

    // running output pointers (this lane's column of the env's first pursuer row at step t)
    real* obs_t = p.obs + (size_t)e * p.Np * p.D + lane;
    real* rew_t = p.rew + (size_t)e * p.Np + lane;
    size_t te = (size_t)e;   // index of (t, e) in the [T][E] done / info tensors
    int pass = (p.mode == 1) ? 1 : 0;  // pass 1 = reset pass: fresh draws, zero action, obs only
    const V2* act_t = reinterpret_cast<const V2*>(p.actions) + (size_t)e * p.Np + lane;

    // POLICY: un-normalised action of pursuer `lane` for the NEXT step (heuristics/waterworld.py:25-44),
    // first from the caller's observation, afterwards from the features this warp has just computed
    real pax = 0, pay = 0;
    if constexpr (POLICY) {
      const real* o0 = p.policy_obs0 + (size_t)e * p.Np * p.D;
      for (int pi = 0; pi < p.Np; ++pi, o0 += p.D) {
        const real cE = o0[7 * K] > (real)0 ? (real)1.5 : (real)1;        // heuristics/waterworld.py:41
        const real cP = o0[7 * K + 1] > (real)0 ? (real)1.5 : (real)1;    // :42
        real wx = 0, wy = 0;
#pragma unroll
        for (int kc = 0; kc < KCH; ++kc) {
          const int k = lane + 32 * kc;
          if (k < K) {
            const real w = (real)0.5 * o0[5 * K + k] + (cE * o0[K + k] - o0[k]) - cP * o0[3 * K + k];
            wx += w * sx_l[kc]; wy += w * sy_l[kc];
          }
        }
        wx = warp_sum(wx); wy = warp_sum(wy);
        if (lane == pi) { pax = wx; pay = wy; }
      }
    }

    // staging registers of the fused exchange
    const int rew_per = 32 / p.Np;                       // steps per coalesced reward run
    const int stage_src = lane % p.Np, stage_step = lane / p.Np;
    const size_t peer_env = (size_t)p.peer_rank * p.E + e;
    real st_rew = 0, r_stage = 0;
    int2 st_info = make_int2(0, 0);
    uint8_t st_done = 0;
    int sc_rew = 0;

    V2 act_nx;
    act_nx.x = 0; act_nx.y = 0;
    if (!POLICY && p.mode == 0 && lane < p.Np) act_nx = *act_t;
    for (int t = 0; t < p.T; ++t) {
      V2 act;
      act.x = 0; act.y = 0;
      if constexpr (POLICY) {
        if (lane < p.Np) {   // heuristics/waterworld.py:44-50: unit vector, or zero when nothing is sensed
          // scaled by the larger component first: the squares of a tiny sum (cancellation leaves ~1e-21) would be
          // denormal in float32 and the "unit" vector off by 1e-4
          const real m = fmax(fabs(pax), fabs(pay));
          if (m > (real)0) {
            const real ux = pax / m, uy = pay / m, n = sqrt(ux * ux + uy * uy);
            act.x = ux / n; act.y = uy / n;
          }
          if (p.actions_out != nullptr)
            reinterpret_cast<V2*>(p.actions_out)[(size_t)t * p.agent_step + (size_t)e * p.Np + lane] = act;
        }
      } else if (p.mode == 0 && lane < p.Np) {
        // double-buffered in registers: the load for step t+1 is issued at the top of step t, so its HBM
        // latency hides behind a whole step (prefetch.global.L1 did not: the first use of the action was 10 % of
        // all stall samples of the C2 kernel; C2 66 -> 74.5 % of the roofline, profiles/r2_ab_action_db.log)
        act = act_nx;
        if (t + 1 < p.T) act_nx = act_t[p.agent_step];
      }
      bool need_reset;
      do {
        if (pass) {
          // ---- reset draws, ww:144-170 (obstacle, pursuers, evaders, poisons) ----------------
          tt = 0; ts = 0;
          if (p.random_obstacle) {
            SeqStream rs;
            rs.init(p.seed, env_id, 0u, ctr);
            obx = rs.next_unit<real>();
            oby = rs.next_unit<real>();
            ctr = rs.counter;
          } else {
            obx = p.obst_x; oby = p.obst_y;
          }
          for (int o = 0; o < Nall; ++o) {
            const bool oU = o < eLo, oE = !oU && o < eHi;
            // ww:164,170 -- poisons also use ev_speed at reset
            const Spawn<real> s = spawn_object<real>(p.seed, env_id, ctr, obx, oby,
                                                     oU ? p.resp2_p : (oE ? p.resp2_e : p.resp2_po),
                                                     p.ev_speed, oU ? 0 : 1);
            ctr = s.ctr;
#pragma unroll
            for (int c = 0; c < OPL; ++c)
              if (o == lane + 32 * c) { x[c] = s.x; y[c] = s.y; vx[c] = s.vx; vy[c] = s.vy; }
          }
          act.x = 0; act.y = 0;
        }
        // ---- integrate pursuers, control penalty, walls: ww:221-245 (pursuers = chunk 0) -------
        real pen;
        {
          real sq = 0;
          if (lane < p.Np) {
            const real ax = act.x * p.action_scale, ay = act.y * p.action_scale;
            vx[0] += ax; vy[0] += ay;
            x[0] += vx[0]; y[0] += vy[0];
            sq = ax * ax + ay * ay;
            const real cx = clip01(x[0]), cy = clip01(y[0]);
            if (x[0] != cx) vx[0] = 0;
            if (y[0] != cy) vy[0] = 0;
            x[0] = cx; y[0] = cy;
          }
          pen = p.control_penalty * (p.reward_global ? warp_sum(sq) : sq);
        }
        // ---- obstacle rebound (velocity only): ww:247-270 ----------------------------------------
#pragma unroll
        for (int c = 0; c < OPL; ++c) {
          const bool oE = (mE[c] >> lane) & 1u, oP = (mP[c] >> lane) & 1u, oU = (mU[c] >> lane) & 1u;
          const real thr = oU ? p.obst2_p : (oE ? p.obst2_e : (oP ? p.obst2_po : (real)-1));
          const real kf = oP ? (real)-1 : (real)-0.5;                  // ww:254,262,270
          const real dx = x[c] - obx, dy = y[c] - oby;
          if (dx * dx + dy * dy <= thr) { vx[c] = kf * vx[c]; vy[c] = kf * vy[c]; }
        }
        // ---- sense: one pursuer at a time -----------------------------------------------------
        real* obs_row = obs_t;
        for (int pi = 0; pi < p.Np; ++pi, obs_row += p.D) {
          const real mx = __shfl_sync(FULL_MASK, x[0], pi), my = __shfl_sync(FULL_MASK, y[0], pi);
          const real mvx = __shfl_sync(FULL_MASK, vx[0], pi), mvy = __shfl_sync(FULL_MASK, vy[0], pi);
          // nearest sensed object per class and sensor chunk (ww:64-72, 312-334)
          real bO[KCH], bE[KCH], bP[KCH], bU[KCH];
          int iE[KCH], iP[KCH], iU[KCH];
          const real orx = obx - mx, ory = oby - my;
          const real od2 = orx * orx + ory * ory;
          real pwx = 0, pwy = 0;       // POLICY: this lane's share of pursuer pi's next action
          unsigned tE = 0u, tP = 0u;   // POLICY: evaders / poisons pursuer pi touches this step (obs[7K], obs[7K+1])
#pragma unroll
          for (int kc = 0; kc < KCH; ++kc) {
            bO[kc] = bE[kc] = bP[kc] = bU[kc] = INF;
            iE[kc] = iP[kc] = iU[kc] = 0;
            if (od2 <= p.cull2) {   // the obstacle is sensed like a point object (pursuer radius only)
              const real sv = sx_l[kc] * orx + sy_l[kc] * ory;
              const bool ok = !((sv < (real)0) | (sv > p.range) | (od2 - sv * sv > p.r_p2));
              bO[kc] = ok ? sv : INF;
            }
          }
          if constexpr (SMEM) {
            constexpr uint32_t S = CandSlot<real>::kStride;
            uint32_t endU = slots, nEc = 0u, top = slots;
#pragma unroll
            for (int c = 0; c < OPL; ++c) {
              // lanes as OBJECTS: geometry, collisions (ww:278-293), conservative range cull, staging
              const real rx = x[c] - mx, ry = y[c] - my;
              const real d2 = rx * rx + ry * ry;
              const bool near = d2 <= cull2_l[c] && !(c == 0 && lane == pi);   // ww:70-71 `same`
              const unsigned cm = __ballot_sync(FULL_MASK, near);
              const bool hit = d2 <= coll2_l[c];
              if (hit) col[c] |= 1u << pi;
              if constexpr (POLICY) { const unsigned hm = __ballot_sync(FULL_MASK, hit); tE |= hm & mE[c]; tP |= hm & mP[c]; }
              // slot = rank among the candidates in ascending object index (= lane + 32 c)
              if (near) CandSlot<real>::put(top + (uint32_t)__popc(cm & lt_mask) * S, rx, ry, d2, vx[c], vy[c]);
              if (c == 0) endU = slots + (uint32_t)__popc(cm & mU[0]) * S;   // pursuers live in chunk 0 (Np <= 32)
              nEc += (uint32_t)__popc(cm & mE[c]);
              top += (uint32_t)__popc(cm) * S;
            }
            __syncwarp();
            // lanes as SENSORS: classes are contiguous in object index, hence in slot order U, E, P
            const uint32_t endE = endU + nEc * S, endP = top;   // the poisons end the list
            const real up = p.range_up;   // `sv < up` <=> `sv <= range`; a best below `up` <=> sensed
            uint32_t aE[KCH], aP[KCH], aU[KCH];
#pragma unroll
            for (int kc = 0; kc < KCH; ++kc) { bE[kc] = bP[kc] = bU[kc] = up; aE[kc] = aP[kc] = aU[kc] = slots; }
#define MADRL_WW_SCAN(A0, A1, BEST, AT)                                                  \
  _Pragma("unroll 2")                                                                  \
  for (uint32_t a = (A0); a != (A1); a += S) {                                           \
    real jx, jy, jd;                                                                     \
    CandSlot<real>::geom(a, jx, jy, jd);                                                 \
    _Pragma("unroll") for (int kc = 0; kc < KCH; ++kc) {                                 \
      const real sv = sx_l[kc] * jx + sy_l[kc] * jy;                                     \
      /* ww:64-72: 0 <= sv (<= range, through the initial best) and within the pursuer's radius of the ray */ \
      if (in_zero_to(sv, BEST[kc]) && !(jd - sv * sv > p.r_p2)) { BEST[kc] = sv; AT[kc] = a; } \
    }                                                                                    \
  }
            MADRL_WW_SCAN(slots, endU, bU, aU)
            MADRL_WW_SCAN(endU, endE, bE, aE)
            MADRL_WW_SCAN(endE, endP, bP, aP)
#undef MADRL_WW_SCAN
#pragma unroll
            for (int kc = 0; kc < KCH; ++kc) {
              const real sx = sx_l[kc], sy = sy_l[kc];
              // features ww:312-353, 388-395: feature-major, sensor-minor
              const int k = lane + 32 * kc;
              const bool hO = bO[kc] < INF, hE = bE[kc] < up, hP = bP[kc] < up, hU = bU[kc] < up;
              const real z = (real)0;
              real* o = obs_row + 32 * kc;   // this lane's column
              if constexpr (POLICY) {
                if (k < K) {
                  const real w = (real)0.5 * (hU ? bU[kc] : z) + ((tE ? (real)1.5 : (real)1) * (hE ? bE[kc] : z) - (hO ? bO[kc] : z)) -
                                 (tP ? (real)1.5 : (real)1) * (hP ? bP[kc] : z);
                  pwx += w * sx; pwy += w * sy;
                }
              }
              if (speed) {
                // slot 0 is read when nothing was sensed; its (possibly stale) value is masked below
                real oEx, oEy, oPx, oPy, oUx, oUy;
                CandSlot<real>::vel(aE[kc], oEx, oEy);
                CandSlot<real>::vel(aP[kc], oPx, oPy);
                CandSlot<real>::vel(aU[kc], oUx, oUy);
                if (k < K) {
                  store_stream(o + 0 * K, hO ? bO[kc] : z);
                  store_stream(o + 1 * K, hE ? bE[kc] : z);
                  store_stream(o + 2 * K, hE ? sx * (oEx - mvx) + sy * (oEy - mvy) : z);
                  store_stream(o + 3 * K, hP ? bP[kc] : z);
                  store_stream(o + 4 * K, hP ? sx * (oPx - mvx) + sy * (oPy - mvy) : z);
                  store_stream(o + 5 * K, hU ? bU[kc] : z);
                  store_stream(o + 6 * K, hU ? sx * (oUx - mvx) + sy * (oUy - mvy) : z);
                }
              } else if (k < K) {
                store_stream(o + 0 * K, hO ? bO[kc] : z);
                store_stream(o + 1 * K, hE ? bE[kc] : z);
                store_stream(o + 2 * K, hP ? bP[kc] : z);
                store_stream(o + 3 * K, hU ? bU[kc] : z);
              }
            }
            __syncwarp();   // the next pursuer's staging overwrites the slots
          } else {
#pragma unroll
          for (int c = 0; c < OPL; ++c) {
            // lanes as OBJECTS: geometry, collisions (ww:278-293), conservative range cull
            const real rx = x[c] - mx, ry = y[c] - my;
            const real d2 = rx * rx + ry * ry;
            unsigned cm = __ballot_sync(FULL_MASK, d2 <= cull2_l[c]);
            if (c == 0) cm &= ~(1u << pi);  // ww:70-71 `same`
            const bool hit = d2 <= coll2_l[c];
            if (hit) col[c] |= 1u << pi;
            if constexpr (POLICY) { const unsigned hm = __ballot_sync(FULL_MASK, hit); tE |= hm & mE[c]; tP |= hm & mP[c]; }
            // lanes as SENSORS: scan the surviving candidates of this chunk, ascending index
#pragma unroll
            for (int kc = 0; kc < KCH; ++kc) {
              const real sx = sx_l[kc], sy = sy_l[kc];
#define MADRL_WW_SCAN(MASK, BEST, IDX)                                                  \
  for (unsigned m = cm & (MASK); m != 0u; m &= m - 1u) {                                 \
    const int j = __ffs(m) - 1;                                                          \
    const real jx = __shfl_sync(FULL_MASK, rx, j), jy = __shfl_sync(FULL_MASK, ry, j);   \
    const real jd = __shfl_sync(FULL_MASK, d2, j);                                       \
    const real sv = sx * jx + sy * jy;                                                   \
    const bool ok = !((sv < (real)0) | (sv > p.range) | (jd - sv * sv > p.r_p2));        \
    if (ok && sv < BEST) { BEST = sv; IDX = j + 32 * c; }                                \
  }
              MADRL_WW_SCAN(mU[c], bU[kc], iU[kc])
              MADRL_WW_SCAN(mE[c], bE[kc], iE[kc])
              MADRL_WW_SCAN(mP[c], bP[kc], iP[kc])
#undef MADRL_WW_SCAN
            }
          }
#pragma unroll
          for (int kc = 0; kc < KCH; ++kc) {
            const real sx = sx_l[kc], sy = sy_l[kc];
            // features ww:312-353, 388-395: feature-major, sensor-minor
            const int k = lane + 32 * kc;
            const bool hO = bO[kc] < INF, hE = bE[kc] < INF, hP = bP[kc] < INF, hU = bU[kc] < INF;
            const real z = (real)0;
            real* o = obs_row + 32 * kc;   // this lane's column
            if constexpr (POLICY) {
              if (k < K) {
                const real w = (real)0.5 * (hU ? bU[kc] : z) + ((tE ? (real)1.5 : (real)1) * (hE ? bE[kc] : z) - (hO ? bO[kc] : z)) -
                               (tP ? (real)1.5 : (real)1) * (hP ? bP[kc] : z);
                pwx += w * sx; pwy += w * sy;
              }
            }
            if (speed) {
              real oEx, oEy, oPx, oPy, oUx, oUy;
              if (OPL == 1) {
                oEx = __shfl_sync(FULL_MASK, vx[0], iE[kc]); oEy = __shfl_sync(FULL_MASK, vy[0], iE[kc]);
                oPx = __shfl_sync(FULL_MASK, vx[0], iP[kc]); oPy = __shfl_sync(FULL_MASK, vy[0], iP[kc]);
                oUx = __shfl_sync(FULL_MASK, vx[0], iU[kc]); oUy = __shfl_sync(FULL_MASK, vy[0], iU[kc]);
              } else {
                oEx = oEy = oPx = oPy = oUx = oUy = z;
#pragma unroll
                for (int c = 0; c < OPL; ++c) {
                  const real ex_ = __shfl_sync(FULL_MASK, vx[c], iE[kc] & 31), ey_ = __shfl_sync(FULL_MASK, vy[c], iE[kc] & 31);
                  const real px_ = __shfl_sync(FULL_MASK, vx[c], iP[kc] & 31), py_ = __shfl_sync(FULL_MASK, vy[c], iP[kc] & 31);
                  const real ux_ = __shfl_sync(FULL_MASK, vx[c], iU[kc] & 31), uy_ = __shfl_sync(FULL_MASK, vy[c], iU[kc] & 31);
                  if ((iE[kc] >> 5) == c) { oEx = ex_; oEy = ey_; }
                  if ((iP[kc] >> 5) == c) { oPx = px_; oPy = py_; }
                  if ((iU[kc] >> 5) == c) { oUx = ux_; oUy = uy_; }
                }
              }
              if (k < K) {
                store_stream(o + 0 * K, hO ? bO[kc] : z);
                store_stream(o + 1 * K, hE ? bE[kc] : z);
                store_stream(o + 2 * K, hE ? sx * (oEx - mvx) + sy * (oEy - mvy) : z);
                store_stream(o + 3 * K, hP ? bP[kc] : z);
                store_stream(o + 4 * K, hP ? sx * (oPx - mvx) + sy * (oPy - mvy) : z);
                store_stream(o + 5 * K, hU ? bU[kc] : z);
                store_stream(o + 6 * K, hU ? sx * (oUx - mvx) + sy * (oUy - mvy) : z);
              }
            } else if (k < K) {
              store_stream(o + 0 * K, hO ? bO[kc] : z);
              store_stream(o + 1 * K, hE ? bE[kc] : z);
              store_stream(o + 2 * K, hP ? bP[kc] : z);
              store_stream(o + 3 * K, hU ? bU[kc] : z);
            }
          }
          }
          if constexpr (POLICY) {   // sum over the sensors; lane pi keeps pursuer pi's next action
            pwx = warp_sum(pwx); pwy = warp_sum(pwy);
            if (lane == pi) { pax = pwx; pay = pwy; }
          }
        }
        // ---- catches, respawn, rewards: ww:285,293,358-385 -----------------------------------------
        unsigned whoE = 0u, whoP = 0u, whoEnc = 0u;
        int nE = 0, nP = 0, nEnc = 0;
#pragma unroll
        for (int c = 0; c < OPL; ++c) {
          const int cnt = __popc(col[c]);
          // collisions needed to be caught: evaders n_coop (ww:285), poisons 1 (ww:293)
          const bool caught = ((mE[c] >> lane) & 1u) ? cnt >= p.n_coop : (((mP[c] >> lane) & 1u) && cnt >= 1);
          const unsigned cmk = __ballot_sync(FULL_MASK, caught);
          const unsigned enc = __ballot_sync(FULL_MASK, cnt >= 1) & mE[c];   // ww:376
          nE += __popc(cmk & mE[c]);
          nP += __popc(cmk & mP[c]);
          nEnc += __popc(enc);
          if (caught) { if ((mE[c] >> lane) & 1u) whoE |= col[c]; else whoP |= col[c]; }
          if ((enc >> lane) & 1u) whoEnc |= col[c];
          col[c] = 0u;
          for (unsigned m = cmk; m != 0u; m &= m - 1u) {   // ascending index: evaders, then poisons
            const int j = __ffs(m) - 1;
            const bool jE = (mE[c] >> j) & 1u;
            const Spawn<real> s = spawn_object<real>(p.seed, env_id, ctr, obx, oby,
                                                     jE ? p.resp2_e : p.resp2_po,
                                                     jE ? p.ev_speed : p.poison_speed, 1);
            ctr = s.ctr;
            if (lane == j) { x[c] = s.x; y[c] = s.y; vx[c] = s.vx; vy[c] = s.vy; }
          }
        }
        whoE = __reduce_or_sync(FULL_MASK, whoE);
        whoP = __reduce_or_sync(FULL_MASK, whoP);
        whoEnc = __reduce_or_sync(FULL_MASK, whoEnc);
        // ww:411-428 tail of every pursuer's row: [touched an evader, touched a poison, id]; lane i
        // writes pursuer i's.  whoEnc / whoP are exactly the any-collision masks (ww:376, ww:293).
        if (lane < p.Np) {
          real* tp = obs_t + (size_t)lane * (p.D - 1) + n_feat * K;   // obs_t already carries +lane
          store_stream(tp, (real)((whoEnc >> lane) & 1u));
          store_stream(tp + 1, (real)((whoP >> lane) & 1u));
          if (p.addid) store_stream(tp + 2, (real)(lane + 1));
        }
        if (!pass && lane < p.Np) {
          real r = pen;
          if (p.reward_global) {
            r += ((real)nE * p.food_reward + (real)nP * p.poison_reward) + (real)nEnc * p.encounter_reward;
          } else {   // fancy-index += : at most once per category (ww:383-385)
            if ((whoE >> lane) & 1u) r += p.food_reward;
            if ((whoP >> lane) & 1u) r += p.poison_reward;
            if ((whoEnc >> lane) & 1u) r += p.encounter_reward;
          }
          store_stream(rew_t, r);
          if (PEER) r_stage = r;
        }
        if (PEER && !pass && p.n_peers > 0) {   // stage this step's rewards: lane s*Np + a <- (step s, agent a)
          const real v = __shfl_sync(FULL_MASK, r_stage, stage_src);
          if (stage_step == sc_rew) st_rew = v;
          if (++sc_rew == rew_per) {
            if (lane < rew_per * p.Np) {
              const size_t off = (peer_env * p.peer_tmax + (size_t)(t + 1 - rew_per)) * p.Np + lane;
              for (int d = 0; d < p.n_peers; ++d) store_stream(p.peer_rew[d] + off, st_rew);
            }
            sc_rew = 0;
          }
        }
        // ---- evaders / poison drift; bounce only if BOTH coordinates left [0,1]: ww:397-409 ---------
#pragma unroll
        for (int c = 0; c < OPL; ++c) {
          if (((mE[c] | mP[c]) >> lane) & 1u) {
            x[c] += vx[c]; y[c] += vy[c];
            const bool ox = (x[c] < (real)0) || (x[c] > (real)1), oy = (y[c] < (real)0) || (y[c] > (real)1);
            if (ox && oy) { vx[c] = -vx[c]; vy[c] = -vy[c]; }
          }
        }
        // ---- bookkeeping ww:433-436 + VecEnvExecutor horizon ---------------------------------------
        tt += 1;
        need_reset = false;
        if (!pass) {
          ts += 1;
          const bool done = (tt >= p.timestep_limit) || (p.max_path_length > 0 && ts >= p.max_path_length);
          if (lane == 0) {
            p.done[te] = done ? 1 : 0;
            reinterpret_cast<int2*>(p.info)[te] = make_int2(nE, nP);
          }
          if (PEER && p.n_peers > 0) {  // stage done / info of step t in lane t % 32; flush every 32 steps
            if (lane == (t & 31)) { st_info = make_int2(nE, nP); st_done = done ? 1 : 0; }
            if ((t & 31) == 31 || t == p.T - 1) {
              if (lane <= (t & 31)) {
                const size_t off = peer_env * p.peer_tmax + (size_t)(t & ~31) + lane;
                for (int d = 0; d < p.n_peers; ++d) {
                  p.peer_done[d][off] = st_done;
                  reinterpret_cast<int2*>(p.peer_info[d])[off] = st_info;
                }
              }
            }
          }
          // VecEnvExecutor.step: a done env is reset in place and its obs slot receives the
          // reset observation (rllab/sandbox/rocky/tf/envs/vec_env_executor.py:24-27)
          need_reset = done && p.auto_reset;
          if (need_reset && p.term_obs != nullptr)
            keep_terminal_rows(obs_t - lane, p.term_obs + ((obs_t - lane) - p.obs), p.Np * p.D, lane);
        }
        pass = need_reset ? 1 : 0;
      } while (need_reset);
      obs_t += p.obs_step;
      act_t += p.agent_step;
      rew_t += p.agent_step;
      te += (size_t)p.E;
    }
    if (PEER && p.n_peers > 0 && sc_rew > 0 && lane < sc_rew * p.Np) {   // partial reward run at the end
      const size_t off = (peer_env * p.peer_tmax + (size_t)(p.T - sc_rew)) * p.Np + lane;
      for (int d = 0; d < p.n_peers; ++d) store_stream(p.peer_rew[d] + off, st_rew);
    }
    // ---- registers -> HBM record ------------------------------------------------------------------
#pragma unroll
    for (int c = 0; c < OPL; ++c) {
      const int o = lane + 32 * c;
      if (o < Nall) { rec[o] = x[c]; rec[Nall + o] = y[c]; rec[2 * Nall + o] = vx[c]; rec[3 * Nall + o] = vy[c]; }
    }
    if (lane == 0) {
      p.obst[2 * (size_t)e] = obx; p.obst[2 * (size_t)e + 1] = oby;
      p.timestep[e] = tt; p.path_len[e] = ts; p.ctr[e] = ctr;
    }
  }
}

}  // namespace madrl

// =================================================================================================
// Host side: C ABI
// =================================================================================================
using namespace madrl;

struct madrl_ww : EnvCore {
  madrl_ww_config cfg;
  madrl_ww_layout lay;
  // peer gather buffers (multi-GPU fused exchange); n_peers == 0: disabled
  int n_peers, peer_rank, peer_tmax;
  void* peer_rew[8];
  void* peer_done[8];
  void* peer_info[8];
};

static int ww_validate(const madrl_ww_config* c) {
  MADRL_REQUIRE(c != nullptr, "config is NULL");
  MADRL_REQUIRE(c->n_envs > 0, "n_envs must be > 0");
  MADRL_REQUIRE(c->n_pursuers >= 1 && c->n_pursuers <= 32,
                "n_pursuers must be in [1,32] (collision rows are 32-bit masks), got %d", c->n_pursuers);
  MADRL_REQUIRE(c->n_evaders >= 1 && c->n_poison >= 1, "n_evaders and n_poison must be >= 1");
  MADRL_REQUIRE(c->n_sensors >= 1 && c->n_sensors <= 64, "n_sensors must be in [1,64], got %d", c->n_sensors);
  MADRL_REQUIRE(c->n_pursuers + c->n_evaders + c->n_poison <= 256,
                "n_pursuers + n_evaders + n_poison must be <= 256 (8 objects per lane)");
  MADRL_REQUIRE(c->n_coop >= 1, "n_coop must be >= 1");
  MADRL_REQUIRE(c->timestep_limit >= 1, "timestep_limit must be >= 1");
  return MADRL_OK;
}

extern "C" int madrl_ww_state_layout(const madrl_ww_config* c, madrl_ww_layout* out) {
  int rc = ww_validate(c);
  if (rc) return rc;
  MADRL_REQUIRE(out != nullptr, "layout out is NULL");
  const size_t rb = c->fp64 ? 8 : 4, E = (size_t)c->n_envs;
  const size_t nobj = (size_t)c->n_pursuers + c->n_evaders + c->n_poison;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  out->rng_counter = take(8 * E);
  out->objs = take(rb * 4 * nobj * E);
  out->obst = take(rb * 2 * E);
  out->timestep = take(4 * E);
  out->path_len = take(4 * E);
  out->sensors = take(rb * 2 * (size_t)c->n_sensors);
  out->total_bytes = off;
  out->n_obj = (int32_t)nobj;
  out->obs_dim = c->n_sensors * (c->speed_features ? 7 : 4) + 2 + (c->addid ? 1 : 0);  // ww:18-24
  out->real_bytes = (int32_t)rb;
  out->_pad = 0;
  return MADRL_OK;
}

extern "C" int madrl_ww_create(const madrl_ww_config* c, void* state_dev, madrl_ww** out) {
  MADRL_REQUIRE(out != nullptr, "out is NULL");
  madrl_ww_layout lay;
  int rc = madrl_ww_state_layout(c, &lay);
  if (rc) return rc;
  madrl_ww* h = new (std::nothrow) madrl_ww();
  if (!h) return MADRL_ENOMEM;
  h->cfg = *c;
  h->lay = lay;
  h->n_peers = 0; h->peer_rank = 0; h->peer_tmax = 0;
  rc = core_init(h, state_dev, lay.total_bytes);
  if (!rc) rc = upload_sensor_table(h->state + lay.sensors, c->n_sensors, c->fp64);
  if (rc) { madrl_ww_destroy(h); return rc; }
  *out = h;
  return MADRL_OK;
}

extern "C" int madrl_ww_destroy(madrl_ww* h) {
  if (!h) return MADRL_OK;
  core_release(h);
  delete h;
  return MADRL_OK;
}

extern "C" void* madrl_ww_state_ptr(madrl_ww* h) { return h ? h->state : nullptr; }

extern "C" int madrl_ww_seed(madrl_ww* h, uint64_t seed, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  h->cfg.seed = seed;
  return core_clear_counters(h, h->lay.rng_counter, h->cfg.n_envs, stream);
}

extern "C" int madrl_ww_set_peers(madrl_ww* h, int n_peers, int rank, int t_max, void* const* rew_peers,
                                  void* const* done_peers, void* const* info_peers) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  MADRL_REQUIRE(n_peers >= 0 && n_peers <= 8, "n_peers must be in [0,8], got %d", n_peers);
  if (n_peers == 0) { h->n_peers = 0; return MADRL_OK; }
  MADRL_REQUIRE(rank >= 0 && t_max >= 1, "bad slot / t_max");
  MADRL_REQUIRE(rew_peers && done_peers && info_peers, "NULL peer pointer table");
  for (int d = 0; d < n_peers; ++d) {
    MADRL_REQUIRE(rew_peers[d] && done_peers[d] && info_peers[d], "NULL peer buffer %d", d);
    MADRL_REQUIRE(((uintptr_t)info_peers[d] & 7) == 0, "peer info buffer %d must be 8-byte aligned", d);
    h->peer_rew[d] = rew_peers[d]; h->peer_done[d] = done_peers[d]; h->peer_info[d] = info_peers[d];
  }
  h->n_peers = n_peers; h->peer_rank = rank; h->peer_tmax = t_max;
  return MADRL_OK;
}

extern "C" int madrl_ww_set_terminal_obs(madrl_ww* h, void* term_obs_dev) {
  return core_set_terminal_obs(h, term_obs_dev);
}

extern "C" int madrl_ww_set_launch(madrl_ww* h, int warps_per_block, int blocks_per_sm) {
  return core_set_launch(h, warps_per_block, blocks_per_sm);
}

template <typename real, int OPL, int KCH, int KC, bool PEER, bool POLICY>
static int ww_launch_inst2(madrl_ww* h, const WWParams<real>& p, cudaStream_t stream) {
  const size_t smem = OPL >= 2 ? (size_t)p.Nall * CandSlot<real>::kStride : 0;   // candidate slots
  return launch_persistent(h, ww_kernel<real, OPL, KCH, KC, PEER, POLICY>, p.E, smem, stream, p);
}

template <typename real, int OPL, int KCH, int KC>
static int ww_launch_inst(madrl_ww* h, const WWParams<real>& p, cudaStream_t stream) {
  if (p.policy_obs0 != nullptr) return ww_launch_inst2<real, OPL, KCH, KC, false, true>(h, p, stream);
  return p.n_peers > 0 ? ww_launch_inst2<real, OPL, KCH, KC, true, false>(h, p, stream)
                       : ww_launch_inst2<real, OPL, KCH, KC, false, false>(h, p, stream);
}

template <typename real>
static int ww_launch(madrl_ww* h, int mode, int T, const void* actions, void* obs, void* rew,
                     uint8_t* done, int32_t* info, const uint8_t* mask, int auto_reset,
                     cudaStream_t stream, const void* policy_obs0 = nullptr, void* actions_out = nullptr) {
  const madrl_ww_config& c = h->cfg;
  WWParams<real> p;
  p.E = c.n_envs; p.env_id_base = c.env_id_base;
  p.Np = c.n_pursuers; p.Ne = c.n_evaders; p.Npo = c.n_poison; p.K = c.n_sensors;
  p.n_coop = c.n_coop; p.D = h->lay.obs_dim; p.Nall = h->lay.n_obj;
  p.reward_global = c.reward_global; p.addid = c.addid; p.speed_features = c.speed_features;
  p.random_obstacle = c.random_obstacle; p.timestep_limit = c.timestep_limit;
  p.max_path_length = c.max_path_length;
  p.T = T; p.mode = mode; p.auto_reset = auto_reset;
  p.obs_step = (size_t)p.E * p.Np * p.D; p.agent_step = (size_t)p.E * p.Np;
  // radii ww:108-118 (double arithmetic as in the reference, then narrowed once)
  const double r_p = c.radius, r_e = c.radius * 2, r_po = c.radius * 3 / 4;
  p.r_p2 = (real)(r_p * r_p);
  p.range = (real)c.sensor_range;
  p.range_up = std::nextafter(p.range, (real)INFINITY);
  // Exact conservative cull: sv <= range and d2 - sv^2 <= r^2 imply d2 <= range^2 + r^2.
  p.cull2 = (real)((c.sensor_range * c.sensor_range + r_p * r_p) * (1.0 + 1e-4) + 1e-12);
  p.coll2_e = exact_sq_threshold<real>(r_p + r_e);
  p.coll2_po = exact_sq_threshold<real>(r_p + r_po);
  p.obst2_p = exact_sq_threshold<real>(r_p + c.obstacle_radius);
  p.obst2_e = exact_sq_threshold<real>(r_e + c.obstacle_radius);
  p.obst2_po = exact_sq_threshold<real>(r_po + c.obstacle_radius);
  p.resp2_p = exact_sq_threshold<real>(r_p * 2 + c.obstacle_radius);
  p.resp2_e = exact_sq_threshold<real>(r_e * 2 + c.obstacle_radius);
  p.resp2_po = exact_sq_threshold<real>(r_po * 2 + c.obstacle_radius);
  p.obst_x = (real)c.obstacle_x; p.obst_y = (real)c.obstacle_y;
  p.ev_speed = (real)c.ev_speed; p.poison_speed = (real)c.poison_speed;
  p.action_scale = (real)c.action_scale;
  p.poison_reward = (real)c.poison_reward; p.food_reward = (real)c.food_reward;
  p.encounter_reward = (real)c.encounter_reward; p.control_penalty = (real)c.control_penalty;
  p.seed = c.seed;
  char* st = h->state;
  p.objs = (real*)(st + h->lay.objs);
  p.obst = (real*)(st + h->lay.obst);
  p.timestep = (int32_t*)(st + h->lay.timestep); p.path_len = (int32_t*)(st + h->lay.path_len);
  p.ctr = (uint64_t*)(st + h->lay.rng_counter);
  p.sensors = (const real*)(st + h->lay.sensors);
  p.actions = (const real*)actions; p.obs = (real*)obs; p.rew = (real*)rew;
  p.done = done; p.info = info; p.mask = mask;
  p.term_obs = (mode == 0) ? (real*)h->term_obs : nullptr;
  p.policy_obs0 = (const real*)policy_obs0; p.actions_out = (real*)actions_out;
  // the policy instantiation is single-GPU: its rows go through the copy-engine exchange, not peer stores
  p.n_peers = (mode == 0 && policy_obs0 == nullptr) ? h->n_peers : 0;
  p.peer_rank = h->peer_rank;
  if (p.n_peers > 0) {
    MADRL_REQUIRE(T <= h->peer_tmax, "rollout of %d steps exceeds the peer buffers (t_max %d)", T, h->peer_tmax);
    p.peer_tmax = h->peer_tmax;
    for (int d = 0; d < 8; ++d) {
      p.peer_rew[d] = (real*)h->peer_rew[d % p.n_peers];
      p.peer_done[d] = (uint8_t*)h->peer_done[d % p.n_peers];
      p.peer_info[d] = (int32_t*)h->peer_info[d % p.n_peers];
    }
  }

  const int opl = (p.Nall + 31) / 32, kch = (p.K + 31) / 32;
#define MADRL_WW_CASE(O, KH, KC_) return ww_launch_inst<real, O, KH, KC_>(h, p, stream)
  if (p.K == 30 && p.speed_features) {   // the reference's defaults (n_sensors = 30, speed features): compile-time K and layout
    if (opl == 1) MADRL_WW_CASE(1, 1, 30);
    if (opl == 2) MADRL_WW_CASE(2, 1, 30);
    if (opl <= 4) MADRL_WW_CASE(4, 1, 30);
    MADRL_WW_CASE(8, 1, 30);
  } else if (kch == 1) {
    if (opl == 1) MADRL_WW_CASE(1, 1, 0);
    if (opl == 2) MADRL_WW_CASE(2, 1, 0);
    if (opl <= 4) MADRL_WW_CASE(4, 1, 0);
    MADRL_WW_CASE(8, 1, 0);
  } else {
    if (opl == 1) MADRL_WW_CASE(1, 2, 0);
    if (opl == 2) MADRL_WW_CASE(2, 2, 0);
    if (opl <= 4) MADRL_WW_CASE(4, 2, 0);
    MADRL_WW_CASE(8, 2, 0);
  }
#undef MADRL_WW_CASE
}

extern "C" int madrl_ww_reset(madrl_ww* h, const uint8_t* mask_dev, void* obs_dev, void* stream) {
  MADRL_REQUIRE(h != nullptr && obs_dev != nullptr, "handle/obs is NULL");
  return h->cfg.fp64 ? ww_launch<double>(h, 1, 1, nullptr, obs_dev, nullptr, nullptr, nullptr, mask_dev, 0, (cudaStream_t)stream)
                     : ww_launch<float>(h, 1, 1, nullptr, obs_dev, nullptr, nullptr, nullptr, mask_dev, 0, (cudaStream_t)stream);
}

extern "C" int madrl_ww_rollout(madrl_ww* h, int T, const void* actions_dev, void* obs_dev,
                                void* rew_dev, uint8_t* done_dev, int32_t* info_dev,
                                int auto_reset, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  MADRL_REQUIRE(T >= 1, "T must be >= 1");
  MADRL_REQUIRE(actions_dev && obs_dev && rew_dev && done_dev && info_dev, "NULL trajectory buffer");
  MADRL_REQUIRE(((uintptr_t)info_dev & 7) == 0, "info_dev must be 8-byte aligned (rows are stored as one 8-byte word)");
  return h->cfg.fp64 ? ww_launch<double>(h, 0, T, actions_dev, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream)
                     : ww_launch<float>(h, 0, T, actions_dev, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream);
}

extern "C" int madrl_ww_rollout_heuristic(madrl_ww* h, int T, const void* obs0_dev, void* actions_out_dev,
                                          void* obs_dev, void* rew_dev, uint8_t* done_dev, int32_t* info_dev,
                                          int auto_reset, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  MADRL_REQUIRE(T >= 1, "T must be >= 1");
  MADRL_REQUIRE(obs0_dev && obs_dev && rew_dev && done_dev && info_dev, "NULL trajectory buffer");
  MADRL_REQUIRE(((uintptr_t)info_dev & 7) == 0, "info_dev must be 8-byte aligned (rows are stored as one 8-byte word)");
  MADRL_REQUIRE(((uintptr_t)actions_out_dev & (h->cfg.fp64 ? 15 : 7)) == 0, "actions_out_dev must be aligned to one (x, y) pair");
  MADRL_REQUIRE(h->cfg.speed_features, "the heuristic policy reads the 7K feature layout (speed_features=True; "
                                       "heuristics/waterworld.py:12-22)");
  return h->cfg.fp64 ? ww_launch<double>(h, 0, T, nullptr, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream, obs0_dev, actions_out_dev)
                     : ww_launch<float>(h, 0, T, nullptr, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream, obs0_dev, actions_out_dev);
}

extern "C" int madrl_ww_step(madrl_ww* h, const void* actions_dev, void* obs_dev, void* rew_dev,
                             uint8_t* done_dev, int32_t* info_dev, int auto_reset, void* stream) {
  return madrl_ww_rollout(h, 1, actions_dev, obs_dev, rew_dev, done_dev, info_dev, auto_reset, stream);
}

// ---- host-buffer entry points -------------------------------------------------------------------
extern "C" int madrl_ww_reset_host(madrl_ww* h, const uint8_t* mask_host, void* obs_host) {
  MADRL_REQUIRE(h != nullptr && obs_host != nullptr, "handle/obs is NULL");
  const size_t E = h->cfg.n_envs;
  return core_reset_host(h, E, E * h->cfg.n_pursuers * h->lay.obs_dim * h->lay.real_bytes, mask_host, obs_host,
                         [&](uint8_t* mask_dev, char* obs_dev) { return madrl_ww_reset(h, mask_dev, obs_dev, nullptr); });
}

extern "C" int madrl_ww_rollout_host2(madrl_ww* h, int T, const void* actions_host, void* obs_host,
                                      void* rew_host, uint8_t* done_host, int32_t* info_host,
                                      int auto_reset, int flags) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  const size_t E = h->cfg.n_envs, Np = h->cfg.n_pursuers, rb = h->lay.real_bytes;
  const StepBytes sb = {E * Np * 2 * rb, E * Np * h->lay.obs_dim * rb, E * Np * rb, E, E * 2 * 4};
  return core_rollout_host(h, T, sb, actions_host, obs_host, rew_host, done_host, info_host, flags,
                           [&](int, int Tc, char* a, char* o, char* r, char* d, char* i, cudaStream_t st) {
                             return madrl_ww_rollout(h, Tc, a, o, r, (uint8_t*)d, (int32_t*)i, auto_reset, st);
                           });
}

extern "C" int madrl_ww_rollout_host(madrl_ww* h, int T, const void* actions_host, void* obs_host,
                                     void* rew_host, uint8_t* done_host, int32_t* info_host,
                                     int auto_reset) {
  return madrl_ww_rollout_host2(h, T, actions_host, obs_host, rew_host, done_host, info_host, auto_reset, 0);
}
