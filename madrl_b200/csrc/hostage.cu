// ContinuousHostageWorld batched engine: persistent warp-per-env rollout kernel for sm_100a.
//
// Reference semantics: madrl_environments/hostage.py (cited as hw:LINE).  Same kernel family as
// waterworld.cu: one warp owns one env for the whole T-step rollout, state in registers (lane l
// holds objects l, l+32, ...; objects ordered rescuers, criminals, hostages), lanes act as
// OBJECTS (geometry, collisions, range cull via __ballot_sync) and then as SENSORS (nearest
// criminal / hostage / key / bomb per sensor via __shfl_sync broadcasts); no shared memory, no
// block barriers; sqrt-free exact squared thresholds.  Reset draws have no rejection loops here,
// so every lane computes its own objects' draws directly from the counter-based stream.
#include <math.h>
#include <cmath>
#include <new>

#include "common.cuh"
#include "philox.cuh"
#include "host_pipeline.cuh"

namespace madrl {

template <typename real>
struct HWParams {
  int E, env_id_base, Nr, Nc, Nh, K, n_coop_save, D, Nall;
  int reward_global, addid, random_key, timestep_limit, max_path_length;
  int T, mode, auto_reset;
  size_t obs_step, agent_step;   // element strides of one lockstep step: E*Nr*D and E*Nr
  real r_r2, range, cull2;                    // sensing thresholds (hw:66-67)
  real coll2_c, coll2_h, coll2_bomb, coll2_key;  // exact squared collision thresholds (hw:269-296)
  real gate_lo;                               // 0.5 + radius (hw:257)
  real key_x, key_y, bad_speed, action_scale;
  real save_reward, hit_reward, encounter_reward, not_saved_reward, bomb_reward, control_penalty;
  uint64_t seed;
  // state: per-env records
  real* objs;        // [E][4][Nall]  rows x, y, vx, vy; rescuers, criminals, hostages
  real* fixed;       // [E][4]        key x, key y, bomb x, bomb y
  uint8_t* saved;    // [E][Nh]       curr_host_saved_mask
  int32_t* flags;    // [E]           bit0 gate open, bit1 bombed, bit2 key location drawn
  int32_t *timestep, *path_len;
  uint64_t* ctr;
  const real* sensors;
  // trajectory tensors
  const real* actions;
  real* obs;
  real* rew;
  uint8_t* done;
  int32_t* info;     // [T][E][2] = (ho_saved, cr_encs)
  const uint8_t* mask;
  real* term_obs;    // optional [T][E][Nr][D]: terminal observations of done steps (see keep_terminal_rows)
};

template <typename real> struct HVec2;
template <> struct HVec2<float> { typedef float2 type; };
template <> struct HVec2<double> { typedef double2 type; };

template <typename real>
__device__ __forceinline__ real hw_warp_sum(real v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}

template <typename real>
__device__ __forceinline__ real unit_at(uint64_t seed, uint32_t env_id, uint64_t n) {
  return (real)(stream_word(seed, env_id, 0u, n) >> 8) * (real)(1.0 / 16777216.0);
}

template <typename real, int OPL, int KCH, int KC>
__global__ void __launch_bounds__(32, (OPL <= 2 ? 28 : 16))
hw_kernel(const __grid_constant__ HWParams<real> p) {
  const real INF = real_inf<real>();
  const int K = KC > 0 ? KC : p.K;
  const int lane = threadIdx.x;
  const int warp_global = blockIdx.x;
  const int warp_stride = gridDim.x;
  const int cLo = p.Nr, hLo = p.Nr + p.Nc, Nall = p.Nall;
  // first object index held in the per-lane object registers (see 1)
  const int obase = p.Nr;

  real cull2_l[OPL], coll2_l[OPL];
  unsigned mC[OPL], mH[OPL];   // warp-uniform class masks (criminals, hostages) per object chunk
#pragma unroll
  for (int c = 0; c < OPL; ++c) {
    const int o = obase + lane + 32 * c;
    const bool isC = o >= cLo && o < hLo, isH = o >= hLo && o < Nall;
    cull2_l[c] = p.cull2;   // uniform: lanes beyond the last object hold a far-away sentinel position instead of a
                            // per-lane validity select (allies are sensed but never emitted, hw:395-397: they
                            // are not among the chunk objects)
    coll2_l[c] = isC ? p.coll2_c : (isH ? p.coll2_h : (real)-1);
    mC[c] = __ballot_sync(FULL_MASK, isC);
    mH[c] = __ballot_sync(FULL_MASK, isH);
  }
  real sx_l[KCH], sy_l[KCH];
#pragma unroll
  for (int kc = 0; kc < KCH; ++kc) {
    const int k = lane + 32 * kc;
    sx_l[kc] = (k < K) ? p.sensors[k] : (real)0;
    sy_l[kc] = (k < K) ? p.sensors[K + k] : (real)0;
  }
  typedef typename HVec2<real>::type V2;

  for (int e = warp_global; e < p.E; e += warp_stride) {
    if (p.mode == 1 && p.mask != nullptr && p.mask[e] == 0) continue;
    const uint32_t env_id = (uint32_t)(p.env_id_base + e);
    real x[OPL], y[OPL], vx[OPL], vy[OPL];
    unsigned col[OPL];
    bool sav[OPL];   // this lane's hostage is saved
    real* rec = p.objs + (size_t)e * 4 * Nall;
#pragma unroll
    for (int c = 0; c < OPL; ++c) {
      const int o = obase + lane + 32 * c;
      const bool v = o < Nall;
      x[c] = v ? rec[o] : (real)1e18;            // sentinel: never in range of anything, never written back
      y[c] = v ? rec[Nall + o] : (real)1e18;
      vx[c] = v ? rec[2 * Nall + o] : (real)0;
      vy[c] = v ? rec[3 * Nall + o] : (real)0;
      col[c] = 0u;
      sav[c] = (o >= hLo && o < Nall) ? (p.saved[(size_t)e * p.Nh + (o - hLo)] != 0) : false;
    }
    real rpx = 0, rpy = 0, rpvx = 0, rpvy = 0;   // rescuer `lane`
    if (lane < p.Nr) { rpx = rec[lane]; rpy = rec[Nall + lane]; rpvx = rec[2 * Nall + lane]; rpvy = rec[3 * Nall + lane]; }
    real kx = p.fixed[4 * (size_t)e], ky = p.fixed[4 * (size_t)e + 1];
    real bx = p.fixed[4 * (size_t)e + 2], by = p.fixed[4 * (size_t)e + 3];
    int flags = p.flags[e];
    int tt = p.timestep[e], ts = p.path_len[e];
    uint64_t ctr = p.ctr[e];

    real* obs_t = p.obs + (size_t)e * p.Nr * p.D + lane;
    real* rew_t = p.rew + (size_t)e * p.Nr + lane;
    size_t te = (size_t)e;
    int pass = (p.mode == 1) ? 1 : 0;
    const V2* act_t = reinterpret_cast<const V2*>(p.actions) + (size_t)e * p.Nr + lane;

    V2 act_nx;
    act_nx.x = 0; act_nx.y = 0;
    if (p.mode == 0 && lane < p.Nr) act_nx = *act_t;
    for (int t = 0; t < p.T; ++t) {
      V2 act;
      act.x = 0; act.y = 0;
      if (p.mode == 0 && lane < p.Nr) {
        // double-buffered in registers: the load for step t+1 is issued at the top of step t, so its HBM
        // latency hides behind a whole step (prefetch.global.L1 did not: the first use of the action was 10 % of
        // all stall samples of the C2 kernel; C2 66 -> 74.5 % of the roofline, profiles/r2_ab_action_db.log)
        act = act_nx;
        if (t + 1 < p.T) act_nx = act_t[p.agent_step];
      }
      bool need_reset;
      do {
        if (pass) {
          // ---- reset(): hw:142-177.  No rejection loops, so draw indices are known per object:
          // [key 2] rescuers 2 each, hostages 3 each, criminals 4 each, bomb 2. -----------------
          tt = 0; ts = 0;
          uint64_t n = ctr;
          if (p.random_key) {
            if (!(flags & 4)) {                                              // hw:148-151 drawn once
              kx = (real)1 - unit_at<real>(p.seed, env_id, n) * (real)0.1;
              ky = (real)1 - unit_at<real>(p.seed, env_id, n + 1) * (real)0.1;
              n += 2;
            }
          } else { kx = p.key_x; ky = p.key_y; }
          flags = 4;   // gate closed, not bombed, key known
          if (lane < p.Nr) {                                                 // hw:155-159
            const uint64_t b = n + 2 * (uint64_t)lane;
            rpx = unit_at<real>(p.seed, env_id, b);
            const real yy = unit_at<real>(p.seed, env_id, b + 1);
            rpy = yy < (real)0.55 ? (real)0.55 : (yy > (real)0.95 ? (real)0.95 : yy);
            rpvx = 0; rpvy = 0;
          }
#pragma unroll
          for (int c = 0; c < OPL; ++c) {
            const int o = obase + lane + 32 * c;
            sav[c] = false;
            if (o < hLo) {                                                   // hw:171-174 (o >= cLo: rescuers are not chunk objects)
              const uint64_t b = n + 2 * (uint64_t)p.Nr + 3 * (uint64_t)p.Nh + 4 * (uint64_t)(o - cLo);
              x[c] = unit_at<real>(p.seed, env_id, b);
              y[c] = unit_at<real>(p.seed, env_id, b + 1);
              vx[c] = unit_at<real>(p.seed, env_id, b + 2) * p.bad_speed;
              vy[c] = unit_at<real>(p.seed, env_id, b + 3) * p.bad_speed;
            } else if (o < Nall) {                                           // hw:162-166
              const uint64_t b = n + 2 * (uint64_t)p.Nr + 3 * (uint64_t)(o - hLo);
              x[c] = unit_at<real>(p.seed, env_id, b);
              const real yy = unit_at<real>(p.seed, env_id, b + 1);
              const real hi = (real)0.35 + unit_at<real>(p.seed, env_id, b + 2) * (real)0.01;
              y[c] = yy < (real)0 ? (real)0 : (yy > hi ? hi : yy);
              vx[c] = 0; vy[c] = 0;
            }
          }
          n += 2 * (uint64_t)p.Nr + 3 * (uint64_t)p.Nh + 4 * (uint64_t)p.Nc;
          {                                                                  // hw:177
            const real u0 = unit_at<real>(p.seed, env_id, n), u1 = unit_at<real>(p.seed, env_id, n + 1);
            bx = u0 > (real)0.25 ? (real)0.25 : u0;
            by = u1 > (real)0.25 ? (real)0.25 : u1;
            n += 2;
          }
          ctr = n;
          act.x = 0; act.y = 0;
        }
        const bool gate_pre = flags & 1;
        // ---- integrate rescuers, penalty, walls, closed gate: hw:236-261 -------------------------
        real pen;
        {
          real sq = 0;
          if (lane < p.Nr) {
            const real ax = act.x * p.action_scale, ay = act.y * p.action_scale;
            rpvx += ax; rpvy += ay;
            rpx += rpvx; rpy += rpvy;
            sq = ax * ax + ay * ay;
            real cx = clip01(rpx), cy = clip01(rpy);
            if (rpx != cx) rpvx = 0;
            if (rpy != cy) rpvy = 0;
            rpx = cx; rpy = cy;
            if (!gate_pre) {
              cx = rpx < p.gate_lo ? p.gate_lo : (rpx > (real)1 ? (real)1 : rpx);
              cy = rpy < p.gate_lo ? p.gate_lo : (rpy > (real)1 ? (real)1 : rpy);
              if (rpx != cx) rpvx = -rpvx;
              if (rpy != cy) rpvy = -rpvy;
              rpx = cx; rpy = cy;
            }
          }
          pen = p.control_penalty * (p.reward_global ? hw_warp_sum(sq) : sq);
        }
        // ---- key / bomb collisions of every rescuer up front (the obs tail needs the post-step
        //      gate flag): hw:286-296 ----------------------------------------------------------------
        unsigned coll_ke, coll_bo;
        unsigned key_near, bomb_near;
        {
          const real dkx = rpx - kx, dky = rpy - ky, dbx = rpx - bx, dby = rpy - by;
          const real dk2 = dkx * dkx + dky * dky, db2 = dbx * dbx + dby * dby;
          coll_ke = __ballot_sync(FULL_MASK, lane < p.Nr && dk2 <= p.coll2_key);
          coll_bo = __ballot_sync(FULL_MASK, lane < p.Nr && db2 <= p.coll2_bomb);
          key_near = __ballot_sync(FULL_MASK, lane < p.Nr && dk2 <= p.cull2);    // conservative range cull;
          bomb_near = __ballot_sync(FULL_MASK, lane < p.Nr && db2 <= p.cull2);   // the exact tests decide
        }
        const bool gate_post = gate_pre || (coll_ke != 0u);
        // ---- sense: one rescuer at a time -----------------------------------------------------------
        real* obs_row = obs_t;
        for (int pi = 0; pi < p.Nr; ++pi, obs_row += p.D) {
          const real mx = __shfl_sync(FULL_MASK, rpx, pi), my = __shfl_sync(FULL_MASK, rpy, pi);
          const real mvx = __shfl_sync(FULL_MASK, rpvx, pi), mvy = __shfl_sync(FULL_MASK, rpvy, pi);
          const real krx = kx - mx, kry = ky - my, kd2 = krx * krx + kry * kry;
          const real brx = bx - mx, bry = by - my, bd2 = brx * brx + bry * bry;
          real bK[KCH], bB[KCH], bC[KCH], bH[KCH];
          int iC[KCH];
#pragma unroll
          for (int kc = 0; kc < KCH; ++kc) {
            bK[kc] = bB[kc] = bC[kc] = bH[kc] = INF;
            iC[kc] = 0;
            const real sx = sx_l[kc], sy = sy_l[kc];
            if (!gate_pre && ((key_near >> pi) & 1u)) {                           // hw:343-345
              const real sv = sx * krx + sy * kry;
              const bool ok = !((sv < (real)0) | (sv > p.range) | (kd2 - sv * sv > p.r_r2));
              bK[kc] = ok ? sv : INF;
            }
            if ((bomb_near >> pi) & 1u) {
              const real sv = sx * brx + sy * bry;
              const bool ok = !((sv < (real)0) | (sv > p.range) | (bd2 - sv * sv > p.r_r2));
              bB[kc] = ok ? sv : INF;
            }
          }
          unsigned candC = 0u;   // warp-uniform: criminals within range of this rescuer
#pragma unroll
          for (int c = 0; c < OPL; ++c) {
            const real rx = x[c] - mx, ry = y[c] - my;
            const real d2 = rx * rx + ry * ry;
            // saved hostages are invisible (pre-step mask, hw:301) but still collide (hw:269-275)
            const unsigned cm = __ballot_sync(FULL_MASK, d2 <= cull2_l[c] && !sav[c]);
            candC |= cm & mC[c];
            const bool hit = d2 <= coll2_l[c];
            if (hit) col[c] |= 1u << pi;
#pragma unroll
            for (int kc = 0; kc < KCH; ++kc) {
              const real sx = sx_l[kc], sy = sy_l[kc];
              for (unsigned m = cm & mC[c]; m != 0u; m &= m - 1u) {
                const int j = __ffs(m) - 1;
                const real jx = __shfl_sync(FULL_MASK, rx, j), jy = __shfl_sync(FULL_MASK, ry, j);
                const real jd = __shfl_sync(FULL_MASK, d2, j);
                const real sv = sx * jx + sy * jy;
                const bool ok = !((sv < (real)0) | (sv > p.range) | (jd - sv * sv > p.r_r2));
                if (ok && sv < bC[kc]) { bC[kc] = sv; iC[kc] = j + 32 * c; }
              }
              if (gate_pre) {                                                      // hw:323-325
                for (unsigned m = cm & mH[c]; m != 0u; m &= m - 1u) {
                  const int j = __ffs(m) - 1;
                  const real jx = __shfl_sync(FULL_MASK, rx, j), jy = __shfl_sync(FULL_MASK, ry, j);
                  const real jd = __shfl_sync(FULL_MASK, d2, j);
                  const real sv = sx * jx + sy * jy;
                  const bool ok = !((sv < (real)0) | (sv > p.range) | (jd - sv * sv > p.r_r2));
                  if (ok && sv < bH[kc]) bH[kc] = sv;
                }
              }
            }
          }
#pragma unroll
          for (int kc = 0; kc < KCH; ++kc) {
            const real sx = sx_l[kc], sy = sy_l[kc];
            // features hw:395-397: [criminal dist, criminal speed, hostage dist, key dist, bomb dist]
            const int k = lane + 32 * kc;
            const real z = (real)0;
            real fC = z, sC = z;
            if (candC != 0u) {
              real oCx = z, oCy = z;
#pragma unroll
              for (int c = 0; c < OPL; ++c) {
                const real cx_ = __shfl_sync(FULL_MASK, vx[c], iC[kc] & 31), cy_ = __shfl_sync(FULL_MASK, vy[c], iC[kc] & 31);
                if (OPL == 1 || (iC[kc] >> 5) == c) { oCx = cx_; oCy = cy_; }
              }
              const bool hC = bC[kc] < INF;
              fC = hC ? bC[kc] : z;
              sC = hC ? sx * (oCx - mvx) + sy * (oCy - mvy) : z;
            }
            if (k < K) {
              real* o = obs_row + 32 * kc;
              store_stream(o + 0 * K, fC);
              store_stream(o + 1 * K, sC);
              store_stream(o + 2 * K, bH[kc] < INF ? bH[kc] : z);
              store_stream(o + 3 * K, bK[kc] < INF ? bK[kc] : z);
              store_stream(o + 4 * K, bB[kc] < INF ? bB[kc] : z);
            }
          }
        }
        // ---- process collisions + rewards: hw:274-284, 368-392 ---------------------------------------
        unsigned whoH = 0u, whoEnc = 0u, whoC = 0u;
        int nH = 0, nEnc = 0, nC = 0, n_unsaved = 0;
#pragma unroll
        for (int c = 0; c < OPL; ++c) {
          const int cnt = __popc(col[c]);
          const bool isH = (mH[c] >> lane) & 1u, isC = (mC[c] >> lane) & 1u;
          const bool hoc = isH && cnt >= p.n_coop_save;     // re-rescue of saved hostages included
          const bool enc = isH && cnt >= 1;
          const bool crc = isC && cnt >= 1;
          nH += __popc(__ballot_sync(FULL_MASK, hoc));
          nEnc += __popc(__ballot_sync(FULL_MASK, enc));
          const unsigned crm = __ballot_sync(FULL_MASK, crc);
          nC += __popc(crm);
          if (hoc) { whoH |= col[c]; sav[c] = true; }
          if (enc) whoEnc |= col[c];
          if (crc) whoC |= col[c];
          col[c] = 0u;
          n_unsaved += __popc(__ballot_sync(FULL_MASK, isH && !sav[c]));
          // criminals that met a rescuer respawn, ascending index, 4 draws each: hw:372-375
          if (crc) {
            const uint64_t b = ctr + 4 * (uint64_t)__popc(crm & ((1u << lane) - 1u));
            x[c] = unit_at<real>(p.seed, env_id, b);
            y[c] = unit_at<real>(p.seed, env_id, b + 1);
            vx[c] = (unit_at<real>(p.seed, env_id, b + 2) - (real)0.5) * p.bad_speed;
            vy[c] = (unit_at<real>(p.seed, env_id, b + 3) - (real)0.5) * p.bad_speed;
          }
          ctr += 4 * (uint64_t)__popc(crm);
        }
        whoH = __reduce_or_sync(FULL_MASK, whoH);
        whoEnc = __reduce_or_sync(FULL_MASK, whoEnc);
        whoC = __reduce_or_sync(FULL_MASK, whoC);
        // tail hw:406-421 of every rescuer's row: coll_ho, coll_cr, coll_key, coll_bomb, gate_open
        // (post), id; lane i writes rescuer i's.  whoEnc / whoC are exactly the any-collision masks.
        if (lane < p.Nr) {
          real* tp = obs_t + (size_t)lane * (p.D - 1) + 5 * K;   // obs_t already carries +lane
          store_stream(tp, (real)((whoEnc >> lane) & 1u));
          store_stream(tp + 1, (real)((whoC >> lane) & 1u));
          store_stream(tp + 2, (real)((coll_ke >> lane) & 1u));
          store_stream(tp + 3, (real)((coll_bo >> lane) & 1u));
          store_stream(tp + 4, gate_post ? (real)1 : (real)0);
          if (p.addid) store_stream(tp + 5, (real)(lane + 1));
        }
        if (coll_bo) flags |= 2;
        if (coll_ke) flags |= 1;
        const bool bombed = flags & 2;
        // criminals drift, bounce only if BOTH coordinates left [0,1]: hw:399-404
#pragma unroll
        for (int c = 0; c < OPL; ++c) {
          if ((mC[c] >> lane) & 1u) {
            x[c] += vx[c]; y[c] += vy[c];
            const bool ox = (x[c] < (real)0) || (x[c] > (real)1), oy = (y[c] < (real)0) || (y[c] > (real)1);
            if (ox && oy) { vx[c] = -vx[c]; vy[c] = -vy[c]; }
          }
        }
        tt += 1;
        const bool env_done = bombed || (n_unsaved == 0) || (tt >= p.timestep_limit);   // hw:181-184
        need_reset = false;
        if (!pass) {
          ts += 1;
          const bool done = env_done || (p.max_path_length > 0 && ts >= p.max_path_length);
          if (lane < p.Nr) {
            real r = pen;
            const real gate_f = gate_post ? (real)1 : (real)0, bomb_f = bombed ? (real)1 : (real)0;
            if (p.reward_global) {
              r += (((real)nEnc * p.encounter_reward * gate_f + (real)nH * p.save_reward) +
                    (real)nC * p.hit_reward) + bomb_f * p.bomb_reward;
            } else {
              if ((whoH >> lane) & 1u) r += p.save_reward;
              if ((whoEnc >> lane) & 1u) r += p.encounter_reward * gate_f;
              if ((whoC >> lane) & 1u) r += p.hit_reward;
              if ((coll_bo >> lane) & 1u) r += bomb_f * p.bomb_reward;
            }
            if (env_done) r += (real)n_unsaved * p.not_saved_reward;             // hw:425-426
            store_stream(rew_t, r);
          }
          if (lane == 0) {
            p.done[te] = done ? 1 : 0;
            reinterpret_cast<int2*>(p.info)[te] = make_int2(nH, nC);
          }
          need_reset = done && p.auto_reset;
          if (need_reset && p.term_obs != nullptr)
            keep_terminal_rows(obs_t - lane, p.term_obs + ((obs_t - lane) - p.obs), p.Nr * p.D, lane);
        }
        pass = need_reset ? 1 : 0;
      } while (need_reset);
      obs_t += p.obs_step;
      act_t += p.agent_step;
      rew_t += p.agent_step;
      te += (size_t)p.E;
    }
#pragma unroll
    for (int c = 0; c < OPL; ++c) {
      const int o = obase + lane + 32 * c;
      if (o < Nall) { rec[o] = x[c]; rec[Nall + o] = y[c]; rec[2 * Nall + o] = vx[c]; rec[3 * Nall + o] = vy[c]; }
      if (o >= hLo && o < Nall) p.saved[(size_t)e * p.Nh + (o - hLo)] = sav[c] ? 1 : 0;
    }
    if (lane < p.Nr) { rec[lane] = rpx; rec[Nall + lane] = rpy; rec[2 * Nall + lane] = rpvx; rec[3 * Nall + lane] = rpvy; }
    if (lane == 0) {
      p.fixed[4 * (size_t)e] = kx; p.fixed[4 * (size_t)e + 1] = ky;
      p.fixed[4 * (size_t)e + 2] = bx; p.fixed[4 * (size_t)e + 3] = by;
      p.flags[e] = flags; p.timestep[e] = tt; p.path_len[e] = ts; p.ctr[e] = ctr;
    }
  }
}

}  // namespace madrl

// =================================================================================================
// Host side: C ABI
// =================================================================================================
using namespace madrl;

struct madrl_hostage : EnvCore {
  madrl_hostage_config cfg;
  madrl_hostage_layout lay;
};

static int hw_validate(const madrl_hostage_config* c) {
  MADRL_REQUIRE(c != nullptr, "config is NULL");
  MADRL_REQUIRE(c->n_envs > 0, "n_envs must be > 0");
  MADRL_REQUIRE(c->n_good >= 1 && c->n_good <= 32, "n_good must be in [1,32], got %d", c->n_good);
  MADRL_REQUIRE(c->n_hostages >= 1 && c->n_bad >= 1, "n_hostages and n_bad must be >= 1");
  MADRL_REQUIRE(c->n_good + c->n_hostages + c->n_bad <= 256, "n_good + n_hostages + n_bad must be <= 256");
  MADRL_REQUIRE(c->n_sensors >= 1 && c->n_sensors <= 64, "n_sensors must be in [1,64], got %d", c->n_sensors);
  MADRL_REQUIRE(c->n_coop_save >= 1, "n_coop_save must be >= 1");
  MADRL_REQUIRE(c->timestep_limit >= 1, "timestep_limit must be >= 1");
  return MADRL_OK;
}

extern "C" int madrl_hostage_state_layout(const madrl_hostage_config* c, madrl_hostage_layout* out) {
  int rc = hw_validate(c);
  if (rc) return rc;
  MADRL_REQUIRE(out != nullptr, "layout out is NULL");
  const size_t rb = c->fp64 ? 8 : 4, E = (size_t)c->n_envs;
  const size_t nobj = (size_t)c->n_good + c->n_bad + c->n_hostages;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  out->rng_counter = take(8 * E);
  out->objs = take(rb * 4 * nobj * E);
  out->fixed = take(rb * 4 * E);
  out->saved = take((size_t)c->n_hostages * E);
  out->flags = take(4 * E);
  out->timestep = take(4 * E);
  out->path_len = take(4 * E);
  out->sensors = take(rb * 2 * (size_t)c->n_sensors);
  out->total_bytes = off;
  out->n_obj = (int32_t)nobj;
  out->obs_dim = c->n_sensors * 5 + 5 + (c->addid ? 1 : 0);   // hw:18-22
  out->real_bytes = (int32_t)rb;
  out->_pad = 0;
  return MADRL_OK;
}

extern "C" int madrl_hostage_create(const madrl_hostage_config* c, void* state_dev, madrl_hostage** out) {
  MADRL_REQUIRE(out != nullptr, "out is NULL");
  madrl_hostage_layout lay;
  int rc = madrl_hostage_state_layout(c, &lay);
  if (rc) return rc;
  madrl_hostage* h = new (std::nothrow) madrl_hostage();
  if (!h) return MADRL_ENOMEM;
  h->cfg = *c; h->lay = lay;
  rc = core_init(h, state_dev, lay.total_bytes);
  if (!rc) rc = upload_sensor_table(h->state + lay.sensors, c->n_sensors, c->fp64);
  if (rc) { madrl_hostage_destroy(h); return rc; }
  *out = h;
  return MADRL_OK;
}

extern "C" int madrl_hostage_destroy(madrl_hostage* h) {
  if (!h) return MADRL_OK;
  core_release(h);
  delete h;
  return MADRL_OK;
}

extern "C" void* madrl_hostage_state_ptr(madrl_hostage* h) { return h ? h->state : nullptr; }

extern "C" int madrl_hostage_seed(madrl_hostage* h, uint64_t seed, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  h->cfg.seed = seed;
  return core_clear_counters(h, h->lay.rng_counter, h->cfg.n_envs, stream);
}

extern "C" int madrl_hostage_set_terminal_obs(madrl_hostage* h, void* term_obs_dev) {
  return core_set_terminal_obs(h, term_obs_dev);
}

extern "C" int madrl_hostage_set_launch(madrl_hostage* h, int warps_per_block, int blocks_per_sm) {
  return core_set_launch(h, warps_per_block, blocks_per_sm);
}

template <typename real, int OPL, int KCH, int KC>
static int hw_launch_inst(madrl_hostage* h, const HWParams<real>& p, cudaStream_t stream) {
  return launch_persistent(h, hw_kernel<real, OPL, KCH, KC>, p.E, 0, stream, p);
}

template <typename real>
static int hw_launch(madrl_hostage* h, int mode, int T, const void* actions, void* obs, void* rew,
                     uint8_t* done, int32_t* info, const uint8_t* mask, int auto_reset, cudaStream_t stream) {
  const madrl_hostage_config& c = h->cfg;
  HWParams<real> p;
  p.E = c.n_envs; p.env_id_base = c.env_id_base; p.Nr = c.n_good; p.Nc = c.n_bad; p.Nh = c.n_hostages;
  p.K = c.n_sensors; p.n_coop_save = c.n_coop_save; p.D = h->lay.obs_dim; p.Nall = h->lay.n_obj;
  p.reward_global = c.reward_global; p.addid = c.addid; p.random_key = c.random_key;
  p.timestep_limit = c.timestep_limit; p.max_path_length = c.max_path_length;
  p.T = T; p.mode = mode; p.auto_reset = auto_reset;
  p.obs_step = (size_t)p.E * p.Nr * p.D; p.agent_step = (size_t)p.E * p.Nr;
  const double r = c.radius;                         // rescuers & criminals; hostages 2r (hw:111-120)
  p.r_r2 = (real)(r * r);
  p.range = (real)c.sensor_range;
  p.cull2 = (real)((c.sensor_range * c.sensor_range + r * r) * (1.0 + 1e-4) + 1e-12);
  p.coll2_c = exact_sq_threshold<real>(r + r);
  p.coll2_h = exact_sq_threshold<real>(r + r * 2);
  p.coll2_bomb = exact_sq_threshold<real>(r + c.bomb_radius);
  p.coll2_key = exact_sq_threshold<real>(r + c.key_radius);
  p.gate_lo = (real)(0.5 + r);
  p.key_x = (real)c.key_x; p.key_y = (real)c.key_y;
  p.bad_speed = (real)c.bad_speed; p.action_scale = (real)c.action_scale;
  p.save_reward = (real)c.save_reward; p.hit_reward = (real)c.hit_reward;
  p.encounter_reward = (real)c.encounter_reward; p.not_saved_reward = (real)c.not_saved_reward;
  p.bomb_reward = (real)c.bomb_reward; p.control_penalty = (real)c.control_penalty;
  p.seed = c.seed;
  char* st = h->state;
  p.objs = (real*)(st + h->lay.objs); p.fixed = (real*)(st + h->lay.fixed);
  p.saved = (uint8_t*)(st + h->lay.saved); p.flags = (int32_t*)(st + h->lay.flags);
  p.timestep = (int32_t*)(st + h->lay.timestep); p.path_len = (int32_t*)(st + h->lay.path_len);
  p.ctr = (uint64_t*)(st + h->lay.rng_counter); p.sensors = (const real*)(st + h->lay.sensors);
  p.actions = (const real*)actions; p.obs = (real*)obs; p.rew = (real*)rew;
  p.done = done; p.info = info; p.mask = mask;
  p.term_obs = (mode == 0) ? (real*)h->term_obs : nullptr;
  const int opl = (p.Nall - p.Nr + 31) / 32, kch = (p.K + 31) / 32;
#define MADRL_HW_CASE(O, KH, KC_) return hw_launch_inst<real, O, KH, KC_>(h, p, stream)
  if (p.K == 30) {
    if (opl == 1) MADRL_HW_CASE(1, 1, 30);
    if (opl == 2) MADRL_HW_CASE(2, 1, 30);
    if (opl <= 4) MADRL_HW_CASE(4, 1, 30);
    MADRL_HW_CASE(8, 1, 30);
  } else if (kch == 1) {
    if (opl == 1) MADRL_HW_CASE(1, 1, 0);
    if (opl == 2) MADRL_HW_CASE(2, 1, 0);
    if (opl <= 4) MADRL_HW_CASE(4, 1, 0);
    MADRL_HW_CASE(8, 1, 0);
  } else {
    if (opl == 1) MADRL_HW_CASE(1, 2, 0);
    if (opl == 2) MADRL_HW_CASE(2, 2, 0);
    if (opl <= 4) MADRL_HW_CASE(4, 2, 0);
    MADRL_HW_CASE(8, 2, 0);
  }
#undef MADRL_HW_CASE
}

extern "C" int madrl_hostage_reset(madrl_hostage* h, const uint8_t* mask_dev, void* obs_dev, void* stream) {
  MADRL_REQUIRE(h != nullptr && obs_dev != nullptr, "handle/obs is NULL");
  return h->cfg.fp64 ? hw_launch<double>(h, 1, 1, nullptr, obs_dev, nullptr, nullptr, nullptr, mask_dev, 0, (cudaStream_t)stream)
                     : hw_launch<float>(h, 1, 1, nullptr, obs_dev, nullptr, nullptr, nullptr, mask_dev, 0, (cudaStream_t)stream);
}

extern "C" int madrl_hostage_rollout(madrl_hostage* h, int T, const void* actions_dev, void* obs_dev, void* rew_dev,
                                     uint8_t* done_dev, int32_t* info_dev, int auto_reset, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  MADRL_REQUIRE(T >= 1, "T must be >= 1");
  MADRL_REQUIRE(actions_dev && obs_dev && rew_dev && done_dev && info_dev, "NULL trajectory buffer");
  MADRL_REQUIRE(((uintptr_t)info_dev & 7) == 0, "info_dev must be 8-byte aligned (rows are stored as one 8-byte word)");
  return h->cfg.fp64 ? hw_launch<double>(h, 0, T, actions_dev, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream)
                     : hw_launch<float>(h, 0, T, actions_dev, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream);
}

extern "C" int madrl_hostage_step(madrl_hostage* h, const void* actions_dev, void* obs_dev, void* rew_dev,
                                  uint8_t* done_dev, int32_t* info_dev, int auto_reset, void* stream) {
  return madrl_hostage_rollout(h, 1, actions_dev, obs_dev, rew_dev, done_dev, info_dev, auto_reset, stream);
}

extern "C" int madrl_hostage_reset_host(madrl_hostage* h, const uint8_t* mask_host, void* obs_host) {
  MADRL_REQUIRE(h != nullptr && obs_host != nullptr, "handle/obs is NULL");
  const size_t E = h->cfg.n_envs;
  return core_reset_host(h, E, E * h->cfg.n_good * h->lay.obs_dim * h->lay.real_bytes, mask_host, obs_host,
                         [&](uint8_t* mask_dev, char* obs_dev) { return madrl_hostage_reset(h, mask_dev, obs_dev, nullptr); });
}

extern "C" int madrl_hostage_rollout_host2(madrl_hostage* h, int T, const void* actions_host, void* obs_host,
                                           void* rew_host, uint8_t* done_host, int32_t* info_host,
                                           int auto_reset, int flags) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  const size_t E = h->cfg.n_envs, Nr = h->cfg.n_good, rb = h->lay.real_bytes;
  const StepBytes sb = {E * Nr * 2 * rb, E * Nr * h->lay.obs_dim * rb, E * Nr * rb, E, E * 2 * 4};
  return core_rollout_host(h, T, sb, actions_host, obs_host, rew_host, done_host, info_host, flags,
                           [&](int, int Tc, char* a, char* o, char* r, char* d, char* i, cudaStream_t st) {
                             return madrl_hostage_rollout(h, Tc, a, o, r, (uint8_t*)d, (int32_t*)i, auto_reset, st);
                           });
}

extern "C" int madrl_hostage_rollout_host(madrl_hostage* h, int T, const void* actions_host, void* obs_host,
                                          void* rew_host, uint8_t* done_host, int32_t* info_host,
                                          int auto_reset) {
  return madrl_hostage_rollout_host2(h, T, actions_host, obs_host, rew_host, done_host, info_host, auto_reset, 0);
}
