// PursuitEvade batched engine: persistent warp-per-env rollout kernel for sm_100a (integer path,
// bit-exact with the reference).
//
// Reference semantics: madrl_environments/pursuit/pursuit_evade.py (pe:LINE) and
// pursuit/utils/{DiscreteAgent.py (da:), AgentLayer.py (al:), agent_utils.py (au:)}.
//
// Design (see DESIGN.md):
//   * One WARP owns one env for the whole T-step rollout.  Agent coordinates live in registers
//     (lane q = pursuer q; lane j (+32c) = evader j); the env's three occupancy layers
//     (pe:244-246 model_state[0:3]) are ONE packed shared-memory word per grid cell
//     (byte0 = building, byte1 = pursuer count, byte2 = evader count), kept up to date
//     incrementally with shared-memory atomics as agents move, so a local-observation cell costs
//     a single LDS.  No block barriers: warps are independent.
//   * The reference never clears channels 1-2 of its persistent local_obs buffer (pe:119,438), so
//     out-of-bounds window cells show stale counts.  That buffer is real state: it is kept as
//     packed u16 (pursuer count | evader count << 8) per window cell in shared memory during the
//     rollout and in HBM between launches.
//   * Evader actions: live evader with live-rank r takes draw (ctr + r) of the env's Philox
//     stream (ct:16 one randint(5) per live evader, in order) -- computed by all lanes at once.
//   * The grid carries a border of off+1 marker cells (bit 31), so a window cell needs no bounds test:
//     its word address is (pursuer cell) + (a per-lane constant), and "out of bounds" is one bit of the
//     word.  Observation rows are written cell-major: lane w handles window cell w for all 3 channels,
//     three coalesced stores per 32 cells.  (Walking the cells of ALL pursuers as one flat list, 12.25
//     full rounds instead of 8 x 2 half-empty ones, was built and measured in SASS: 51 instructions per
//     round against 60 per pursuer here -- the per-pursuer form shares its shuffles and loop overhead
//     between two cells per lane.)
#include <math.h>
#include <string.h>
#include <new>

#include "common.cuh"
#include "philox.cuh"
#include "host_pipeline.cuh"

namespace madrl {

struct PEParams {
  int E, env_id_base, Np, Ne, R, off, xs, ys, n_maps, D;
  int n_catch, surround, reward_global, include_id, sample_maps, max_path_length, flatten, max_opponents;
  int T, mode, auto_reset;
  size_t obs_step, agent_step;    // element strides of one lockstep step: E*Np*D and E*Np
  int smem_per_warp, cells_pad;   // bytes of shared memory per warp; padded grid cells rounded up to 32
  int pad, ysP, ncellP;           // border width (off + 1), padded row length ys + 2 pad, padded cell count
  double constraint_window, catchr, term_pursuit, urgency;
  float wall_val, one_val;        // float32(1/layer_norm) the two ways the reference gets it
  uint64_t seed;
  const uint32_t* maps;           // [n_maps][ncellP] the empty bordered cell grid of each map, as the kernel keeps it in shared memory
  const float* lut;               // [256] float32(count)/float32(layer_norm)
  const float* idv;               // [Np]  float32(float64(i)/Np)
  // state records
  uint8_t* pos;                   // [E][2][Np+Ne]  x row, y row; pursuers then evaders
  uint64_t* gone;                 // [E] bit j = evader j removed
  int32_t* map_id;                // [E]
  int32_t* path_len;              // [E]
  uint64_t* ctr;                  // [E]
  uint16_t* stale;                // [E][Np][R*R]  pursuer count | evader count << 8
  // trajectory tensors
  const int32_t* actions;         // [T][E][Np]
  float* obs;                     // [T][E][Np][D]
  float* rew;                     // [T][E][Np]
  uint8_t* done;                  // [T][E]
  int32_t* info;                  // [T][E]  removed
  const uint8_t* mask;
  float* term_obs;                // optional [T][E][Np][D]: terminal observations of done steps
  // in-kernel action source (POLICY instantiation, madrl_pursuit_rollout_heuristic): the reference's
  // hand-written policy (heuristics/pursuit.py:18-50) closes the loop inside the launch
  const float* policy_obs0;       // [E][Np][D] the observation the FIRST action is computed from
  int32_t* actions_out;           // [T][E][Np] the actions taken (NULL = not recorded)
  int policy_c2;                  // twice the policy's window centre: R (x = R/2) or 2*(R//2) (Python 2 `/`)
  uint8_t policy_lut[128];        // window cell of the nearest visible evader -> action (host-computed, see pe_policy_table)
};

// Stream family of the policy's own draws (heuristics/pursuit.py:48,50 `action_space.sample()`): pursuer q
// deciding on an observation that was produced when the env's draw counter stood at c takes word 32 c + q.
constexpr uint32_t PE_POLICY_TAG = 2u;

// float64 `ndarray.mean()` exactly as NumPy (>= 1.22, checked against 2.3.5) computes it for a
// contiguous vector of n <= 128 elements: DOUBLE_pairwise_sum over the WHOLE vector
// (numpy/_core/src/umath/loops_utils.h.src: n < 8 -> sequential from -0.0; else 8 interleaved
// accumulators combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)), then the tail), divided by n.
__device__ __forceinline__ double numpy_mean(const double* a, int n) {
  double res;
  if (n < 8) {
    res = -0.0;
    for (int i = 0; i < n; ++i) res = __dadd_rn(res, a[i]);
  } else {
    double r[8];
    for (int j = 0; j < 8; ++j) r[j] = a[j];
    int i;
    for (i = 8; i < n - (n % 8); i += 8)
      for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], a[i + j]);
    res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                    __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < n; ++i) res = __dadd_rn(res, a[i]);
  }
  return __ddiv_rn(res, (double)n);
}

// EPL = evaders per lane (ceil(Ne/32)); CPL = window cells per lane (ceil(R*R/32));
// RC = compile-time obs_range (0 = runtime p.R).
// POLICY = the pursuers' actions come from the in-kernel heuristic policy instead of the action tensor
// (a separate instantiation: the open-loop kernel carries none of its instructions).
// FLAT = flatten=True layout (3R^2 [+1]); false = the (R, R, 4) conv layout: compile-time, so the window loop has no
// layout branch.
template <int EPL, int CPL, int RC, bool POLICY, bool FLAT>
__global__ void __launch_bounds__(32, 28) pe_kernel(const __grid_constant__ PEParams p) {
  extern __shared__ __align__(16) uint32_t smem_u32[];
  const int lane = threadIdx.x, wib = 0;
  const int warp_global = blockIdx.x;
  const int warp_stride = gridDim.x;
  const int R = RC > 0 ? RC : p.R, RR = R * R, xs = p.xs, ys = p.ys;
  const int Np = p.Np, Ne = p.Ne, Nag = Np + Ne;

  // shared memory: block-wide count->value table, then per warp: cell words, stale window counts
  for (int i = threadIdx.x; i < 256; i += blockDim.x) reinterpret_cast<float*>(smem_u32)[i] = p.lut[i];
  __syncthreads();   // the only block barrier: once, before the persistent loop
  uint32_t lut_a = smem_addr(smem_u32);
  uint32_t cell_a = lut_a + 1024u + (uint32_t)wib * (uint32_t)p.smem_per_warp;
  // keep both in registers: ptxas otherwise re-derives them from SR_CgaCtaId in front of every shared access
  asm volatile("" : "+r"(lut_a), "+r"(cell_a));
  const uint32_t stale_a = cell_a + 4u * (uint32_t)p.cells_pad;
  const uint32_t wcache_a = cell_a + (uint32_t)p.smem_per_warp - 512u;   // last 512 bytes of the warp's region
  // map cell (x, y) lives at cell0 + 4 (x ysP + y): a border of `pad` marker cells surrounds the map
  const int ysP = p.ysP;
  const uint32_t cell0 = cell_a + 4u * (uint32_t)(p.pad * ysP + p.pad);
  // border cells hold 0x80000001: bit 31 = outside the map; byte 0 = 1: nobody moves there (no bounds tests in the moves)
  const float my_idv = (lane < p.Np) ? p.idv[lane] : 0.0f;   // lane i keeps float32(i / Np)

  // per-lane window cells: local_obs[i, ch, wx, wy] <-> map cell (x - off + wx, y - off + wy) (pe:430-438), as a byte
  // offset from the pursuer's cell in the bordered grid; bit 31 = not a window cell of this lane / a cell of an even
  // window beyond 2*off, which the reference never writes
  uint32_t woff[CPL];
#pragma unroll
  for (int it = 0; it < CPL; ++it) {
    const int w = lane + 32 * it, wdx = w / R - p.off, wdy = w % R - p.off;
    const bool cell = w < RR && wdx <= p.off && wdy <= p.off;
    woff[it] = cell ? 4u * (uint32_t)((wdx + p.pad) * ysP + (wdy + p.pad)) : 0x80000000u;
  }
  const int n_tail = p.include_id ? 1 : 0;
  // POLICY: sort key of window cell w as "nearest visible evader" (heuristics/pursuit.py:28-31): squared
  // distance to the window centre in doubled coordinates (sqrt is monotonic and these small integers have
  // distinct roots), then the row-major cell index -- np.nonzero order, np.argmin keeps the first minimum
  uint32_t pkey[CPL];
#pragma unroll
  for (int it = 0; it < CPL; ++it) {
    const int w = lane + 32 * it;
    const int ddx = 2 * (w / R) - p.policy_c2, ddy = 2 * (w % R) - p.policy_c2;
    pkey[it] = ((uint32_t)(ddx * ddx + ddy * ddy) << 8) | (uint32_t)w;
  }

  for (int e = warp_global; e < p.E; e += warp_stride) {
    if (p.mode == 1 && p.mask != nullptr && p.mask[e] == 0) continue;
    const uint32_t env_id = (uint32_t)(p.env_id_base + e);
    // ---- state -> registers / shared memory --------------------------------------------------
    const uint8_t* prec = p.pos + (size_t)e * 2 * Nag;
    int px = 0, py = 0, ex[EPL], ey[EPL];
    if (lane < Np) { px = prec[lane]; py = prec[Nag + lane]; }
    unsigned live[EPL];   // warp-uniform: evaders of chunk c still on the map
    const uint64_t gone0 = p.gone[e];
#pragma unroll
    for (int c = 0; c < EPL; ++c) {
      const int j = lane + 32 * c;
      ex[c] = ey[c] = 0;
      if (j < Ne) { ex[c] = prec[Np + j]; ey[c] = prec[Nag + Np + j]; }
      const unsigned valid = __ballot_sync(FULL_MASK, j < Ne);
      live[c] = valid & ~(unsigned)(gone0 >> (32 * c));
    }
    int map_id = p.map_id[e], ts = p.path_len[e];
    uint64_t ctr = p.ctr[e];
    const uint32_t* map = p.maps + (size_t)map_id * p.ncellP + (p.pad * ysP + p.pad);   // cell (x, y) at map[x ysP + y]
    for (int i = lane; i < Np * RR; i += 32) sts_u16(stale_a + 2u * i, p.stale[(size_t)e * Np * RR + i]);
    bool rebuild = true;   // cell words must be (re)built from map + positions
    int coff = -1;   // word offset of draw `ctr` inside the warp's cache of 32 Philox blocks (warp-uniform); < 0 = cache empty

    float* obs_t = p.obs + (size_t)e * Np * p.D;
    float* rew_t = p.rew + (size_t)e * Np + lane;
    const int32_t* act_t = p.actions + (size_t)e * Np + lane;
    size_t te = (size_t)e;
    int pass = (p.mode == 1) ? 1 : 0;   // pass 1 = reset(): draws + obs only
    // POLICY: pursuer `lane`'s action for the NEXT step, first from the caller's observation
    int next_act = 4;
    if constexpr (POLICY) {
      const float* o0 = p.policy_obs0 + (size_t)e * Np * p.D;
      for (int i = 0; i < Np; ++i, o0 += p.D) {
        uint32_t key = 0xffffffffu;
#pragma unroll
        for (int it = 0; it < CPL; ++it) {
          const int w = lane + 32 * it;
          if (w < RR && (FLAT ? o0[2 * RR + w] : o0[4 * w + 2]) > 0.0f) key = min(key, pkey[it]);
        }
        key = __reduce_min_sync(FULL_MASK, key);
        if (lane == i)
          next_act = key != 0xffffffffu ? (int)p.policy_lut[key & 0xffu]
                                        : u32_to_range(stream_word(p.seed, env_id, PE_POLICY_TAG, ctr * 32u + (uint64_t)i), 0, 5);
      }
    }
    int act_nx = 4;
    if (!POLICY && p.mode == 0 && lane < Np) act_nx = *act_t;
    for (int t = 0; t < p.T; ++t) {
      int act = 4;
      if constexpr (POLICY) {
        if (lane < Np) {
          act = next_act;
          if (p.actions_out != nullptr) p.actions_out[(size_t)t * p.agent_step + (size_t)e * Np + lane] = act;
        }
      } else if (p.mode == 0 && lane < Np) {
        // double-buffered in registers: the load for step t+1 is issued at the top of step t, so its HBM
        // latency hides behind a whole step (prefetch.global.L1 did not: the first use of the action was 10 % of
        // all stall samples of the C2 kernel; C2 66 -> 74.5 % of the roofline, profiles/r2_ab_action_db.log)
        act = act_nx;
        if (t + 1 < p.T) act_nx = act_t[p.agent_step];
      }
      bool need_reset;
      do {
        int removed = 0;
        unsigned sur_mask = 0u;      // pursuers that surrounded / tagged a removed evader
        unsigned caught[EPL];
        int rcount = 0;              // this pursuer's neighbouring-evader count (pe:374-380)
#pragma unroll
        for (int c = 0; c < EPL; ++c) caught[c] = 0u;
        if (pass) {
          // ---- reset(): pe:173-203.  All lanes run the same stream (warp-uniform). ------------
          SeqStream rs;
          rs.init(p.seed, env_id, 0u, ctr);
          // pe:177-181 random_opponents: this episode has randint(1, max_opponents) evaders; the others
          // never exist (not spawned, no draws, not live)
          const int n_ev = p.max_opponents > 0 ? rs.next_range(1, p.max_opponents) : Ne;
          if (p.sample_maps) map_id = rs.next_range(0, p.n_maps);                    // pe:183
          map = p.maps + (size_t)map_id * p.ncellP + (p.pad * ysP + p.pad);
          const double span = 1.0 - p.constraint_window;
          const double xws = 0.0 + (span - 0.0) * rs.next_unit<double>();             // pe:185
          const double yws = 0.0 + (span - 0.0) * rs.next_unit<double>();             // pe:186
          const int xl = (int)((double)xs * xws), xu = (int)((double)xs * (xws + p.constraint_window));
          const int yl = (int)((double)ys * yws), yu = (int)((double)ys * (yws + p.constraint_window));
          for (int a = 0; a < Np + n_ev; ++a) {                                       // au:31-47
            int x, y;
            do {
              x = rs.next_range(xl, xu);
              y = rs.next_range(yl, yu);
            } while ((map[x * ysP + y] & 1u) != 0u);
            if (a < Np) { if (lane == a) { px = x; py = y; } }
            else {
              const int j = a - Np;
#pragma unroll
              for (int c = 0; c < EPL; ++c) if (j == lane + 32 * c) { ex[c] = x; ey[c] = y; }
            }
          }
          ctr = rs.counter;
          coff = -1;   // the reset consumed draws: the cached words no longer start at `ctr`
          ts = 0;
#pragma unroll
          for (int c = 0; c < EPL; ++c) live[c] = __ballot_sync(FULL_MASK, lane + 32 * c < n_ev);
          rebuild = true;
        }
        if (rebuild) {   // cell words from scratch: building flag + occupancy counts
          __syncwarp();
          // the empty grid of this map (building flags, need_to_surround bits, border markers) is a table the host
          // laid out exactly like the shared-memory grid: the rebuild is a straight copy
          {
            const uint32_t* grid = map - (p.pad * ysP + p.pad);
            for (int i = lane; i < p.ncellP; i += 32) sts_u32(cell_a + 4u * i, __ldg(grid + i));
          }
          __syncwarp();
          if (lane < Np) reds_add_u32(cell0 + 4u * (px * ysP + py), 1u << 8);
#pragma unroll
          for (int c = 0; c < EPL; ++c)
            if ((live[c] >> lane) & 1u) reds_add_u32(cell0 + 4u * (ex[c] * ysP + ey[c]), 1u << 16);
          __syncwarp();
          rebuild = false;
        }
        if (!pass) {
          // ---- reward from the PRE-move state: pe:213, 359-381 ---------------------------------
          if (lane < Np) {
            const int xm = max(px - 1, 0), xp = min(px + 1, xs - 1);
            const int ym = max(py - 1, 0), yp = min(py + 1, ys - 1);
            rcount = (int)((lds_u32(cell0 + 4u * (xm * ysP + py)) >> 16) & 0xff) +
                     (int)((lds_u32(cell0 + 4u * (xp * ysP + py)) >> 16) & 0xff) +
                     (int)((lds_u32(cell0 + 4u * (px * ysP + yp)) >> 16) & 0xff) +
                     (int)((lds_u32(cell0 + 4u * (px * ysP + ym)) >> 16) & 0xff);
          }
          __syncwarp();
          // ---- move pursuers: pe:227-235, da:69-97 ---------------------------------------------
          if (lane < Np) {
            const int a = act;
            const int dx = (a == 0) ? -1 : (a == 1 ? 1 : 0), dy = (a == 2) ? 1 : (a == 3 ? -1 : 0);
            const int nx = px + dx, ny = py + dy;
            const uint32_t cur = cell0 + 4u * (px * ysP + py), nxt = cell0 + 4u * (nx * ysP + ny);
            // da:69-97: no move out of bounds or into a building -- both are "byte 0 set" in the bordered grid
            if ((unsigned)a < 4u && lds_low_byte(cur) == 0u && lds_low_byte(nxt) == 0u) {
              reds_add_u32(cur, 0u - (1u << 8));
              reds_add_u32(nxt, 1u << 8);
              px = nx; py = ny;
            }
          }
          // ---- move live evaders, one stream draw each in index order: pe:238-241, ct:16 -------
          int base_rank = 0;
          {
            int n_draws = 0;
#pragma unroll
            for (int c = 0; c < EPL; ++c) n_draws += __popc(live[c]);
            // words [ctr, ctr + n_draws) must lie in the 128 cached words
            if (coff < 0 || coff + n_draws > 128) {
              __syncwarp();   // every lane's reads of the previous fill precede the overwrite
              coff = (int)(ctr & 3u);
              const uint64_t b = (ctr >> 2) + (uint64_t)lane;
              const Philox4 blk = philox4x32_10((uint32_t)b, (uint32_t)(b >> 32), env_id, 0u, (uint32_t)p.seed,
                                                (uint32_t)(p.seed >> 32));
#pragma unroll
              for (int k = 0; k < 4; ++k) sts_u32(wcache_a + 16u * (uint32_t)lane + 4u * k, blk.w[k]);
              __syncwarp();
            }
          }
#pragma unroll
          for (int c = 0; c < EPL; ++c) {
            const bool alive = (live[c] >> lane) & 1u;
            const int rank = base_rank + __popc(live[c] & lanemask_lt());
            if (alive) {
              const uint32_t word = lds_u32(wcache_a + 4u * (uint32_t)(coff + rank));
              const int a = u32_to_range(word, 0, 5);
              const int dx = (a == 0) ? -1 : (a == 1 ? 1 : 0), dy = (a == 2) ? 1 : (a == 3 ? -1 : 0);
              const int nx = ex[c] + dx, ny = ey[c] + dy;
              const uint32_t cur = cell0 + 4u * (ex[c] * ysP + ey[c]), nxt = cell0 + 4u * (nx * ysP + ny);
              if (a < 4 && lds_low_byte(cur) == 0u && lds_low_byte(nxt) == 0u) {
                reds_add_u32(cur, 0u - (1u << 16));
                reds_add_u32(nxt, 1u << 16);
                ex[c] = nx; ey[c] = ny;
              }
            }
            base_rank += __popc(live[c]);
          }
          ctr += (uint64_t)base_rank;
          coff += base_rank;
          __syncwarp();
          // ---- remove_agents: pe:463-521 -----------------------------------------------------------
#pragma unroll
          for (int c = 0; c < EPL; ++c) {
            bool got = false;
            if ((live[c] >> lane) & 1u) {
              const int x = ex[c], y = ey[c];
              if (p.surround) {
                // neighbours holding >= 1 pursuer (pe:482-485) vs need_to_surround (pe:523-540).  need_to_surround
                // depends on the map only (borders, buildings next to the cell, the row/column-0 quirk of pe:536): the
                // host tabulates it per cell (pe_need_to_surround) and the rebuild keeps it in bits 24-26 of the cell
                // word; border cells hold no pursuers, so the four neighbour loads need no bounds tests
                const uint32_t own = cell0 + 4u * (uint32_t)(x * ysP + y);
                const int need = (int)((lds_u32(own) >> 24) & 7u);
                const int adj = (int)(((lds_u32(own - 4u * (uint32_t)ysP) >> 8) & 0xffu) != 0u) +
                                (int)(((lds_u32(own + 4u * (uint32_t)ysP) >> 8) & 0xffu) != 0u) +
                                (int)(((lds_u32(own + 4u) >> 8) & 0xffu) != 0u) +
                                (int)(((lds_u32(own - 4u) >> 8) & 0xffu) != 0u);
                got = (adj == need);
              } else {
                got = (int)((lds_u32(cell0 + 4u * (x * ysP + y)) >> 8) & 0xff) >= p.n_catch;   // pe:498
              }
            }
            caught[c] = __ballot_sync(FULL_MASK, got);
            removed += __popc(caught[c]);
            // which pursuers take the credit (pe:489-495 / pe:503-506): rare, warp-uniform loop
            for (unsigned m = caught[c]; m != 0u; m &= m - 1u) {
              const int j = __ffs(m) - 1;
              const int cx = __shfl_sync(FULL_MASK, ex[c], j), cy = __shfl_sync(FULL_MASK, ey[c], j);
              const int ddx = px - cx, ddy = py - cy;
              const bool credit = p.surround ? (abs(ddx) + abs(ddy) == 1) : (ddx == 0 && ddy == 0);
              sur_mask |= __ballot_sync(FULL_MASK, lane < Np && credit);
            }
          }
        }
        // ---- collect_obs: pe:418-461 (flatten): channel-major, then x, then y, then id ----------
        {
          float* row = obs_t;
          uint32_t st_row = stale_a + 2u * lane;
          for (int i = 0; i < Np; ++i, row += p.D, st_row += 2u * RR) {
            const int pxi = __shfl_sync(FULL_MASK, px, i), pyi = __shfl_sync(FULL_MASK, py, i);
            const uint32_t pcell = cell_a + 4u * (uint32_t)(pxi * ysP + pyi);   // + woff: this lane's window cells
            // explicit software pipeline over the (unrolled) window chunks: all shared loads
            // first, then the dependent table lookups, then the coalesced stores
            uint32_t wv[CPL], c12[CPL];
            bool inb[CPL];
#pragma unroll
            for (int it = 0; it < CPL; ++it) {
              // the border marker (bit 31 of the word) replaces the four bounds tests; lanes past the window and
              // the never-written cells of an even window carry the same bit in their constant
              wv[it] = lds_u32(pcell + (woff[it] & 0x7fffffffu));
              inb[it] = ((wv[it] | woff[it]) >> 31) == 0u;
              c12[it] = (lane + 32 * it < RR) ? lds_u16(st_row + 64u * it) : 0u;   // stale pursuer | evader << 8
            }
            float v1[CPL], v2[CPL];
#pragma unroll
            for (int it = 0; it < CPL; ++it) {
              if (inb[it]) c12[it] = __byte_perm(wv[it], 0u, 0x4421u);   // (wv >> 8) & 0xffff: pursuer | evader << 8
              if (lane + 32 * it < RR) sts_u16(st_row + 64u * it, c12[it]);
              // byte extraction as PRMT so that the table address is one LEA (was shift + mask + add per lookup)
              v1[it] = lds_f32(lut_a + 4u * __byte_perm(c12[it], 0u, 0x4440u));   // float32(k) / float32(layer_norm)
              v2[it] = lds_f32(lut_a + 4u * __byte_perm(c12[it], 0u, 0x4441u));
            }
            if constexpr (POLICY) {   // heuristics/pursuit.py:18-50 on the evader channel just assembled
              uint32_t key = 0xffffffffu;
#pragma unroll
              for (int it = 0; it < CPL; ++it)
                if (lane + 32 * it < RR && (c12[it] >> 8) != 0u) key = min(key, pkey[it]);
              key = __reduce_min_sync(FULL_MASK, key);
              if (lane == i)
                next_act = key != 0xffffffffu ? (int)p.policy_lut[key & 0xffu]
                                              : u32_to_range(stream_word(p.seed, env_id, PE_POLICY_TAG, ctr * 32u + (uint64_t)i), 0, 5);
            }
            if constexpr (FLAT) {
#pragma unroll
              for (int it = 0; it < CPL; ++it) {
                const int w = lane + 32 * it;
                if (w < RR) {
                  const float v0 = inb[it] ? ((wv[it] & 0xff) ? p.one_val : 0.0f) : p.wall_val;   // pe:433,438
                  store_stream(row + w, v0);
                  store_stream(row + RR + w, v1[it]);
                  store_stream(row + 2 * RR + w, v2[it]);
                }
              }
            } else {
              // flatten=False: np.rollaxis(local_obs[i], 0, 3) -> [x][y][channel], channel 3 holds
              // i/Np at the window centre and zeros elsewhere (pe:440-449): one 16-byte store per cell
              const float idval = __shfl_sync(FULL_MASK, my_idv, i);
              const int centre = (R / 2) * R + (R / 2);
#pragma unroll
              for (int it = 0; it < CPL; ++it) {
                const int w = lane + 32 * it;
                if (w < RR) {
                  const float v0 = inb[it] ? ((wv[it] & 0xff) ? p.one_val : 0.0f) : p.wall_val;
                  __stcs(reinterpret_cast<float4*>(row) + w, make_float4(v0, v1[it], v2[it], w == centre ? idval : 0.0f));
                }
              }
            }
          }
          if (FLAT && n_tail && lane < Np) store_stream(obs_t + (size_t)lane * p.D + 3 * RR, my_idv);   // pe:444-445
        }
        need_reset = false;
        if (!pass) {
          // ---- rewards (float64 like the reference, narrowed once): pe:254-262 ------------------
          double r = 0.0;
          if (lane < Np) {
            // explicit round-to-nearest ops: no FMA contraction, so every intermediate rounds
            // exactly like NumPy's float64 arithmetic
            r = __dmul_rn(p.catchr, (double)rcount);
            r = __dadd_rn(r, __dmul_rn(p.term_pursuit, ((sur_mask >> lane) & 1u) ? 1.0 : 0.0));
            r = __dadd_rn(r, p.urgency);
          }
          if (p.reward_global) {
            double all[32];
            for (int q = 0; q < Np; ++q) all[q] = __shfl_sync(FULL_MASK, r, q);
            r = numpy_mean(all, Np);
          }
          if (lane < Np) store_stream(rew_t, (float)r);
          // ---- the captured evaders leave the map only now (still visible in this obs) -----------
          __syncwarp();   // every lane's window reads of the cell words precede the decrements below
          int n_live = 0;
#pragma unroll
          for (int c = 0; c < EPL; ++c) {
            if ((caught[c] >> lane) & 1u) reds_add_u32(cell0 + 4u * (ex[c] * ysP + ey[c]), 0u - (1u << 16));
            live[c] &= ~caught[c];
            n_live += __popc(live[c]);
          }
          __syncwarp();
          ts += 1;
          const bool done = (n_live == 0) || (p.max_path_length > 0 && ts >= p.max_path_length);  // pe:384-389
          if (lane == 0) {
            p.done[te] = done ? 1 : 0;
            p.info[te] = removed;
          }
          need_reset = done && p.auto_reset;   // VecEnvExecutor.step (vec_env_executor.py:24-27)
          if (need_reset && p.term_obs != nullptr)
            keep_terminal_rows(obs_t, p.term_obs + (obs_t - p.obs), Np * p.D, lane);
        }
        pass = need_reset ? 1 : 0;
      } while (need_reset);
      obs_t += p.obs_step;
      rew_t += p.agent_step;
      act_t += p.agent_step;
      te += (size_t)p.E;
    }
    // ---- registers / shared memory -> state records ---------------------------------------------
    __syncwarp();
    uint8_t* wrec = p.pos + (size_t)e * 2 * Nag;
    if (lane < Np) { wrec[lane] = (uint8_t)px; wrec[Nag + lane] = (uint8_t)py; }
    uint64_t gone = 0;
#pragma unroll
    for (int c = 0; c < EPL; ++c) {
      const int j = lane + 32 * c;
      if (j < Ne) { wrec[Np + j] = (uint8_t)ex[c]; wrec[Nag + Np + j] = (uint8_t)ey[c]; }
      const unsigned valid = __ballot_sync(FULL_MASK, j < Ne);
      gone |= (uint64_t)(valid & ~live[c]) << (32 * c);
    }
    for (int i = lane; i < Np * RR; i += 32) p.stale[(size_t)e * Np * RR + i] = (uint16_t)lds_u16(stale_a + 2u * i);
    if (lane == 0) { p.gone[e] = gone; p.map_id[e] = map_id; p.path_len[e] = ts; p.ctr[e] = ctr; }
    __syncwarp();
  }
}

}  // namespace madrl

// =================================================================================================
// Host side: C ABI
// =================================================================================================
using namespace madrl;

struct madrl_pursuit : EnvCore {
  madrl_pursuit_config cfg;
  madrl_pursuit_layout lay;
};

static int pe_validate(const madrl_pursuit_config* c) {
  MADRL_REQUIRE(c != nullptr, "config is NULL");
  MADRL_REQUIRE(c->n_envs > 0, "n_envs must be > 0");
  MADRL_REQUIRE(c->n_pursuers >= 1 && c->n_pursuers <= 32, "n_pursuers must be in [1,32], got %d", c->n_pursuers);
  MADRL_REQUIRE(c->n_evaders >= 1 && c->n_evaders <= 64, "n_evaders must be in [1,64], got %d", c->n_evaders);
  MADRL_REQUIRE(c->xs >= 2 && c->ys >= 2 && c->xs <= 255 && c->ys <= 255 && c->xs * c->ys <= 4096,
                "map must be between 2x2 and 4096 cells (<= 255 per side)");
  MADRL_REQUIRE(c->n_maps >= 1, "n_maps must be >= 1");
  MADRL_REQUIRE(c->obs_range >= 1 && c->obs_range * c->obs_range <= 128, "obs_range must be in [1,11]");
  MADRL_REQUIRE(c->layer_norm != 0.0, "layer_norm must be non-zero");
  MADRL_REQUIRE(c->constraint_window > 0.0 && c->constraint_window <= 1.0, "constraint_window must be in (0,1]");
  // random_opponents: randint(1, max_opponents) evaders per episode; the reference indexes its
  // evaders_gone array (sized n_evaders at construction) with them (pursuit_evade.py:138,477-487)
  MADRL_REQUIRE(c->max_opponents == 0 || (c->max_opponents >= 2 && c->max_opponents - 1 <= c->n_evaders),
                "max_opponents must be 0 (off) or in [2, n_evaders + 1], got %d", c->max_opponents);
  return MADRL_OK;
}

extern "C" int madrl_pursuit_state_layout(const madrl_pursuit_config* c, madrl_pursuit_layout* out) {
  int rc = pe_validate(c);
  if (rc) return rc;
  MADRL_REQUIRE(out != nullptr, "layout out is NULL");
  const size_t E = (size_t)c->n_envs, Nag = (size_t)c->n_pursuers + c->n_evaders;
  const size_t RR = (size_t)c->obs_range * c->obs_range;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  out->rng_counter = take(8 * E);
  out->gone = take(8 * E);
  out->pos = take(2 * Nag * E);
  out->map_id = take(4 * E);
  out->path_len = take(4 * E);
  out->stale = take(2 * (size_t)c->n_pursuers * RR * E);
  {
    const size_t pad = (size_t)(c->obs_range - 1) / 2 + 1;
    out->maps = take(4 * (size_t)c->n_maps * (c->xs + 2 * pad) * (c->ys + 2 * pad));
  }
  out->lut = take(4 * 256);
  out->idv = take(4 * 32);

  out->total_bytes = off;
  out->n_agents = (int32_t)Nag;
  out->obs_dim = c->flatten ? (int32_t)(3 * RR + (c->include_id ? 1 : 0))   // pe:108-112
                            : (int32_t)(4 * RR);                            // (R, R, 4), pe:440-449
  return MADRL_OK;
}

extern "C" int madrl_pursuit_create(const madrl_pursuit_config* c, const int32_t* map_pool_host,
                                    void* state_dev, madrl_pursuit** out) {
  MADRL_REQUIRE(out != nullptr && map_pool_host != nullptr, "out / map_pool is NULL");
  madrl_pursuit_layout lay;
  int rc = madrl_pursuit_state_layout(c, &lay);
  if (rc) return rc;
  madrl_pursuit* h = new (std::nothrow) madrl_pursuit();
  if (!h) return MADRL_ENOMEM;
  h->cfg = *c; h->lay = lay;
  rc = core_init(h, state_dev, lay.total_bytes);   // zeroed: agents start at (0,0), local_obs zeroed (pe:119, au:22)
  if (rc) { madrl_pursuit_destroy(h); return rc; }
  // constant table: per map the EMPTY bordered cell grid exactly as the kernel keeps it in shared memory (a rebuild
  // is a straight copy).  Word of map cell (x, y) at [(x + pad) ysP + (y + pad)]:
  //   bit 0      building (da:110-113)
  //   bits 24-26 need_to_surround of the cell (pe:523-540), static per map:
  //              4 - [x on an x-border] - [y on a y-border] - #{in-bounds neighbours with xn > 0 and yn > 0 that are
  //              buildings} (pe:536 skips neighbours with xn <= 0 or yn <= 0: a building in row / column 0 never subtracts)
  //   border cells (a frame of `pad` cells): 0x80000001 = outside the map + nobody moves there
  const size_t ncell = (size_t)c->xs * c->ys, nm = (size_t)c->n_maps;
  const int pad = (c->obs_range - 1) / 2 + 1, ysP = c->ys + 2 * pad, xsP = c->xs + 2 * pad;
  const size_t ncellP = (size_t)xsP * ysP;
  uint32_t* m8 = new (std::nothrow) uint32_t[nm * ncellP];
  if (!m8) { madrl_pursuit_destroy(h); return MADRL_ENOMEM; }
  for (size_t mi = 0; mi < nm; ++mi) {
    const int32_t* mp = map_pool_host + mi * ncell;
    uint32_t* g = m8 + mi * ncellP;
    for (size_t i = 0; i < ncellP; ++i) g[i] = 0x80000001u;
    for (int x = 0; x < c->xs; ++x)
      for (int y = 0; y < c->ys; ++y) {
        int need = 4;
        if (x == 0 || x == c->xs - 1) need -= 1;
        if (y == 0 || y == c->ys - 1) need -= 1;
        const int dxs[4] = {-1, 1, 0, 0}, dys[4] = {0, 0, 1, -1};                       // pe:150 surround_mask
        for (int m = 0; m < 4; ++m) {
          const int xn = x + dxs[m], yn = y + dys[m];
          if (xn > 0 && yn > 0 && xn < c->xs && yn < c->ys && mp[xn * c->ys + yn] == -1) need -= 1;
        }
        g[(size_t)(x + pad) * ysP + (y + pad)] = (mp[x * c->ys + y] == -1 ? 1u : 0u) | ((uint32_t)(need < 0 ? 0 : need) << 24);
      }
  }
  float lut[256], idv[32];
  const float lnf = (float)c->layer_norm;
  for (int k = 0; k < 256; ++k) lut[k] = (float)k / lnf;            // float32 |count| / layer_norm (pe:438)
  for (int i = 0; i < 32; ++i) idv[i] = (float)((double)i / (double)c->n_pursuers);   // pe:445
  cudaError_t e = cudaMemcpy(h->state + lay.maps, m8, 4 * nm * ncellP, cudaMemcpyHostToDevice);
  delete[] m8;
  if (e == cudaSuccess) e = cudaMemcpy(h->state + lay.lut, lut, sizeof(lut), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(h->state + lay.idv, idv, sizeof(idv), cudaMemcpyHostToDevice);

  if (e != cudaSuccess) { set_error("cudaMemcpy(tables): %s", cudaGetErrorString(e)); madrl_pursuit_destroy(h); return MADRL_ECUDA; }
  *out = h;
  return MADRL_OK;
}

extern "C" int madrl_pursuit_destroy(madrl_pursuit* h) {
  if (!h) return MADRL_OK;
  core_release(h);
  delete h;
  return MADRL_OK;
}

extern "C" void* madrl_pursuit_state_ptr(madrl_pursuit* h) { return h ? h->state : nullptr; }

extern "C" int madrl_pursuit_seed(madrl_pursuit* h, uint64_t seed, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  h->cfg.seed = seed;
  return core_clear_counters(h, h->lay.rng_counter, h->cfg.n_envs, stream);
}

extern "C" int madrl_pursuit_set_terminal_obs(madrl_pursuit* h, void* term_obs_dev) {
  return core_set_terminal_obs(h, term_obs_dev);
}

extern "C" int madrl_pursuit_set_launch(madrl_pursuit* h, int warps_per_block, int blocks_per_sm) {
  return core_set_launch(h, warps_per_block, blocks_per_sm);
}

extern "C" int madrl_pursuit_set_params(madrl_pursuit* h, double catchr, double constraint_window) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  MADRL_REQUIRE(constraint_window > 0.0 && constraint_window <= 1.0, "constraint_window must be in (0,1]");
  h->cfg.catchr = catchr; h->cfg.constraint_window = constraint_window;
  return MADRL_OK;
}

// heuristics/pursuit.py:23-48 for every window cell the nearest visible evader can occupy: the action a
// pursuer at the window centre (x, y) = (c2/2, c2/2) takes towards cell (xc, yc).  Same double arithmetic as
// the reference (libm atan2, Python's float `%`), evaluated once on the host.
void pe_policy_table(int R, int c2, uint8_t* lut) {
  const double pi = 3.141592653589793;   // np.pi
  const double x = 0.5 * (double)c2, y = 0.5 * (double)c2;
  for (int w = 0; w < R * R && w < 128; ++w) {
    const double xc = (double)(w / R), yc = (double)(w % R);
    int a;
    if (xc == x && yc == y) a = 4;                                     // STAY  :33-34
    else {
      double ang = atan2(yc - y, xc - x);                              // :35
      double m = fmod(ang + pi, 2 * pi);                               // :36  Python `%`: sign of the divisor
      if (m < 0) m += 2 * pi;
      ang = m - pi;
      if (-pi / 4 <= ang && ang < pi / 4) a = 1;                       // RIGHT :38
      else if (pi / 4 <= ang && ang < 3 / 4. * pi) a = 2;              // UP    :41
      else if (ang >= 3 / 4. * pi || ang < -3 / 4. * pi) a = 0;        // LEFT  :44
      else a = 3;                                                      // DOWN  :47 (the final `else` is unreachable)
    }
    lut[w] = (uint8_t)a;
  }
}

template <int EPL, int CPL, int RC, bool POLICY, bool FLAT>
static int pe_launch_inst3(madrl_pursuit* h, PEParams& p, cudaStream_t stream) {
  const size_t smem = 1024 + (size_t)p.smem_per_warp;   // block LUT + per-warp regions
  MADRL_REQUIRE(smem <= 200 * 1024, "map too large for shared memory (%zu B per block)", smem);
  return launch_persistent(h, pe_kernel<EPL, CPL, RC, POLICY, FLAT>, p.E, smem, stream, p);
}

template <int EPL, int CPL, int RC, bool POLICY>
static int pe_launch_inst2(madrl_pursuit* h, PEParams& p, cudaStream_t stream) {
  return p.flatten ? pe_launch_inst3<EPL, CPL, RC, POLICY, true>(h, p, stream)
                   : pe_launch_inst3<EPL, CPL, RC, POLICY, false>(h, p, stream);
}

template <int EPL, int CPL, int RC>
static int pe_launch_inst(madrl_pursuit* h, PEParams& p, cudaStream_t stream) {
  return p.policy_obs0 != nullptr ? pe_launch_inst2<EPL, CPL, RC, true>(h, p, stream)
                                  : pe_launch_inst2<EPL, CPL, RC, false>(h, p, stream);
}

static int pe_launch(madrl_pursuit* h, int mode, int T, const int32_t* actions, float* obs, float* rew,
                     uint8_t* done, int32_t* info, const uint8_t* mask, int auto_reset, cudaStream_t stream,
                     const float* policy_obs0 = nullptr, int32_t* actions_out = nullptr, int policy_c2 = 0) {
  const madrl_pursuit_config& c = h->cfg;
  PEParams p;
  p.policy_obs0 = policy_obs0; p.actions_out = actions_out; p.policy_c2 = policy_c2;
  memset(p.policy_lut, 4, sizeof(p.policy_lut));
  if (policy_obs0 != nullptr) pe_policy_table(c.obs_range, policy_c2, p.policy_lut);
  p.E = c.n_envs; p.env_id_base = c.env_id_base; p.Np = c.n_pursuers; p.Ne = c.n_evaders;
  p.R = c.obs_range; p.off = (int)((c.obs_range - 1) / 2);   // pe:65
  p.xs = c.xs; p.ys = c.ys; p.n_maps = c.n_maps; p.D = h->lay.obs_dim;
  p.n_catch = c.n_catch; p.surround = c.surround; p.reward_global = c.reward_global;
  p.include_id = c.include_id; p.sample_maps = c.sample_maps; p.max_path_length = c.max_path_length;
  p.max_opponents = c.max_opponents;
  p.flatten = c.flatten;
  p.T = T; p.mode = mode; p.auto_reset = auto_reset;
  p.obs_step = (size_t)p.E * p.Np * p.D; p.agent_step = (size_t)p.E * p.Np;
  const int RR = c.obs_range * c.obs_range;
  p.pad = p.off + 1; p.ysP = c.ys + 2 * p.pad; p.ncellP = (c.xs + 2 * p.pad) * p.ysP;
  p.cells_pad = (p.ncellP + 31) / 32 * 32;
  p.smem_per_warp = (int)align_up((size_t)p.cells_pad * 4 + (size_t)c.n_pursuers * RR * 2, 16) +
                    512;   // + the warp's Philox word cache
  p.constraint_window = c.constraint_window; p.catchr = c.catchr; p.term_pursuit = c.term_pursuit;
  p.urgency = c.urgency_reward;
  p.wall_val = (float)(1.0 / c.layer_norm);           // local_obs[i][0].fill(1.0 / layer_norm): f64 -> f32
  p.one_val = 1.0f / (float)c.layer_norm;             // float32 |+-1| / layer_norm
  p.seed = c.seed;
  char* st = h->state;
  p.maps = (const uint32_t*)(st + h->lay.maps); p.lut = (const float*)(st + h->lay.lut);
  p.idv = (const float*)(st + h->lay.idv);
  p.pos = (uint8_t*)(st + h->lay.pos); p.gone = (uint64_t*)(st + h->lay.gone);
  p.map_id = (int32_t*)(st + h->lay.map_id); p.path_len = (int32_t*)(st + h->lay.path_len);
  p.ctr = (uint64_t*)(st + h->lay.rng_counter); p.stale = (uint16_t*)(st + h->lay.stale);
  p.actions = actions; p.obs = obs; p.rew = rew; p.done = done; p.info = info; p.mask = mask;
  p.term_obs = (mode == 0) ? (float*)h->term_obs : nullptr;
  const int epl = (p.Ne + 31) / 32, cpl = (RR + 31) / 32;
#define MADRL_PE_CASE(EP, CP, RC_) return pe_launch_inst<EP, CP, RC_>(h, p, stream)
  if (p.R == 7) { if (epl == 1) MADRL_PE_CASE(1, 2, 7); MADRL_PE_CASE(2, 2, 7); }
  if (cpl == 1) { if (epl == 1) MADRL_PE_CASE(1, 1, 0); MADRL_PE_CASE(2, 1, 0); }
  if (cpl == 2) { if (epl == 1) MADRL_PE_CASE(1, 2, 0); MADRL_PE_CASE(2, 2, 0); }
  if (epl == 1) MADRL_PE_CASE(1, 4, 0);
  MADRL_PE_CASE(2, 4, 0);
#undef MADRL_PE_CASE
}

extern "C" int madrl_pursuit_reset(madrl_pursuit* h, const uint8_t* mask_dev, float* obs_dev, void* stream) {
  MADRL_REQUIRE(h != nullptr && obs_dev != nullptr, "handle/obs is NULL");
  return pe_launch(h, 1, 1, nullptr, obs_dev, nullptr, nullptr, nullptr, mask_dev, 0, (cudaStream_t)stream);
}

extern "C" int madrl_pursuit_rollout(madrl_pursuit* h, int T, const int32_t* actions_dev, float* obs_dev,
                                     float* rew_dev, uint8_t* done_dev, int32_t* info_dev,
                                     int auto_reset, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  MADRL_REQUIRE(T >= 1, "T must be >= 1");
  MADRL_REQUIRE(actions_dev && obs_dev && rew_dev && done_dev && info_dev, "NULL trajectory buffer");
  return pe_launch(h, 0, T, actions_dev, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream);
}

extern "C" int madrl_pursuit_rollout_heuristic(madrl_pursuit* h, int T, const float* obs0_dev, int32_t* actions_out_dev,
                                               float* obs_dev, float* rew_dev, uint8_t* done_dev, int32_t* info_dev,
                                               int auto_reset, int floor_centre, void* stream) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  MADRL_REQUIRE(T >= 1, "T must be >= 1");
  MADRL_REQUIRE(obs0_dev && obs_dev && rew_dev && done_dev && info_dev, "NULL trajectory buffer");
  MADRL_REQUIRE(h->cfg.layer_norm > 0.0, "the heuristic policy tests `evader channel > 0`: layer_norm must be positive");
  const int R = h->cfg.obs_range;
  return pe_launch(h, 0, T, nullptr, obs_dev, rew_dev, done_dev, info_dev, nullptr, auto_reset, (cudaStream_t)stream,
                   obs0_dev, actions_out_dev, floor_centre ? 2 * (R / 2) : R);
}

extern "C" int madrl_pursuit_step(madrl_pursuit* h, const int32_t* actions_dev, float* obs_dev, float* rew_dev,
                                  uint8_t* done_dev, int32_t* info_dev, int auto_reset, void* stream) {
  return madrl_pursuit_rollout(h, 1, actions_dev, obs_dev, rew_dev, done_dev, info_dev, auto_reset, stream);
}

extern "C" int madrl_pursuit_reset_host(madrl_pursuit* h, const uint8_t* mask_host, float* obs_host) {
  MADRL_REQUIRE(h != nullptr && obs_host != nullptr, "handle/obs is NULL");
  const size_t E = h->cfg.n_envs;
  return core_reset_host(h, E, E * h->cfg.n_pursuers * h->lay.obs_dim * 4, mask_host, obs_host,
                         [&](uint8_t* mask_dev, char* obs_dev) { return madrl_pursuit_reset(h, mask_dev, (float*)obs_dev, nullptr); });
}

extern "C" int madrl_pursuit_rollout_host2(madrl_pursuit* h, int T, const int32_t* actions_host, float* obs_host,
                                           float* rew_host, uint8_t* done_host, int32_t* info_host, int auto_reset,
                                           int flags) {
  MADRL_REQUIRE(h != nullptr, "handle is NULL");
  const size_t E = h->cfg.n_envs, Np = h->cfg.n_pursuers;
  const StepBytes sb = {E * Np * 4, E * Np * h->lay.obs_dim * 4, E * Np * 4, E, E * 4};
  return core_rollout_host(h, T, sb, actions_host, obs_host, rew_host, done_host, info_host, flags,
                           [&](int, int Tc, char* a, char* o, char* r, char* d, char* i, cudaStream_t st) {
                             return madrl_pursuit_rollout(h, Tc, (const int32_t*)a, (float*)o, (float*)r, (uint8_t*)d,
                                                          (int32_t*)i, auto_reset, st);
                           });
}

extern "C" int madrl_pursuit_rollout_host(madrl_pursuit* h, int T, const int32_t* actions_host, float* obs_host,
                                          float* rew_host, uint8_t* done_host, int32_t* info_host, int auto_reset) {
  return madrl_pursuit_rollout_host2(h, T, actions_host, obs_host, rew_host, done_host, info_host, auto_reset, 0);
}
