// ppg_eco.cu — the ECO environment step as one fused, persistent sm_100a kernel.
//
// Reproduces, for B independent env instances in lockstep, `PredPreyGrass.step()` / `reset()` of
//   ECO    = predpreygrass/evolutionary/eco_evolutionary/predpreygrass_rllib_env.py
//   GENOME = predpreygrass/evolutionary/eco_evolutionary/utils/genome.py
// (heritable speed trait, 5x5 action table with speed gating, locomotion cost, ageing, carcasses,
// float32 grid, own-speed observation plane).  Same machinery as ppg_base.cu — one warp per env, owner
// maps instead of a float grid, two-level gather for the observation rows, deterministic cross-env row
// allocation (ppg_step_common.cuh) — with ECO's phase order (ECO:295-507):
//   decay + ageing (ECO:582-616)  ->  age-outs in `self.agents` order  ->  grass regrowth (ECO:618-626)
//   ->  movement in action order (ECO:628-695)  ->  starvation in `agent_energies` order (ECO:311-316)
//   ->  prey eat grass (ECO:885-941)  ->  predators bite prey (ECO:786-883)  ->  removals
//   ->  reproduction with trait mutation (ECO:1092-1275, GENOME:49-59)  ->  outputs (ECO:372-501).
// List order = ascending agent id per species = the reference's `predator_positions` / `prey_positions`
// insertion order (ids come from an ascending deque and are never reused, ECO:238-272); the order ACROSS
// species (`self.agents`, `agent_energies`) is the per-agent insertion sequence number `seq`.
// A non-zero cell of the reference's float32 grid always equals float32(current energy) of the agent that
// wrote it last (every energy change is followed by a grid write: ECO:597,651-655,817,829,913,1154-1155), so
// the blocked test `grid > 0` (ECO:690) is `owner != 0 && (float)E[owner] > 0`.
//
// One exception has no owner: a prey that aged out in this step's ageing loop (grid cell zeroed, ECO:1073) is still in
// `agent_positions` when the predators engage (removal is Step 5, ECO:332-351); bitten under a finite intake cap it is
// written back to the grid as a carcass (ECO:826-832) and then removed WITHOUT the grid being zeroed — a stale positive
// value stays in the prey channel, blocks prey movers and shows up in observations until something overwrites or zeroes
// that cell.  These GHOST cells are carried per env in HBM (gh_cell / gh_val, at most PPG_MAX_GHOSTS) and loaded as
// pseudo-slots at the top of the prey list (not alive, no row, energy = the stale value), so the owner-map machinery
// treats them like the reference's grid does.
#include <cuda_runtime.h>

#include "ppg_step_common.cuh"

namespace ppg {

#define SEL(a) (s == 0 ? a[0] : a[1])

template <typename MapT>
struct EcoSmem {
  double* spd[2];
  uint16_t* age[2];
  uint16_t* seq[2];
  uint16_t* mord[2];  // mord[k] = slot of the k-th mover of the species (action-dict order, ECO:632)
  double* acc[2];     // CAD: move accumulators (cadence handles only)
};

template <typename MapT>
__device__ __forceinline__ EcoSmem<MapT> carve_eco(unsigned char* base, const StepParams& p) {
  EcoSmem<MapT> s;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    s.spd[k] = reinterpret_cast<double*>(base + p.so_spd[k]);
    s.age[k] = reinterpret_cast<uint16_t*>(base + p.so_age[k]);
    s.seq[k] = reinterpret_cast<uint16_t*>(base + p.so_seq[k]);
    s.mord[k] = reinterpret_cast<uint16_t*>(base + p.so_mord[k]);
    s.acc[k] = reinterpret_cast<double*>(base + p.so_acc[k]);
  }
  return s;
}

// own-speed plane value (ECO:707-711): float32((speed - lo) / (hi - lo)); 0 without a genome
#ifndef PPG_EXP_PLANE_NOINLINE
#define PPG_EXP_PLANE_NOINLINE 0
#endif
#if PPG_EXP_PLANE_NOINLINE
static __device__ __noinline__ float speed_plane(const StepParams& p, double spd) {
#else
__device__ __forceinline__ float speed_plane(const StepParams& p, double spd) {
#endif
  if (!p.speed_in_obs || spd < 0.0) return 0.f;
  if (p.trait_mode == PPG_TRAIT_CADENCE) return (float)spd;  // CAD:746: the genome value itself
  return (float)((spd - p.sp_lo) / (p.sp_hi - p.sp_lo));
}

// _genome_speed_to_move_rate / _get_agent_move_rate (CAD:556-575): 1 / max_cooldown .. 1, linear in the clamped speed
__device__ __forceinline__ double cad_move_rate(const StepParams& p, double spd) {
  if (spd < 0.0) return 1.0;  // no genome
  const double nrm = spd > 1.0 ? 1.0 : spd;
  const double min_rate = 1.0 / (double)p.max_cooldown;
  return min_rate + nrm * (1.0 - min_rate);
}

// speed ** exponent (ECO:559-563): CPython's float power = glibc pow, repeated bit for bit (include/ppg_pow.h)
#if defined(PPG_EXP_FASTPOW) && PPG_EXP_FASTPOW  // experiment only (NOT bit-exact): what the exact pow costs the kernel
static __device__ __forceinline__ double speed_cost_factor(double speed, double exponent) { return speed * speed; }
#else
static __device__ __noinline__ double speed_cost_factor(double speed, double exponent) { return ppg_pow(speed, exponent); }
#endif

// trait variants: gain factor metabolic_rate ** alpha (MR:751,807), 1.0 ** alpha = 1 without a genome
static __device__ __noinline__ double gain_factor(double rate, double alpha) { return ppg_pow(rate >= 0.0 ? rate : 1.0, alpha); }

// Founders of the NEXT episode of a trait-variant env (MR:189-192: two `rng.integers(min, max + 1)` draws, predators
// first): from the cell tape if it still has entries, else the FOUNDERS Philox stream keyed by the episode about to
// start.  Drawn when the reset is scheduled (episode end with auto-reset, ppg_reset), because the row allocator must know
// how many rows the reset will produce before it runs.  Packed pred | prey << 16 into EnvHdr.pad[0]; pad[1] bit 31 = drawn.
__device__ __forceinline__ void draw_next_founders(const StepParams& p, EnvHdr& h, unsigned genv) {
  if ((unsigned)h.pad[1] & 0x80000000u) return;  // already drawn for the pending reset
  int v[2];
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    const int lo = p.n_init_min[s], hi = p.n_init[s];
    int x;
    if (p.tape_cells != nullptr && h.tape_pos < h.tape_end) x = p.tape_cells[h.tape_pos++];
    else x = lo + (int)ppg_bounded(ppg_draw_u32(h.seed_key, genv, h.episode + 1u, PPG_STREAM_FOUNDERS, (unsigned)s), (unsigned)(hi - lo + 1));
    v[s] = x < lo ? lo : (x > hi ? hi : x);
  }
  h.pad[0] = v[0] | (v[1] << 16);
  h.pad[1] = (int)((unsigned)h.pad[1] | 0x80000000u);
}

// ---- lineage tracking (ECO:1422-1470), global arrays indexed by agent id; called by lane 0 only ----
// _set_lineage_alive_flag + _propagate_lineage_delta: a change of the agent's own alive flag moves the live-descendant
// count of every ancestor, dead or alive
static __device__ __noinline__ void lineage_set_alive(const StepParams& p, int env, int s, int id, int alive) {
  const size_t b = (size_t)env * p.n_possible[s];
  if (p.lin_alive[s][b + id] == (uint8_t)alive) return;
  p.lin_alive[s][b + id] = (uint8_t)alive;
  for (unsigned a = p.lin_parent[s][b + id]; a != 0xFFFFu; a = p.lin_parent[s][b + a])
    p.lin_live[s][b + a] = (int16_t)(p.lin_live[s][b + a] + (alive ? 1 : -1));
}
// _handle_lineage_birth (ECO:1461-1465)
static __device__ __noinline__ void lineage_birth(const StepParams& p, int env, int s, int id, unsigned parent) {
  const size_t b = (size_t)env * p.n_possible[s];
  p.lin_parent[s][b + id] = (uint16_t)parent; p.lin_live[s][b + id] = 0; p.lin_prev[s][b + id] = 0; p.lin_alive[s][b + id] = 0;
  lineage_set_alive(p, env, s, id, 1);
}

// one tape-or-Philox real draw (uniform lanes)
__device__ __forceinline__ bool take_real(const StepParams& p, EcoHdr& eh, EnvHdr& h, double& out) {
  if (p.tape_reals != nullptr) {
    if (eh.real_pos < eh.real_end) { out = p.tape_reals[eh.real_pos++]; return true; }
    h.status |= PPG_STATUS_TAPE_EXHAUSTED;
  }
  return false;
}

// smallest key > last among the agents selected by `pred` (key = seq << 16 | species << 15 | slot): the next agent in
// `self.agents` order.  Returns 0xFFFFFFFF when there is none.
template <typename F>
__device__ __forceinline__ unsigned next_in_seq_order(const uint16_t* const seq[2], const int n[2], long long last, int lane, F pred) {
  unsigned best = 0xFFFFFFFFu;
#pragma unroll
  for (int s = 0; s < 2; ++s)
    #pragma unroll 1
    for (int i = lane; i < n[s]; i += 32) {
      const unsigned key = ((unsigned)seq[s][i] << 16) | ((unsigned)s << 15) | (unsigned)i;
      if ((long long)key > last && pred(s, i)) best = min(best, key);
    }
  return __reduce_min_sync(FULL, best);
}

// _apply_cooperative_donation (COOP:537-589), warp-cooperative with uniform arguments: a cooperation_rate share of a
// positive gain goes in equal parts to the live agents of the donor's species within Chebyshev distance
// cooperation_range; every receiver's cell is re-written (COOP:573: of co-located receivers the later one in
// `predator_positions` / `prey_positions` order — the higher slot — shows).  Returns what the donor keeps.
template <typename MapT>
__device__ __noinline__ double coop_donation(unsigned char* sbase, const StepParams& p, int s, int slot, int n_s, double gain, int lane, double* donated) {
  const EnvSmem<MapT> S = carve<MapT>(sbase, p);
  const EcoSmem<MapT> X = carve_eco<MapT>(sbase, p);
  const int PP = p.P, PS = p.PS;
  if (!p.genome_enabled || !(gain > 0.0)) return gain;
  const double rate = SEL(X.spd)[slot] >= 0.0 ? SEL(X.spd)[slot] : 0.0;
  if (!(rate > 0.0)) return gain;
  const unsigned ps = SEL(S.pos)[slot];
  const int px = ps >> 8, py = ps & 255, r = p.coop_range;
  int cnt = 0;
  for (int b0 = 0; b0 < n_s; b0 += 32) {
    const int i = b0 + lane;
    bool nb = false;
    if (i < n_s && i != slot && (SEL(S.flg)[i] & F_ALIVE)) {
      const unsigned q = SEL(S.pos)[i];
      nb = max(abs((int)(q >> 8) - px), abs((int)(q & 255u) - py)) <= r;
    }
    cnt += __popc(__ballot_sync(FULL, nb));
  }
  if (cnt == 0) return gain;
  const double total = rate * gain, share = total / (double)cnt;
  if (donated != nullptr && lane == 0) *donated += total;  // total_energy_donated / total_energy_received (COOP:585-586), in call order
  for (int b0 = 0; b0 < n_s; b0 += 32) {
    const int i = b0 + lane;
    bool nb = false;
    int cell = 0;
    if (i < n_s && i != slot && (SEL(S.flg)[i] & F_ALIVE)) {
      const unsigned q = SEL(S.pos)[i];
      nb = max(abs((int)(q >> 8) - px), abs((int)(q & 255u) - py)) <= r;
      cell = CELLP(q);
    }
    if (nb) { SEL(S.E)[i] = SEL(S.E)[i] + share; SEL(S.map)[cell] = (MapT)(i + 1); }
    __syncwarp();
    bool need = nb && SEL(S.map)[cell] < (unsigned)(i + 1);
    while (__any_sync(FULL, need)) {
      if (need) SEL(S.map)[cell] = (MapT)(i + 1);
      __syncwarp();
      need = nb && SEL(S.map)[cell] < (unsigned)(i + 1);
    }
  }
  __syncwarp();
  return gain - total;
}

// TRAITS: false = eco_evolutionary itself (heritable speed), true = its sibling trait variants (p.trait_mode).  Two kernels,
// because the step kernels are bound by instruction delivery (DESIGN.md §3): the speed kernel carries none of the variants'
// code and the variants' kernel none of the speed / carcass / ageing code.
// KIND 2 = eco_evolutionary with lineage survival rewards (lineage_reward_coeff != 0; the shipped config has 0): a third
// kernel for the same reason.  KIND 10 + PPG_TRAIT_x = the kernel of ONE trait variant (trait_mode a compile-time constant:
// none of the other variants' code), used by the two-kernel step; KIND 1 keeps trait_mode a runtime value (one-kernel fallback).
template <int W, typename MapT, bool SPLIT, int KIND>
__global__ void __launch_bounds__(W * 32, 16 / W) ppg_step_eco_kernel(const __grid_constant__ StepParams p) {
  constexpr bool TRAITS = KIND == 1 || KIND >= 10, LIN = KIND == 2;
  // KIND 3 = eco_evolutionary WITHOUT the carcass machinery: max_energy_gain_per_prey = inf (every catch eats the whole prey:
  // no dead_prey, no ghost cells), no carcass_only_predator_age, no per-episode sums — the shipped config (BASELINE configs[3]).
  // The kernel is bound by instruction delivery: what the config cannot reach is not compiled in.
  constexpr bool LEAN = KIND == 3;
  constexpr unsigned FC = LEAN ? 0u : (unsigned)F_CARC;
  const int carcass_age = LEAN ? -1 : p.carcass_age;
  const double bite_cap_prey = LEAN ? HUGE_VAL : p.bite_cap_prey;
  double* const ep_sums = LEAN ? nullptr : p.ep_sums;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  wait_for_stream_predecessor();  // PDL chain: this grid may have become resident under the tail of the kernel before it
  if (SPLIT) allow_dependent_launch();  // the observation kernel may start filling the SMs' free slots right away
  unsigned char* const sbase = smem_raw + (size_t)warp * p.smem_per_env;
  const EnvSmem<MapT> S = carve<MapT>(sbase, p);
  const EcoSmem<MapT> X = carve_eco<MapT>(sbase, p);
  const RowDesc D = carve_desc(sbase, p);
  const unsigned sb32 = (unsigned)__cvta_generic_to_shared(sbase);
  const int G = p.G, GG = p.GG, PP = p.P, PS = p.PS;
  const unsigned lt_mask = (1u << lane) - 1u;
  const int AR = p.action_range, AD = (p.action_range - 1) / 2;

  #pragma unroll 1
  for (int i = lane; i < p.init_bytes / 16; i += 32)
    reinterpret_cast<uint4*>(sbase + p.so_map[0])[i] = __ldg(reinterpret_cast<const uint4*>(p.init_image) + i);
  unsigned rowctr = 0;
  EnvLoop L = env_loop(p, false);  // an env at its episode end may wait for the births of lower envs: index order
  __syncwarp();

  if (lane == 0) next_ticket(p, L, true);
  for (;;) {
    const int env = __shfl_sync(FULL, L.env_next, 0);
    if (env >= p.B) break;

    int n[2] = {0, 0};
    int births[2] = {0, 0};
    int old_base[2] = {0, 0};
    int new_base[2] = {0, 0};
    int next_live[2] = {0, 0};
    int mode = 0;
    unsigned env_flags = 0;
    EnvStats st = {};
    bool over = false, trunc = false, done = false, have_new_base = false;
    int n_gh = 0;  // ghost cells loaded into the pseudo-slots cap[1]-1, cap[1]-2, ...
    double ep_dist[2] = {0.0, 0.0}, ep_cost[2] = {0.0, 0.0};  // this step's distance moved / locomotion energy per species (per lane)
    // trait variants: the episode's event counters behind `training_metrics` (births blocked by the id pool / the density cap,
    // catches blocked by satiation, energy donated; MR:1347-1350, COOP:1365-1368) are bumped in place by lane 0 — rare events
    double* const ep_ev = (TRAITS && ep_sums != nullptr) ? ep_sums + (size_t)env * PPG_EP_STRIDE : nullptr;

    const long long t_env0 = clock64();
    const unsigned t_ns0 = globaltimer_lo();
    // ONE round trip for everything the env needs from HBM/L2 (ppg_base.cu): headers, prefix words, the first 32 entries of
    // both agent lists (speculatively: how many are valid is in the header), grass and the ghost count are all requested
    // before any of them is looked at.
    EnvHdr h = p.hdr[env];
    EcoHdr eh = p.ehdr[env];
    int prow_r[2] = {0, 0};
    double e_r[2] = {0.0, 0.0}, spd_r[2] = {0.0, 0.0};
    unsigned idpos_r[2] = {0, 0}, agseq_r[2] = {0, 0}, dead_r[2] = {0, 0};
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      if (lane < p.cap[s]) {
        const size_t b = (size_t)env * p.cap[s] + lane;
        prow_r[s] = p.ag_prow[s][b];
        e_r[s] = p.ag_e[s][b];
        spd_r[s] = p.ag_spd[s][b];
        idpos_r[s] = (unsigned)p.ag_id[s][b] | ((unsigned)p.ag_pos[s][b] << 16);
        agseq_r[s] = (unsigned)p.ag_age[s][b] | ((unsigned)p.ag_seq[s][b] << 16);
        dead_r[s] = p.ag_dead[s][b];
      }
    }
    unsigned gp_r[4] = {0, 0, 0, 0};
    double ge_r[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int g = lane + 32 * q;
      if (g < p.n_grass) { gp_r[q] = p.gr_pos[(size_t)env * p.n_grass + g]; ge_r[q] = p.gr_e[(size_t)env * p.n_grass + g]; }
    }
    const int n_gh_r = LEAN ? 0 : p.gh_n[env];
    const int tm = KIND >= 10 ? KIND - 10 : TRAITS ? p.trait_mode : PPG_TRAIT_SPEED;  // PPG_TRAIT_*: 0 = ECO (speed)
    if (TRAITS && tm == PPG_TRAIT_SPEED) __builtin_unreachable();
    // founders of the episode a reset starts: constant for ECO, drawn per episode by the trait variants (MR:189-192)
    int nf[2] = {p.n_init[0], p.n_init[1]};
    if (ppg_random_founders(tm) && ((unsigned)h.pad[1] & 0x80000000u)) { nf[0] = h.pad[0] & 0xFFFF; nf[1] = (h.pad[0] >> 16) & 0x7FFF; }
    mode = env_begin<SPLIT>(p, L, env, h.state, nf, old_base, next_live, lane);
    const unsigned genv = (unsigned)(env + p.env_base);

    if (PPG_UNLIKELY(mode == 1)) {
      // ------------------------------------------------------------------ reset() (ECO:274-293,123-223,1733-1792)
      h.episode += 1;
      h.step = 0;
      h.spawn_draws = 0;
      h.status = 0;
      h.state = 0;
      eh.trait_draws = 0;
      const int n_f = nf[0] + nf[1], n_total = n_f + p.n_grass;
      h.pad[1] = nf[0] | (nf[1] << 16);  // founders of the running episode; clears the "next founders drawn" bit
      // founder genomes first (ECO:216-221 register the founders before the placement draw, ECO:1752)
      if (p.genome_enabled) {
        double* sp0 = X.spd[0];
        double* sp1 = X.spd[1];
        if (p.tape_reals != nullptr && eh.real_pos + n_f <= eh.real_end) {
          #pragma unroll 1
          for (int k = lane; k < n_f; k += 32) {
            const double v = p.tape_reals[eh.real_pos + k];
            const double c = v < p.sp_lo ? p.sp_lo : (v > p.sp_hi ? p.sp_hi : v);
            if (k < nf[0]) sp0[k] = c; else sp1[k - nf[0]] = c;
          }
          eh.real_pos += n_f;
        } else {
          if (p.tape_reals != nullptr) h.status |= PPG_STATUS_TAPE_EXHAUSTED;
          // the polar method consumes a variable number of counters per draw; 32 attempts are evaluated at once and the
          // accepted ones handed to the founders in counter order (same stream as sequential draws)
          unsigned ctr = eh.trait_draws;
#pragma unroll 1
          for (int s = 0; s < 2; ++s) {
            if (p.f_std[s] > 0) {
              ctr = draw_normals_batched(SEL(X.spd), SEL(nf), p.f_mean[s], p.f_std[s], p.sp_lo, p.sp_hi, h.seed_key, genv, h.episode,
                                         PPG_STREAM_TRAIT, ctr, lane);
            } else {
              const double v = p.f_mean[s];
              #pragma unroll 1
              for (int i = lane; i < SEL(nf); i += 32) SEL(X.spd)[i] = v < p.sp_lo ? p.sp_lo : (v > p.sp_hi ? p.sp_hi : v);
            }
          }
          eh.trait_draws = ctr;
        }
      }
      if (tm == PPG_TRAIT_CADENCE) {  // CAD:1327: a random accumulator phase per founder, after the speeds
        if (p.tape_reals != nullptr && eh.real_pos + n_f <= eh.real_end) {
          #pragma unroll 1
          for (int k = lane; k < n_f; k += 32) {
            const double v = p.tape_reals[eh.real_pos + k];
            if (k < nf[0]) X.acc[0][k] = v; else X.acc[1][k - nf[0]] = v;
          }
          eh.real_pos += n_f;
        } else {
          if (p.tape_reals != nullptr) h.status |= PPG_STATUS_TAPE_EXHAUSTED;
          #pragma unroll 1
          for (int k = lane; k < n_f; k += 32) {
            unsigned ctr = eh.trait_draws + (unsigned)k;
            const double v = ppg_draw_u01(h.seed_key, genv, h.episode, PPG_STREAM_TRAIT, &ctr);
            if (k < nf[0]) X.acc[0][k] = v; else X.acc[1][k - nf[0]] = v;
          }
          eh.trait_draws += (unsigned)n_f;
        }
      }
      __syncwarp();
      int* cells = reinterpret_cast<int*>(S.vt[0]);
      unsigned* first = reinterpret_cast<unsigned*>(S.E[0]);
      bool from_tape = false;
      if (p.tape_cells != nullptr) {
        if (h.tape_pos + n_total <= h.tape_end) {
          #pragma unroll 1
          for (int i = lane; i < n_total; i += 32) cells[i] = p.tape_cells[h.tape_pos + i];
          h.tape_pos += n_total;
          from_tape = true;
        } else {
          h.status |= PPG_STATUS_TAPE_EXHAUSTED;
        }
      }
      if (!from_tape) philox_placement(cells, first, n_total, GG, genv, h.episode, h.seed_key, lane);
      __syncwarp();
      {
        int k0 = 0;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          #pragma unroll 1
          for (int i = lane; i < nf[s]; i += 32) {
            const int c = cells[k0 + i];
            const int cx = c / G, cy = c % G;
            S.id[s][i] = (uint16_t)i;
            S.pos[s][i] = (uint16_t)((cx << 8) | cy);
            S.flg[s][i] = F_ALIVE;
            X.age[s][i] = (uint16_t)((s == 0 && carcass_age >= 0) ? carcass_age : 0);  // ECO:1060-1068
            X.seq[s][i] = (uint16_t)(k0 + i);
            if (!p.genome_enabled) X.spd[s][i] = -1.0;
            S.map[s][CELLXY(cx, cy)] = (MapT)(i + 1);
          }
          k0 += nf[s];
          n[s] = nf[s];
          h.next_idx[s] = (unsigned short)nf[s];
        }
        __syncwarp();  // `first` aliases the energy arrays: write the energies only after the placement is read
#pragma unroll
        for (int s = 0; s < 2; ++s)
          #pragma unroll 1
          for (int i = lane; i < nf[s]; i += 32) S.E[s][i] = p.init_e[s];
        #pragma unroll 1
        for (int g = lane; g < p.n_grass; g += 32) {
          const int c = cells[k0 + g];
          const int cx = c / G, cy = c % G;
          S.gpos[g] = (uint16_t)((cx << 8) | cy);
          S.gE[g] = p.init_e_grass;
          S.map[2][CELLXY(cx, cy)] = (MapT)(g + 1);
        }
      }
      __syncwarp();
      eh.active[0] = nf[0]; eh.active[1] = nf[1];  // ECO:281-282
      if (LIN) {  // lineage_tracker = {} and one entry per founder: no parent, alive (ECO:171,1525-1526)
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const size_t b = (size_t)env * p.n_possible[s];
          #pragma unroll 1
          for (int i = lane; i < p.n_possible[s]; i += 32) {
            p.lin_parent[s][b + i] = 0xFFFFu; p.lin_live[s][b + i] = 0; p.lin_prev[s][b + i] = 0; p.lin_alive[s][b + i] = i < nf[s] ? 1 : 0;
          }
        }
      }
      eh.next_seq = (unsigned)n_f;
      next_live[0] = n[0]; next_live[1] = n[1];
      env_flags = PPG_ENV_RESET;
    } else if (mode == 2) {
      // ------------------------------------------------------------------ step() (ECO:295-507)
      n[0] = h.n_list[0]; n[1] = h.n_list[1];
      // second (and last) dependent round trip: the actions of the rows the agents occupied in the previous output
      int act_r[2] = {0, 0};
#pragma unroll
      for (int s = 0; s < 2; ++s)
        if (lane < SEL(n)) act_r[s] = p.actions[s][prow_r[s]];
      // meanwhile the grass from the registers: positions, and last step's energies (what the grass channel shows to the
      // agents that age out below; the regrowth is applied in place afterwards)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int g = lane + 32 * q;
        if (g < p.n_grass) { S.gpos[g] = (uint16_t)gp_r[q]; S.gE[g] = ge_r[q]; S.map[2][CELLP(gp_r[q])] = (MapT)(g + 1); }
      }
      #pragma unroll 1
      for (int g = lane + 128; g < p.n_grass; g += 32) {  // more than 128 patches: the rest the plain way
        const size_t b = (size_t)env * p.n_grass;
        const unsigned gp = p.gr_pos[b + g];
        S.gpos[g] = (uint16_t)gp; S.gE[g] = p.gr_e[b + g]; S.map[2][CELLP(gp)] = (MapT)(g + 1);
      }
      unsigned bad = 0;
      bool aged_any = false;
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        const size_t b = (size_t)env * p.cap[s];
        const int32_t* ordp = p.order[s];
        bool use_order = ordp != nullptr;
        if (PPG_UNLIKELY(use_order)) {  // must be a permutation of [0, n) (ppg_step_ordered); else fall back to list order
          bool ok = true;
          #pragma unroll 1
          for (int i = lane; i < SEL(n); i += 32) {
            const int d = ordp[p.ag_prow[s][b + i]];
            if ((unsigned)d < (unsigned)SEL(n)) SEL(X.mord)[d] = (uint16_t)i; else ok = false;
          }
          __syncwarp();
          #pragma unroll 1
          for (int i = lane; i < SEL(n); i += 32) {
            const int d = ordp[p.ag_prow[s][b + i]];
            if ((unsigned)d < (unsigned)SEL(n)) ok &= SEL(X.mord)[d] == (uint16_t)i;
          }
          use_order = __all_sync(FULL, ok);
          if (!use_order) bad = PPG_STATUS_BAD_ACTION;
          __syncwarp();
        }
        #pragma unroll 1
        for (int i = lane; i < SEL(n); i += 32) {
          // entries 0..31 are already in registers, with their actions
          int a;
          double e0, tr;
          unsigned idpos, agseq, deadv;
          if (i < 32) {
            a = SEL(act_r); e0 = SEL(e_r); tr = SEL(spd_r); idpos = SEL(idpos_r); agseq = SEL(agseq_r); deadv = SEL(dead_r);
          } else {
            a = p.actions[s][p.ag_prow[s][b + i]];
            e0 = p.ag_e[s][b + i]; tr = p.ag_spd[s][b + i];
            idpos = (unsigned)p.ag_id[s][b + i] | ((unsigned)p.ag_pos[s][b + i] << 16);
            agseq = (unsigned)p.ag_age[s][b + i] | ((unsigned)p.ag_seq[s][b + i] << 16);
            deadv = p.ag_dead[s][b + i];
          }
          if ((unsigned)a >= (unsigned)p.n_actions) { a = p.n_actions / 2; bad = PPG_STATUS_BAD_ACTION; }
          const bool carc = tm == PPG_TRAIT_SPEED && deadv != 0;  // trait variants: no carcasses (ag_dead[0] = satiation)
          unsigned age = agseq & 0xFFFFu;
          if (!carc) age += 1;  // carcasses do not age (ECO:600-601)
          SEL(S.id)[i] = (uint16_t)idpos;
          SEL(S.pos)[i] = (uint16_t)(idpos >> 16);
          // ECO:596; MR:555-561: the basal cost scales with the metabolic rate (1.0 without a genome); CAD:626-633: with 1 + coeff * speed
          double decay = tm == PPG_TRAIT_METABOLIC ? p.loss[s] * (tr >= 0.0 ? tr : 1.0) : p.loss[s];
          if (tm == PPG_TRAIT_CADENCE) {
            if (p.genome_enabled && p.meta_coeff > 0.0 && tr >= 0.0) decay = decay * (1.0 + p.meta_coeff * tr);
            SEL(X.acc)[i] = p.ag_acc[s][b + i];
          }
          SEL(S.E)[i] = e0 - decay;
          SEL(X.spd)[i] = tr;
          SEL(X.age)[i] = (uint16_t)age;
          SEL(X.seq)[i] = (uint16_t)(agseq >> 16);
          SEL(S.act)[i] = (uint8_t)a;
          SEL(S.flg)[i] = (uint8_t)(F_ALIVE | (carc ? FC : 0));
          if (!use_order) SEL(X.mord)[i] = (uint16_t)i;
          if (!carc && p.max_age[s] >= 0 && (int)age >= p.max_age[s]) aged_any = true;  // ECO:1052-1058
        }
      }
      h.status |= (unsigned char)__reduce_or_sync(FULL, bad);
      __syncwarp();
      // owner maps as the grid stands after the decay loop: of agents sharing a cell the later one in list order wrote last
#pragma unroll 1
      for (int s = 0; s < 2; ++s)
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int i = b0 + lane;
          const bool v = i < SEL(n);
          int cell = 0;
          if (v) { cell = CELLP((unsigned)SEL(S.pos)[i]); SEL(S.map)[cell] = (MapT)(i + 1); }
          __syncwarp();
          bool need = v && SEL(S.map)[cell] < (unsigned)(i + 1);
          while (__any_sync(FULL, need)) {
            if (need) SEL(S.map)[cell] = (MapT)(i + 1);
            __syncwarp();
            need = v && SEL(S.map)[cell] < (unsigned)(i + 1);
          }
        }
      __syncwarp();
      // ghost cells: the stale value is still on the grid unless a prey standing there has just re-written it (ECO:597)
      n_gh = n_gh_r;
      if (PPG_UNLIKELY(n_gh)) {
        if (lane < n_gh) {
          const int gs = p.cap[1] - 1 - lane;
          const unsigned gp = p.gh_cell[(size_t)env * PPG_MAX_GHOSTS + lane];
          const float gv = p.gh_val[(size_t)env * PPG_MAX_GHOSTS + lane];
          S.pos[1][gs] = (uint16_t)gp;
          S.E[1][gs] = (double)gv;
          S.flg[1][gs] = 0;
          S.vt[1][1 + gs] = gv;  // outside the range refresh_tables rewrites
          const int c = CELLP(gp);
          if (S.map[1][c] == 0) S.map[1][c] = (MapT)(gs + 1);
        }
        __syncwarp();
      }

      // age-outs (ECO:602-616,1060-1090), in self.agents order; the grass channel still shows last step's energies
      if (PPG_UNLIKELY(__any_sync(FULL, aged_any))) {
        long long last = -1;
        for (;;) {
          const unsigned key = next_in_seq_order(X.seq, n, last, lane, [&](int s, int i) {
            return !(S.flg[s][i] & FC) && p.max_age[s] >= 0 && (int)X.age[s][i] >= p.max_age[s];
          });
          if (key == 0xFFFFFFFFu) break;
          last = (long long)key;
          const int s = (key >> 15) & 1, slot = key & 0x7FFF;
          const int cell = CELLP((unsigned)SEL(S.pos)[slot]);
          rowctr = emit_row_now<MapT, false, true>(sbase, p, p.obs[s] + (size_t)(SEL(old_base) + slot) * p.elems[s], cell, s, n[0], n[1], rowctr,
                                                   lane, speed_plane(p, SEL(X.spd)[slot]));
          if (lane == 0) {
            SEL(S.map)[cell] = 0;
            SEL(S.flg)[slot] = F_DIED;
            if (LIN) lineage_set_alive(p, env, s, SEL(S.id)[slot], 0);  // ECO:1069
          }
          if (s == 0) eh.active[0] = max(eh.active[0] - 1, 0); else eh.active[1] = max(eh.active[1] - 1, 0);
          __syncwarp();
        }
      }
      // grass regrowth (ECO:618-626)
      #pragma unroll 1
      for (int g = lane; g < p.n_grass; g += 32) {
        const double v = S.gE[g] + p.grass_gain;
        S.gE[g] = v < p.grass_cap ? v : p.grass_cap;
      }
      __syncwarp();

      // movements in action-dict order per species (ECO:628-695)
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        MapT* own = SEL(S.map);
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int k = b0 + lane;
          int j = 0, oc = 0, tc = 0, nx0 = 0, ny0 = 0, d2 = 0;
          bool v = false;
          double fac_l = 1.0, dist_l = 0.0;  // speed ** exponent and step length of this lane's agent: ONE lane-parallel pow / sqrt per batch, also for the replay below
          if (k < SEL(n)) {
            j = SEL(X.mord)[k];
            const unsigned f = SEL(S.flg)[j];
            v = (f & F_ALIVE) && !(f & FC);  // terminated (ECO:633) and dead prey (ECO:636) do not move
            if (tm == PPG_TRAIT_CADENCE && v) {  // cadence gate (CAD:674-681): frozen agents keep their place, the accumulator still advances
              const double a = SEL(X.acc)[j] + cad_move_rate(p, SEL(X.spd)[j]);
              v = a >= 1.0;
              SEL(X.acc)[j] = v ? a - 1.0 : a;
            }
          }
          if (v) {
            const unsigned ps = SEL(S.pos)[j];
            const int a = SEL(S.act)[j];
            const int x = ps >> 8, y = ps & 255;
            int dx = a / AR - AD, dy = a % AR - AD;  // ECO:225-232
            const double sp = SEL(X.spd)[j];
            const int maxd = (sp >= 0.0 && sp >= p.sp_thr) ? p.fast_dist : p.slow_dist;  // ECO:551-557
            if (max(abs(dx), abs(dy)) > maxd) { dx = (dx > 0) - (dx < 0); dy = (dy > 0) - (dy < 0); dx *= maxd; dy *= maxd; }  // ECO:673-677
            nx0 = min(max(x + dx, 0), G - 1); ny0 = min(max(y + dy, 0), G - 1);
            d2 = (nx0 - x) * (nx0 - x) + (ny0 - y) * (ny0 - y);
            oc = CELLXY(x, y); tc = CELLXY(nx0, ny0);
            red_shared_add(reinterpret_cast<unsigned*>(S.scr) + (oc >> 2), 1u << ((oc & 3) * 8));
            if (tc != oc) red_shared_add(reinterpret_cast<unsigned*>(S.scr) + (tc >> 2), 1u << ((tc & 3) * 8));
            // _get_movement_energy_cost's speed factor (ECO:559-563; MR:531-539 (MR / INV / COOP): no speed factor), needed only by
            // an agent that can leave its cell
            if (tc != oc) {
              dist_l = sqrt((double)d2);
              if (sp >= 0.0 && !ppg_random_founders(tm)) fac_l = speed_cost_factor(sp, p.move_exp);
            }
          }
          __syncwarp();
          const bool dirty = v && (S.scr[oc] > 1 || S.scr[tc] > 1);
          __syncwarp();
          if (v) { S.scr[oc] = 0; S.scr[tc] = 0; }
          if (v && !dirty) {
            const unsigned ow = own[tc];
            const bool blocked = ow != 0 && (float)SEL(S.E)[ow - 1] > 0.f;  // float32 grid > 0 (ECO:690)
            const int nc = blocked ? oc : tc;
            if (!blocked && d2 > 0) {  // _get_movement_energy_cost (ECO:565-573)
              const double dist = dist_l, cost = p.move_cost[s] * dist * fac_l;
              SEL(S.E)[j] = SEL(S.E)[j] - cost;
              SEL(S.pos)[j] = (uint16_t)((nx0 << 8) | ny0);
              if (ep_sums) { if (s == 0) { ep_dist[0] += dist; ep_cost[0] += cost; } else { ep_dist[1] += dist; ep_cost[1] += cost; } }
            }
            own[oc] = 0;              // ECO:653,657
            own[nc] = (MapT)(j + 1);  // ECO:654,658
          }
          __syncwarp();
          unsigned dm = __ballot_sync(FULL, dirty);
          while (dm) {  // warp-uniform replay, in action order, of the agents that may interact
            const int l = __ffs(dm) - 1;
            dm &= dm - 1;
            const int jj = __shfl_sync(FULL, j, l);
            const double fac = __shfl_sync(FULL, fac_l, l), dist = __shfl_sync(FULL, dist_l, l);  // dd is 0 or the agent's own d2 (its cell has not changed yet)
            const unsigned ps = SEL(S.pos)[jj];
            const int a = SEL(S.act)[jj];
            const int xx = ps >> 8, yy = ps & 255;
            int dx = a / AR - AD, dy = a % AR - AD;
            const double sp = SEL(X.spd)[jj];
            const int maxd = (sp >= 0.0 && sp >= p.sp_thr) ? p.fast_dist : p.slow_dist;
            if (max(abs(dx), abs(dy)) > maxd) { dx = (dx > 0) - (dx < 0); dy = (dy > 0) - (dy < 0); dx *= maxd; dy *= maxd; }
            const int tx = min(max(xx + dx, 0), G - 1), ty = min(max(yy + dy, 0), G - 1);
            const unsigned ow = own[CELLXY(tx, ty)];
            const bool blocked = ow != 0 && (float)SEL(S.E)[ow - 1] > 0.f;
            const int nx = blocked ? xx : tx, ny = blocked ? yy : ty;
            const int dd = (nx - xx) * (nx - xx) + (ny - yy) * (ny - yy);
            double e = SEL(S.E)[jj];
            if (dd > 0) {
              const double cost = p.move_cost[s] * dist * fac;
              e = e - cost;
              if (ep_sums && lane == 0) { if (s == 0) { ep_dist[0] += dist; ep_cost[0] += cost; } else { ep_dist[1] += dist; ep_cost[1] += cost; } }
            }
            __syncwarp();
            if (lane == 0) {  // one writer: the two map stores may hit the same cell (blocked move) and must keep their order
              SEL(S.E)[jj] = e;
              own[CELLXY(xx, yy)] = 0;
              own[CELLXY(nx, ny)] = (MapT)(jj + 1);
              SEL(S.pos)[jj] = (uint16_t)((nx << 8) | ny);
            }
            __syncwarp();
          }
        }
      }

      // Step 4a: starvation over agent_energies = self.agents order (ECO:311-316,766-784); agents that aged out above are
      // handled again if their energy is <= 0 (no `terminations` guard: quirk 13)
      {
        bool sv = false;
#pragma unroll
        for (int s = 0; s < 2; ++s)
          #pragma unroll 1
          for (int i = lane; i < n[s]; i += 32) sv |= S.E[s][i] <= 0.0;
        if (__any_sync(FULL, sv)) {
          long long last = -1;
          for (;;) {
            const unsigned key = next_in_seq_order(X.seq, n, last, lane, [&](int s, int i) { return S.E[s][i] <= 0.0; });
            if (key == 0xFFFFFFFFu) break;
            last = (long long)key;
            const int s = (key >> 15) & 1, slot = key & 0x7FFF;
            const int cell = CELLP((unsigned)SEL(S.pos)[slot]);
            rowctr = emit_row_now<MapT, false, true>(sbase, p, p.obs[s] + (size_t)(SEL(old_base) + slot) * p.elems[s], cell, s, n[0], n[1],
                                                     rowctr, lane, speed_plane(p, SEL(X.spd)[slot]));
            if (lane == 0) {
              SEL(S.map)[cell] = 0;
              SEL(S.flg)[slot] = F_DIED;  // also drops FC (dead_prey.discard, ECO:768-769) and F_CAUGHT (reward 0, ECO:772)
              if (LIN) lineage_set_alive(p, env, s, SEL(S.id)[slot], 0);  // ECO:770
            }
            if (s == 0) { eh.active[0] -= 1; st.starved[0]++; } else { eh.active[1] -= 1; st.starved[1]++; }
            __syncwarp();
          }
        }
      }

      // COOP: a meal changes the neighbours' energies (COOP:828), so the prey go one by one in prey_positions order
      if (tm == PPG_TRAIT_COOPERATION) {
        for (int sl = 0; sl < n[1]; ++sl) {
          const unsigned f = S.flg[1][sl];
          if (!(f & F_ALIVE)) continue;
          const int cl = CELLP((unsigned)S.pos[1][sl]);
          const int gg = S.map[2][cl];
          if (!gg) continue;
          const double keep_gain = coop_donation<MapT>(sbase, p, 1, sl, n[1], S.gE[gg - 1], lane, ep_ev ? ep_ev + PPG_EP_DONATED + 1 : nullptr);
          const double en = S.E[1][sl] + keep_gain;
          __syncwarp();
          if (lane == 0) {
            S.E[1][sl] = en;
            S.map[1][cl] = (MapT)(sl + 1);
            S.gE[gg - 1] = 0.0;
            S.flg[1][sl] = (uint8_t)(f | F_ATE);
          }
          st.grass++;
          __syncwarp();
        }
      }
      // Step 4b: prey eat grass, prey_positions order (ECO:318-323,885-941)
      for (int b0 = 0; tm != PPG_TRAIT_COOPERATION && b0 < n[1]; b0 += 32) {
        const int slot = b0 + lane;
        int cell = 0, g = 0;
        bool act = false;
        if (slot < n[1]) {
          const unsigned f = S.flg[1][slot];
          act = (f & F_ALIVE) && !(f & FC);
          cell = CELLP((unsigned)S.pos[1][slot]);
          g = S.map[2][cell];
        }
        const bool eat = act && g != 0;
        if (eat) S.gtag[g - 1] = (uint8_t)lane;
        __syncwarp();
        const bool clash = eat && S.gtag[g - 1] != (uint8_t)lane;
        if (!__any_sync(FULL, clash)) {
          if (eat) {
            const double ge = S.gE[g - 1];
            const double bite = ge < p.bite_cap_grass ? ge : p.bite_cap_grass;  // ECO:909-911
            const double rem = ge - bite;
            // MR:807: gain = grass_energy * metabolic_rate ** alpha
            S.E[1][slot] = S.E[1][slot] + (tm == PPG_TRAIT_METABOLIC ? bite * gain_factor(X.spd[1][slot], p.trait_alpha) : bite);
            S.map[1][cell] = (MapT)(slot + 1);  // ECO:915
            S.gE[g - 1] = rem > 0.0 ? rem : 0.0;
            S.flg[1][slot] |= F_ATE;
          }
          st.grass += __popc(__ballot_sync(FULL, eat));
          __syncwarp();
          continue;
        }
        __syncwarp();
        const int kend = min(b0 + 32, n[1]);
        for (int sl = b0; sl < kend; ++sl) {  // two prey of this chunk share a patch: exact order
          const unsigned f = S.flg[1][sl];
          if (!(f & F_ALIVE) || (f & FC)) continue;
          const int cl = CELLP((unsigned)S.pos[1][sl]);
          const int gg = S.map[2][cl];
          if (gg) {
            const double ge = S.gE[gg - 1];
            const double bite = ge < p.bite_cap_grass ? ge : p.bite_cap_grass;
            const double rem = ge - bite;
            const double en = S.E[1][sl] + (tm == PPG_TRAIT_METABOLIC ? bite * gain_factor(X.spd[1][sl], p.trait_alpha) : bite);
            __syncwarp();
            if (lane == 0) {
              S.E[1][sl] = en;
              S.map[1][cl] = (MapT)(sl + 1);
              S.gE[gg - 1] = rem > 0.0 ? rem : 0.0;
              S.flg[1][sl] = (uint8_t)(f | F_ATE);
            }
            st.grass++;
            __syncwarp();
          }
        }
      }
      __syncwarp();

      // Step 4c: predators, predator_positions order (ECO:325-330,786-883).  Every prey still in agent_positions counts —
      // also those terminated earlier in this step (removal is Step 5) and carcasses.
      {
        const bool satiation = tm == PPG_TRAIT_METABOLIC || tm == PPG_TRAIT_INVESTMENT;
        if (satiation) {  // steps a predator still digests (agent_satiation_until - current_step, MR:734-740); mord is free after the moves
          #pragma unroll 1
          for (int i = lane; i < n[0]; i += 32) X.mord[0][i] = p.ag_dead[0][(size_t)env * p.cap[0] + i];
        }
        #pragma unroll 1
        for (int i = lane; i < n[1]; i += 32) S.scr[CELLP((unsigned)S.pos[1][i])] = 1;
        __syncwarp();
        for (int b0 = 0; b0 < n[0]; b0 += 32) {
          const int k = b0 + lane;
          bool cand = false;
          if (k < n[0]) {
            const int c0 = CELLP((unsigned)S.pos[0][k]);
            cand = S.scr[c0] != 0;
            if (tm == PPG_TRAIT_CADENCE)  // catch radius 1 (CAD:837-848): any prey on the 3x3 block (the halo of `scr` is never marked)
              cand = cand || S.scr[c0 - 1] || S.scr[c0 + 1] || S.scr[c0 - PS] || S.scr[c0 + PS] || S.scr[c0 - PS - 1] || S.scr[c0 - PS + 1] ||
                     S.scr[c0 + PS - 1] || S.scr[c0 + PS + 1];
            cand = cand && (S.flg[0][k] & F_ALIVE);
          }
          // MR:747-751 gain factor metabolic_rate ** alpha of the candidates: one lane-parallel pow, not one per catch in the ordered loop
          double gf_l = 1.0;
          if (tm == PPG_TRAIT_METABOLIC && cand) gf_l = gain_factor(X.spd[0][k], p.trait_alpha);
          unsigned m = __ballot_sync(FULL, cand);
          while (m) {
            const int slot = b0 + __ffs(m) - 1;
            m &= m - 1;
            const double gf = tm == PPG_TRAIT_METABOLIC ? __shfl_sync(FULL, gf_l, slot - b0) : 1.0;
            const unsigned ps = S.pos[0][slot];
            const int cell = CELLP(ps);
            // first prey in agent_positions order on my cell = lowest id = lowest list slot (ECO:797-799)
            unsigned best = 0xFFFFFFFFu;
            if (tm == PPG_TRAIT_CADENCE) {  // the nearest prey within Chebyshev distance 1, the first in agent_positions order on ties
              const int px = (int)(ps >> 8), py = (int)(ps & 255u);
              #pragma unroll 1
              for (int i = lane; i < n[1]; i += 32) {
                const unsigned qp = S.pos[1][i];
                const int d = max(abs(px - (int)(qp >> 8)), abs(py - (int)(qp & 255u)));
                if (d <= 1) best = min(best, ((unsigned)d << 16) | (unsigned)i);
              }
            } else {
              #pragma unroll 1
              for (int i = lane; i < n[1]; i += 32)
                if (S.pos[1][i] == ps) best = min(best, (unsigned)i);
            }
            best = __reduce_min_sync(FULL, best);
            if (best == 0xFFFFFFFFu) continue;
            const int q = (int)(best & 0xFFFFu);
            const int qcell = CELLP((unsigned)S.pos[1][q]);  // the prey's own cell (= `cell` except for cadence's radius-1 catches)
            const unsigned qf = S.flg[1][q];
            const bool was_dead = (qf & FC) != 0 || ((qf & F_DIED) && (qf & F_CAUGHT));  // dead_prey membership
            if (!was_dead && carcass_age >= 0 && (int)X.age[0][slot] < carcass_age) continue;  // juvenile: carcasses only (ECO:802-804)
            if (satiation && X.mord[0][slot] != 0) {  // still digesting: does not hunt this step (MR:734-740)
              if (ep_ev && lane == 0) ep_ev[PPG_EP_SATIATION_BLOCKED] += 1.0;  // satiation_blocked_catches_predator (MR:739)
              continue;
            }
            const double pe = S.E[1][q];
            const double bite = LEAN ? pe : (pe < bite_cap_prey ? pe : bite_cap_prey);  // ECO:812-814
            double rem = LEAN ? 0.0 : pe - bite;
            double en;
            if (tm == PPG_TRAIT_SPEED) en = S.E[0][slot] + bite;
            else {  // the trait variants always consume the prey (MR:759-773)
              rem = 0.0;
              if (tm == PPG_TRAIT_COOPERATION) en = S.E[0][slot] + coop_donation<MapT>(sbase, p, 0, slot, n[0], pe, lane, ep_ev ? ep_ev + PPG_EP_DONATED : nullptr);  // COOP:777
              else en = S.E[0][slot] + (tm == PPG_TRAIT_METABOLIC ? bite * gf : bite);  // MR:747-751
            }
            __syncwarp();
            if (lane == 0) {
              if (LIN && !was_dead) lineage_set_alive(p, env, 1, S.id[1][q], 0);  // the first bite is the prey's death for its lineage (ECO:840-841,848-849)
              S.E[0][slot] = en;
              S.map[0][cell] = (MapT)(slot + 1);  // ECO:817
              S.flg[0][slot] |= F_ATE;
              if (satiation && p.sat_cd > 0) X.mord[0][slot] = (uint16_t)p.sat_cd;  // MR:756-757
            }
            if (rem > 0.0) {  // carcass (ECO:826-845)
              if (lane == 0) {
                S.E[1][q] = rem;
                // a prey that aged out this step (F_DIED) is removed in Step 5 without the grid being zeroed: the entry written
                // here outlives its owner and becomes a ghost cell at write-back (see the header)
                S.map[1][qcell] = (MapT)(q + 1);
                S.flg[1][q] = (uint8_t)(qf | FC);
              }
              __syncwarp();
            } else {  // fully eaten (ECO:846-866); its observation is captured now
              __syncwarp();
              rowctr = emit_row_now<MapT, false, true>(sbase, p, p.obs[1] + (size_t)(old_base[1] + q) * p.elems[1], qcell, 1, n[0], n[1], rowctr,
                                                       lane, speed_plane(p, X.spd[1][q]));
              if (lane == 0) {
                S.map[1][qcell] = 0;
                S.flg[1][q] = (uint8_t)((qf & F_ATE) | F_DIED | F_CAUGHT);
              }
              eh.active[1] -= 1;  // also for a prey that already starved or aged out this step (quirk 4)
              st.eaten++;
              __syncwarp();
            }
          }
        }
        __syncwarp();  // every lane's candidate reads of the marks are done (racecheck: read / write on `scr`)
        #pragma unroll 1
        for (int i = lane; i < n[1]; i += 32) S.scr[CELLP((unsigned)S.pos[1][i])] = 0;
        __syncwarp();
      }

      // Step 6: reproduction, predators then prey, snapshot order (ECO:353-367,1092-1275).  If the episode may end on this
      // step the newborn rows are written at birth (ECO:1179 stays in self.observations, ECO:417-420).
      const bool maybe_done = eh.active[0] <= 0 || eh.active[1] <= 0;
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int k = b0 + lane;
          bool elig = false;
          if (k < SEL(n)) {
            const unsigned f = SEL(S.flg)[k];
            elig = (f & F_ALIVE) && !(f & FC) && SEL(S.E)[k] >= p.thr[s];
          }
          unsigned m = __ballot_sync(FULL, elig);
          while (m) {
            const int ps_slot = b0 + __ffs(m) - 1;
            m &= m - 1;
            if (s == 0 && tm == PPG_TRAIT_METABOLIC && p.repro_ratio >= 0.0 && (double)eh.active[0] >= p.repro_ratio * (double)eh.active[1]) {
              if (ep_ev && lane == 0) ep_ev[PPG_EP_BLOCKED_DENSITY] += 1.0;  // reproduction_blocked_due_to_density_predator (MR:852)
              continue;  // density-dependent soft cap (MR:843-854)
            }
            if ((s == 0 ? h.next_idx[0] : h.next_idx[1]) >= p.n_possible[s]) {  // ECO:1104-1111
              h.status |= PPG_STATUS_ID_POOL_EMPTY;
              if (ep_ev && lane == 0) ep_ev[PPG_EP_BLOCKED_CAPACITY + s] += 1.0;  // reproduction_blocked_due_to_capacity_* (MR:857,943)
              continue;
            }
            if (SEL(n) + SEL(births) >= p.cap[s] - (s == 1 ? n_gh : 0)) { h.status |= PPG_STATUS_SLOT_OVERFLOW; continue; }
            // mutate_genome (GENOME:49-59): the draws precede the spawn search (ECO:1119 before :1136)
            double spd = SEL(X.spd)[ps_slot];
            if (p.genome_enabled && p.mut_rate > 0 && p.mut_std > 0) {
              double u, d;
              if (!take_real(p, eh, h, u)) u = ppg_draw_u01(h.seed_key, genv, h.episode, PPG_STREAM_TRAIT, &eh.trait_draws);
              if (u < p.mut_rate) {
                if (!take_real(p, eh, h, d)) d = p.mut_std * ppg_draw_normal(h.seed_key, genv, h.episode, PPG_STREAM_TRAIT, &eh.trait_draws);
                const double v = spd + d;
                spd = v < p.sp_lo ? p.sp_lo : (v > p.sp_hi ? p.sp_hi : v);
              }
            }
            double acc0 = 0.0;
            if (tm == PPG_TRAIT_CADENCE && !take_real(p, eh, h, acc0))  // CAD:1327: after the genome, before the spawn search
              acc0 = ppg_draw_u01(h.seed_key, genv, h.episode, PPG_STREAM_TRAIT, &eh.trait_draws);
            const unsigned pp = SEL(S.pos)[ps_slot];
            const int px = pp >> 8, py = pp & 255;
            int nl[2] = {n[0] + births[0], n[1] + births[1]};
            int sx = -1, sy = -1;  // _find_available_spawn_position (ECO:732-764)
            int vx[4] = {0, 0, 0, 0}, vy[4] = {0, 0, 0, 0}, nv = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int cx = px + (c == 0 ? -1 : (c == 1 ? 1 : 0));
              const int cy = py + (c == 2 ? -1 : (c == 3 ? 1 : 0));
              if ((sx < 0 || tm == PPG_TRAIT_CADENCE) && cx >= 0 && cx < G && cy >= 0 && cy < G) {
                if (!any_agent_at(S, nl, (unsigned)((cx << 8) | cy), lane)) {
                  if (sx < 0) { sx = cx; sy = cy; }
                  if (tm == PPG_TRAIT_CADENCE) {
                    if (nv == 0) { vx[0] = cx; vy[0] = cy; } else if (nv == 1) { vx[1] = cx; vy[1] = cy; } else if (nv == 2) { vx[2] = cx; vy[2] = cy; } else { vx[3] = cx; vy[3] = cy; }
                    ++nv;
                  }
                }
              }
            }
            if (tm == PPG_TRAIT_CADENCE && nv > 0) {  // CAD:795 `valid_positions[rng.integers(len(valid_positions))]`
              if (p.tape_cells != nullptr && h.tape_pos < h.tape_end) {
                const int c = p.tape_cells[h.tape_pos++];  // the recorded choice
                sx = c / G; sy = c % G;
              } else {
                if (p.tape_cells != nullptr) h.status |= PPG_STATUS_TAPE_EXHAUSTED;
                const unsigned k = ppg_bounded(ppg_draw_u32(h.seed_key, genv, h.episode, PPG_STREAM_SPAWN, h.spawn_draws++), (unsigned)nv);
                sx = k == 0 ? vx[0] : (k == 1 ? vx[1] : (k == 2 ? vx[2] : vx[3]));
                sy = k == 0 ? vy[0] : (k == 1 ? vy[1] : (k == 2 ? vy[2] : vy[3]));
              }
            }
            if (PPG_UNLIKELY(sx < 0)) {
              st.fallback++;
              if (p.tape_cells != nullptr && h.tape_pos < h.tape_end) {
                const int c = p.tape_cells[h.tape_pos++];
                sx = c / G; sy = c % G;
              } else {
                if (p.tape_cells != nullptr) h.status |= PPG_STATUS_TAPE_EXHAUSTED;
                const int c = philox_free_cell<MapT>(sbase, p, nl[0], nl[1],
                                                     ppg_draw_u32(h.seed_key, genv, h.episode, PPG_STREAM_SPAWN, h.spawn_draws), lane);
                if (c >= 0) { h.spawn_draws++; sx = c >> 8; sy = c & 255; }
              }
              if (sx < 0) { h.status |= PPG_STATUS_NO_SPAWN_CELL; continue; }  // reference raises RuntimeError (ECO:1142-1143)
            }
            const int cs = SEL(n) + SEL(births);
            if (s == 0) births[0]++; else births[1]++;
            const int child_id = s == 0 ? h.next_idx[0]++ : h.next_idx[1]++;  // smallest never-used id (ECO:260-272)
            double child_e = p.init_e[s];
            if (tm == PPG_TRAIT_INVESTMENT) {  // INV:546-557,890,977: the PARENT's fraction of the parent's energy
              const double fr = SEL(X.spd)[ps_slot];
              child_e = SEL(S.E)[ps_slot] * (fr >= 0.0 ? fr : p.f_mean[s]);
            }
            const double pe = SEL(S.E)[ps_slot] - child_e;                    // ECO:1150
            __syncwarp();
            if (lane == 0) {  // one writer for the warp-uniform stores
              SEL(S.id)[cs] = (uint16_t)child_id;
              SEL(S.pos)[cs] = (uint16_t)((sx << 8) | sy);
              SEL(S.E)[cs] = child_e;
              SEL(S.flg)[cs] = (uint8_t)(F_ALIVE | F_NEWBORN | (maybe_done ? F_BORNROW : 0));
              SEL(X.age)[cs] = 0;
              SEL(X.seq)[cs] = (uint16_t)eh.next_seq;
              SEL(X.spd)[cs] = p.genome_enabled ? spd : -1.0;
              if (tm == PPG_TRAIT_CADENCE) SEL(X.acc)[cs] = acc0;
              if (LIN) lineage_birth(p, env, s, child_id, SEL(S.id)[ps_slot]);  // ECO:1525-1526
              SEL(S.E)[ps_slot] = pe;
              SEL(S.map)[CELLXY(sx, sy)] = (MapT)(cs + 1);       // ECO:1154
              SEL(S.map)[CELLXY(px, py)] = (MapT)(ps_slot + 1);  // ECO:1155
              SEL(S.flg)[ps_slot] |= F_REPRO;
            }
            eh.next_seq++;
            if (s == 0) eh.active[0] += 1; else eh.active[1] += 1;  // ECO:1157
            __syncwarp();
            if (SPLIT && maybe_done && cs - SEL(n) < PPG_BORN_K) {
              // the at-birth observation waits in the env's scratch rows; the observation kernel moves it to its row
              rowctr = emit_row_now<MapT, false, true>(sbase, p, p.born_obs[s] + ((size_t)env * PPG_BORN_K + (size_t)(cs - SEL(n))) * p.elems[s],
                                                       CELLXY(sx, sy), s, n[0] + births[0], n[1] + births[1], rowctr, lane,
                                                       speed_plane(p, SEL(X.spd)[cs]));
              __syncwarp();
            } else if (maybe_done) {
              if (!have_new_base) {
                newborn_base(p, L, env, lane, new_base);
                have_new_base = true;
              }
              rowctr = emit_row_now<MapT, false, true>(sbase, p, p.obs[s] + (size_t)(SEL(new_base) + cs - SEL(n)) * p.elems[s], CELLXY(sx, sy), s,
                                                       n[0] + births[0], n[1] + births[1], rowctr, lane, speed_plane(p, SEL(X.spd)[cs]));
              __syncwarp();
            }
          }
        }
      }
      __syncwarp();

      // Step 7: episode end (ECO:392), time limit (ECO:452)
      done = eh.active[1] <= 0 || eh.active[0] <= 0;
      h.step += 1;
      trunc = !done && h.step >= p.max_steps;
      over = done || trunc;
      env_flags = (done ? PPG_ENV_TERMINATED : 0) | (trunc ? PPG_ENV_TRUNCATED : 0);
      if (over) {
        if (p.autoreset) {
          if (ppg_random_founders(tm)) { draw_next_founders(p, h, genv); nf[0] = h.pad[0] & 0xFFFF; nf[1] = (h.pad[0] >> 16) & 0x7FFF; }
          next_live[0] = nf[0]; next_live[1] = nf[1];
        }
      } else {
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          int c = 0;
          #pragma unroll 1
          for (int i = lane; i < n[s] + births[s]; i += 32) c += (S.flg[s][i] & F_ALIVE) ? 1 : 0;
          next_live[s] = __reduce_add_sync(FULL, c);
        }
      }
    } else {
      env_flags = PPG_ENV_IDLE;
    }

    env_publish<SPLIT>(p, L, env, mode, next_live, births, 0, true, lane);

    // ------------------------------------------------- rows: metadata, observations, state write-back
    if (lane == 0) {
      p.old_off[0][env] = old_base[0];
      p.old_off[1][env] = old_base[1];
    }
    if (mode != 0) {
      const bool keep = !(over && p.autoreset);
      refresh_tables(S, p, n[0] + births[0], n[1] + births[1], lane);
      int wpos[2] = {0, 0};
      for (int pass = 0; pass < 2; ++pass) {  // 0: rows of the agents that acted, 1: newborn rows
        if (pass == 1) {
          if (births[0] + births[1] == 0) break;
          if (!SPLIT && !have_new_base) newborn_base(p, L, env, lane, new_base);
        }
#pragma unroll 1
        for (int s = 0; s < 2; ++s) {
          const size_t sb = (size_t)env * p.cap[s];
          float* obs_s = p.obs[s];
          const int elems = p.elems[s];
          const int k_lo = pass == 0 ? 0 : SEL(n), tot = pass == 0 ? SEL(n) : SEL(n) + SEL(births);
          if (k_lo >= tot) continue;
          RowRel rr;
          if (!SPLIT) rr = load_rel(p, s, sb32, lane);
          for (int b0 = k_lo; b0 < tot; b0 += 32) {
            const int slot = b0 + lane;
            int row = 0, cellp = 0;
            bool alive = false, emit = false;
            float sv = 0.f;
            unsigned nb_lab = 0;
            if (slot < tot) {
              const bool newborn = slot >= SEL(n);
              row = newborn ? SEL(new_base) + (slot - SEL(n)) : SEL(old_base) + slot;
              const unsigned f = SEL(S.flg)[slot];
              alive = (f & F_ALIVE) != 0;
              double rew = 0.0;
              if (mode == 2 && !newborn) {
                if (f & F_DIED) rew = (f & F_CAUGHT) ? p.pen_caught : 0.0;  // ECO:772,851 (aged out: rewards.get -> 0, ECO:1072)
                else {
                  rew = s == 0 ? ((f & F_ATE) ? p.r_catch : p.r_pstep) : ((f & F_ATE) ? p.r_eat : p.r_qstep);
                  if (f & F_REPRO) rew = p.r_repro[s];  // ECO:1161 overwrites
                  if (LIN) {  // Step 6.5 (ECO:943-984): coeff * change of the live-descendant count, for the living
                    const size_t li = (size_t)env * p.n_possible[s] + SEL(S.id)[slot];
                    const int cur_d = __ldcg(p.lin_live[s] + li), delta = cur_d - __ldcg(p.lin_prev[s] + li);  // written by lane 0 earlier in this step: read at L2
                    if (delta != 0) { p.lin_prev[s][li] = (int16_t)cur_d; rew = rew + p.lin_coeff[s] * (double)delta; }
                  }
                }
              }
              unsigned rf = 0;
              if ((f & F_DIED) || (alive && done)) rf |= PPG_ROW_TERMINATED;  // ECO:393-398
              if (alive && trunc) rf |= PPG_ROW_TRUNCATED;                    // ECO:452-472
              if (f & F_NEWBORN) rf |= PPG_ROW_NEWBORN;
              if (mode == 1) rf |= PPG_ROW_FOUNDER;
              if (f & F_ATE) rf |= PPG_ROW_ATE;
              if (f & F_REPRO) rf |= PPG_ROW_REPRODUCED;
              if (alive && (f & FC)) rf |= PPG_ROW_CARCASS;
              // CAD:577-585,746-753: the action mask of the row looks one increment ahead of the stored accumulator
              if (tm == PPG_TRAIT_CADENCE && !(SEL(X.acc)[slot] + cad_move_rate(p, SEL(X.spd)[slot]) >= 1.0)) rf |= PPG_ROW_FROZEN;
              if (!(SPLIT && newborn)) {
                p.row_env[s][row] = env;
                p.row_agent[s][row] = SEL(S.id)[slot];
                p.reward[s][row] = (float)rew;
                p.flags[s][row] = (uint8_t)rf;
              }
              nb_lab = (unsigned)SEL(S.id)[slot] | (rf << 16);
              cellp = CELLP((unsigned)SEL(S.pos)[slot]);
              emit = alive && !(done && (f & F_BORNROW));  // a newborn of the episode's last step keeps its at-birth observation
              sv = speed_plane(p, SEL(X.spd)[slot]);
            }
            const unsigned ma = __ballot_sync(FULL, alive);
            int dst = 0xFFFF;
            if (keep && alive) {
              dst = SEL(wpos) + __popc(ma & lt_mask);
              p.ag_id[s][sb + dst] = SEL(S.id)[slot];
              p.ag_pos[s][sb + dst] = SEL(S.pos)[slot];
              p.ag_e[s][sb + dst] = SEL(S.E)[slot];
              p.ag_prow[s][sb + dst] = row;
              p.ag_age[s][sb + dst] = SEL(X.age)[slot];
              p.ag_seq[s][sb + dst] = SEL(X.seq)[slot];
              p.ag_spd[s][sb + dst] = SEL(X.spd)[slot];
              if (tm == PPG_TRAIT_CADENCE) p.ag_acc[s][sb + dst] = SEL(X.acc)[slot];
              if (tm == PPG_TRAIT_SPEED) p.ag_dead[s][sb + dst] = (SEL(S.flg)[slot] & FC) ? 1 : 0;
              else {  // predators: steps of digestion left at the next step (MR:734-740,756-757)
                const unsigned rmn = (mode == 2 && s == 0 && slot < n[0] && (tm == PPG_TRAIT_METABOLIC || tm == PPG_TRAIT_INVESTMENT)) ? X.mord[0][slot] : 0u;
                p.ag_dead[s][sb + dst] = (uint8_t)(rmn > 0u ? rmn - 1u : 0u);
              }
            }
            if (s == 0) wpos[0] += __popc(ma); else wpos[1] += __popc(ma);
            if (SPLIT) {
              if (slot < tot) {
                const bool stashed = !emit && alive && slot >= SEL(n) && slot - SEL(n) < PPG_BORN_K;  // at-birth row in born_obs
                SEL(D.dsc)[slot] = (uint16_t)(emit ? (unsigned)cellp : (stashed ? DSC_COPY : DSC_SKIP));
                SEL(D.dsx)[slot] = stashed ? (unsigned)(slot - SEL(n)) : __float_as_uint(sv);
                if (pass == 1) p.nb_info[s][sb + (slot - SEL(n))] = (unsigned long long)nb_lab | ((unsigned long long)(unsigned)dst << 32);
              }
            } else {
              unsigned m = __ballot_sync(FULL, emit);
              while (m) {
                const int l = __ffs(m) - 1;
                m &= m - 1;
                const int cp = __shfl_sync(FULL, cellp, l);
                const int r = __shfl_sync(FULL, row, l);
                const float selfv = __shfl_sync(FULL, sv, l);
                emit_row<MapT, false, true>(p, sb32, obs_s + (size_t)r * elems, cp, s, rr, rowctr, lane, selfv);
              }
            }
          }
        }
      }
      env_rows_done<SPLIT>(p, L, sbase, env, mode, keep, old_base, n, births, new_base, next_live, lane);
      // ghost cells of the next step: loaded ghosts whose entry nobody overwrote or zeroed, and prey that aged out this
      // step and were written back as carcasses (their entry outlives them).  Only a finite intake cap can create them.
      {
        int kept = 0;
        if (keep && mode == 2 && (n_gh > 0 || bite_cap_prey < HUGE_VAL)) {
          const size_t gb = (size_t)env * PPG_MAX_GHOSTS;
          for (int b0 = -32; b0 < n[1]; b0 += 32) {  // first round: the loaded ghosts (pseudo-slots), then the list
            const int sl = b0 < 0 ? (lane < n_gh ? p.cap[1] - 1 - lane : -1) : (b0 + lane < n[1] ? b0 + lane : -1);
            bool gh = false;
            unsigned gp = 0;
            if (sl >= 0) {
              const unsigned f = S.flg[1][sl];
              gp = S.pos[1][sl];
              gh = (b0 < 0 || ((f & F_DIED) && (f & FC))) && S.map[1][CELLP(gp)] == (MapT)(sl + 1);
            }
            const unsigned m = __ballot_sync(FULL, gh);
            const int at = kept + __popc(m & lt_mask);
            if (gh && at < PPG_MAX_GHOSTS) {
              p.gh_cell[gb + at] = (uint16_t)gp;
              p.gh_val[gb + at] = (float)S.E[1][sl];
            }
            kept += __popc(m);
          }
          if (kept > PPG_MAX_GHOSTS) { h.status |= PPG_STATUS_GHOST_CELL; kept = PPG_MAX_GHOSTS; }
        }
        if (lane == 0 && (kept > 0 || n_gh > 0 || mode == 1)) p.gh_n[env] = (uint8_t)kept;
      }
      // leave the maps empty for the next env of this warp.  A carcass bitten after it aged out keeps an entry while its
      // owner is gone, so every loaded slot is un-written, alive or not (and so are the ghost pseudo-slots).
#pragma unroll
      for (int s = 0; s < 2; ++s)
        #pragma unroll 1
        for (int i = lane; i < n[s] + births[s]; i += 32) S.map[s][CELLP((unsigned)S.pos[s][i])] = 0;
      if (lane < n_gh) S.map[1][CELLP((unsigned)S.pos[1][p.cap[1] - 1 - lane])] = 0;
      #pragma unroll 1
      for (int g = lane; g < p.n_grass; g += 32) S.map[2][CELLP((unsigned)S.gpos[g])] = 0;
      if (keep) {
        h.n_list[0] = (unsigned short)wpos[0];
        h.n_list[1] = (unsigned short)wpos[1];
        const size_t gb = (size_t)env * p.n_grass;
        #pragma unroll 1
        for (int g = lane; g < p.n_grass; g += 32) {
          p.gr_e[gb + g] = S.gE[g];
          if (mode == 1) p.gr_pos[gb + g] = S.gpos[g];
        }
      }
      if (ep_sums) {
        // per-episode totals behind `_build_episode_training_metrics` (ECO:1613-1661): distance moved and locomotion energy of
        // all agents of a species (record["distance_traveled"], record["movement_energy_spent"], ECO:659-660)
        double v[4] = {ep_dist[0], ep_dist[1], ep_cost[0], ep_cost[1]};
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) v[q] += __shfl_xor_sync(FULL, v[q], d);
        if (lane < 4) {
          double* dst = ep_sums + (size_t)env * PPG_EP_STRIDE + lane;
          const double add = lane == 0 ? v[0] : lane == 1 ? v[1] : lane == 2 ? v[2] : v[3];
          *dst = mode == 1 ? 0.0 : *dst + add;
        } else if (lane < PPG_EP_STRIDE && mode == 1) ep_sums[(size_t)env * PPG_EP_STRIDE + lane] = 0.0;  // the event counters start with the episode

      }
      if (over) h.state = p.autoreset ? ST_NEEDS_RESET : ST_IDLE;
      if (lane == 0) { p.hdr[env] = h; p.ehdr[env] = eh; }
      add_stats(p, env, mode, n, births, over, trunc, h.step, st, lane);
    } else {
      env_idle<SPLIT>(p, sbase, env, old_base, lane);
    }
    env_end<SPLIT>(p, L, env, mode, n, births, env_flags, h, t_env0, t_ns0, eh.active, true, lane);
  }
  if (SPLIT) queue_push(p, L.pend, L.pend_env, lane);
}

// trait variants: founders of the episode a scheduled reset will start (see draw_next_founders), after ppg_reset marked the envs
__global__ void ppg_eco_founders_kernel(const StepParams p) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.B) return;
  EnvHdr h = p.hdr[e];
  if (!(h.state & ST_NEEDS_RESET)) return;
  draw_next_founders(p, h, (unsigned)(e + p.env_base));
  p.hdr[e] = h;
}

// reals cursor of the replay tape
__global__ void ppg_set_tape_reals_kernel(EcoHdr* ehdr, int B, const long long* real_off) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  ehdr[e].real_pos = real_off ? real_off[e] : 0;
  ehdr[e].real_end = real_off ? real_off[e + 1] : 0;
}

template <typename MapT>
static StepKernel eco_kernel(const StepParams& p) {
  const bool split = p.obs_split != 0;
  if (p.trait_mode != PPG_TRAIT_SPEED) {
    if (!split) return {ppg_step_eco_kernel<1, MapT, false, 1>, 32};
    switch (p.trait_mode) {
      case PPG_TRAIT_METABOLIC: return {ppg_step_eco_kernel<1, MapT, true, 10 + PPG_TRAIT_METABOLIC>, 32};
      case PPG_TRAIT_INVESTMENT: return {ppg_step_eco_kernel<1, MapT, true, 10 + PPG_TRAIT_INVESTMENT>, 32};
      case PPG_TRAIT_COOPERATION: return {ppg_step_eco_kernel<1, MapT, true, 10 + PPG_TRAIT_COOPERATION>, 32};
      case PPG_TRAIT_CADENCE: return {ppg_step_eco_kernel<1, MapT, true, 10 + PPG_TRAIT_CADENCE>, 32};
      default: return {nullptr, 0};
    }
  }
  if (p.lin_on) return {split ? ppg_step_eco_kernel<1, MapT, true, 2> : ppg_step_eco_kernel<1, MapT, false, 2>, 32};
  // the shipped config reaches none of the carcass / ghost-cell / juvenile / episode-sum code: the kernel without it (KIND 3)
  bool lean = split && !(p.bite_cap_prey < HUGE_VAL) && p.carcass_age < 0 && p.ep_sums == nullptr;
  if (const char* ev = getenv("PPG_ECO_LEAN")) lean = lean && atoi(ev) != 0;
  if (lean) return {ppg_step_eco_kernel<1, MapT, true, 3>, 32};
  return {split ? ppg_step_eco_kernel<1, MapT, true, 0> : ppg_step_eco_kernel<1, MapT, false, 0>, 32};
}

StepKernel step_kernel_eco(const StepParams& p) {
  return p.map_bytes == 1 ? eco_kernel<uint8_t>(p) : eco_kernel<uint16_t>(p);
}

cudaError_t launch_eco_founders(const StepParams& p, cudaStream_t s) {
  ppg_eco_founders_kernel<<<(p.B + 127) / 128, 128, 0, s>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_set_tape_reals(EcoHdr* ehdr, int B, const long long* real_off, cudaStream_t s) {
  ppg_set_tape_reals_kernel<<<(B + 255) / 256, 256, 0, s>>>(ehdr, B, real_off);
  return cudaGetLastError();
}

}  // namespace ppg
