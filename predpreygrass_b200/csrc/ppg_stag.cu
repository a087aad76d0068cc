// ppg_stag.cu — the STAG environment step as one fused, persistent sm_100a kernel.
//
// Reproduces, for B independent env instances in lockstep, `PredPreyGrass.step()` / `reset()` of
//   STAG = predpreygrass/evolutionary/stag_hunt_forward_view_nature_nurture/predpreygrass_rllib_env.py
// (two prey types — mammoths and rabbits — on separate grid channels, predator action [move, join_hunt], Moore-
// neighbourhood team capture with the nature/nurture success law, heritable cooperation trait, predator facing and
// the forward-shifted predator window, float32 grid, ended agents observed as all-zero rows).
// Same machinery as ppg_base.cu / ppg_eco.cu — one warp per env, owner maps instead of a float grid (one map per
// grid channel: predators, mammoths, rabbits, grass), two-level gather for the observation rows, deterministic
// cross-env row allocation (ppg_step_common.cuh) — with STAG's phase order (STAG:432-718):
//   decay + ageing (STAG:720-759)  ->  grass regrowth (STAG:761-769)  ->  movement in action order (STAG:801-890)
//   ->  starvation (STAG:448-453)  ->  prey engagements in prey_positions order: team capture, else grass
//   (STAG:456-460,1152-1500)  ->  reproduction, predators then prey (STAG:483-496,1502-1684)  ->  outputs (STAG:548-716).
// List order per species = insertion order of `self.agents` (founders, then births); nothing in the step depends on
// the order ACROSS species (movement blocks on the mover's own channels only, STAG:862-874).
// A non-zero cell of the reference's float32 grid always equals float32(current energy) of the agent that wrote it
// last (every energy change is followed by a grid write: STAG:744,820,1190,1294,1346,1468,1566-1567), so the blocked
// test `grid > 0` is `owner != 0 && (float)E[owner] > 0`.
#include <cuda_runtime.h>

#include "ppg_step_common.cuh"

namespace ppg {

#define SEL(a) (s == 0 ? a[0] : a[1])

// (1 - p0) ** ratio of the capture law (STAG:1137): CPython's float power = glibc pow, repeated bit for bit (include/ppg_pow.h)
static __device__ __noinline__ double capture_pow(double base, double exponent) { return ppg_pow(base, exponent); }

template <typename MapT>
struct StagSmem {
  MapT* map3;         // rabbits (grid channel 3); EnvSmem::map[1] holds the mammoths (channel 2), map[2] the grass
  double* trait;      // predator_cooperation_trait
  uint8_t* face;      // predator_facing as an index into _predator_facing_options (STAG:197-206)
  uint8_t* join;      // predator_join_intent of the running step
  uint16_t* age[2];
  uint16_t* mord[2];  // mord[k] = slot of the k-th mover of the species (action-dict order, STAG:805)
  uint16_t* jl;       // joiners of the capture attempt being resolved, predator_positions order (STAG:1069-1078,1161-1164)
  uint16_t* rl;       // free riders of the attempt
};

template <typename MapT>
__device__ __forceinline__ StagSmem<MapT> carve_stag(unsigned char* base, const StepParams& p) {
  StagSmem<MapT> s;
  s.map3 = reinterpret_cast<MapT*>(base + p.so_map[3]);
  s.trait = reinterpret_cast<double*>(base + p.so_trait);
  s.face = base + p.so_face;
  s.join = base + p.so_join;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    s.age[k] = reinterpret_cast<uint16_t*>(base + p.so_age[k]);
    s.mord[k] = reinterpret_cast<uint16_t*>(base + p.so_mord[k]);
  }
  s.jl = reinterpret_cast<uint16_t*>(base + p.so_ord[0]);  // the BASE family's engagement-order arrays are free here
  s.rl = reinterpret_cast<uint16_t*>(base + p.so_rnk[0]);
  return s;
}

// one tape-or-Philox real draw (uniform lanes)
__device__ __forceinline__ bool stag_take_real(const StepParams& p, StagHdr& sh, EnvHdr& h, double& out) {
  if (p.tape_reals != nullptr) {
    if (sh.real_pos < sh.real_end) { out = p.tape_reals[sh.real_pos++]; return true; }
    h.status |= PPG_STATUS_TAPE_EXHAUSTED;
  }
  return false;
}
__device__ __forceinline__ bool stag_take_int(const StepParams& p, EnvHdr& h, int& out) {
  if (p.tape_cells != nullptr) {
    if (h.tape_pos < h.tape_end) { out = p.tape_cells[h.tape_pos++]; return true; }
    h.status |= PPG_STATUS_TAPE_EXHAUSTED;
  }
  return false;
}

// Python's builtin sum() over floats (CPython >= 3.12: the first item exactly, the rest with Neumaier's compensated
// summation) of the energies of the listed predators
__device__ __forceinline__ double py_sum_energies(const double* E, const uint16_t* list, int n) {
  if (n == 0) return 0.0;
  double f = E[list[0]], c = 0.0;
  for (int k = 1; k < n; ++k) {
    const double x = E[list[k]], t = f + x;
    if (fabs(f) >= fabs(x)) c += (f - t) + x; else c += (x - t) + f;
    f = t;
  }
  if (c != 0.0 && isfinite(c)) f += c;
  return f;
}

// Window geometry of one row (STAG:944-1008).  Prey: centred on the agent.  Predators: centre shifted by facing * offset
// (`_get_predator_view_center`), and `_obs_clip` saturates when the shifted centre lies below 0: the window then
// behaves like one centred on coordinate 0 that is cut off after grid coordinate `centre + offset` (SURVEY quirk 11).
// Returns the padded cell index of the effective centre; ihi / jhi = last window row / column that may be non-zero.
__device__ __forceinline__ int stag_view(const StepParams& p, int s, unsigned ps, int f, int PP, int PS, int& ihi, int& jhi) {
  int x = (int)(ps >> 8), y = (int)(ps & 255u);
  const int R = p.R[s], off = p.off[s];
  ihi = R - 1; jhi = R - 1;
  if (s == 0) {
    const int q = f < 4 ? f : f + 1;  // facing index -> (dx + 1) * 3 + (dy + 1), the centre of the 3x3 is not a facing
    x += (q / 3 - 1) * off; y += (q % 3 - 1) * off;
    if (x < 0) { ihi = x + 2 * off; x = 0; }
    if (y < 0) { jhi = y + 2 * off; y = 0; }
  }
  return CELLXY(x, y);
}

template <typename MapT>
__device__ bool los_blocked(const MapT* wm, MapT WALL, int PS, int oc, int tc);

// `_get_move`'s block tests (STAG:860-890) for a move from padded cell `oc` to `tc`: a wall cell (static WALL entry of the
// predator map) blocks everybody; predators are blocked by a predator with energy > 0 — and the reference's `elif` chain
// ends there for them; prey by a prey of either type, else (respect_los_for_movement) by a wall corner cut diagonally or a
// wall strictly between the end points of the integer Bresenham walk (STAG:892-925).
template <typename MapT>
__device__ __forceinline__ bool move_blocked(const MapT* wm, const MapT* map1, const MapT* map3, const double* E0, const double* E1,
                                             const StepParams& p, int s, int oc, int tc) {
  const MapT WALL = (MapT)p.wall_idx;
  const unsigned ow = wm[tc];
  if (p.n_walls && ow == WALL) return true;
  if (s == 0) return ow != 0 && (float)E0[ow - 1] > 0.f;
  const unsigned o1 = map1[tc], o3 = map3[tc];
  if ((o1 != 0 && (float)E1[o1 - 1] > 0.f) || (o3 != 0 && (float)E1[o3 - 1] > 0.f)) return true;
  if (!p.los_move || !p.n_walls || tc == oc) return false;
  return los_blocked<MapT>(wm, WALL, p.PS, oc, tc);
}

// corner cutting and the Bresenham walk of `_line_of_sight_clear` (STAG:875-925) on the padded predator map
template <typename MapT>
__device__ __noinline__ bool los_blocked(const MapT* wm, MapT WALL, int PS, int oc, int tc) {
  // padded index -> (row, column) differences: rows are PS apart, |dy| < PS / 2
  int dxy = tc - oc, mx = 0;
  while (dxy > PS / 2) { dxy -= PS; ++mx; }
  while (dxy < -(PS / 2)) { dxy += PS; --mx; }
  const int my = dxy;
  const int adx = abs(mx), ady = abs(my);
  if (adx == 1 && ady == 1) return wm[oc + mx * PS] == WALL || wm[oc + my] == WALL;  // no corner cutting
  const int sx = mx > 0 ? 1 : -1, sy = my > 0 ? 1 : -1;
  int c = oc;
  if (adx >= ady) {
    double err = adx / 2.0;
    for (int i = 0; i < adx; ++i) {
      if (c != oc && c != tc && wm[c] == WALL) return true;
      err -= ady;
      if (err < 0) { c += sy; err += adx; }
      c += sx * PS;
    }
  } else {
    double err = ady / 2.0;
    for (int i = 0; i < ady; ++i) {
      if (c != oc && c != tc && wm[c] == WALL) return true;
      err -= adx;
      if (err < 0) { c += sx * PS; err += ady; }
      c += sy;
    }
  }
  return false;
}

template <int W, typename MapT, bool SPLIT>
__global__ void __launch_bounds__(W * 32, 16 / W) ppg_step_stag_kernel(const __grid_constant__ StepParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  wait_for_stream_predecessor();  // PDL chain: this grid may have become resident under the tail of the kernel before it
  if (SPLIT) allow_dependent_launch();  // the observation kernel may start filling the SMs' free slots right away
  unsigned char* const sbase = smem_raw + (size_t)warp * p.smem_per_env;
  const EnvSmem<MapT> S = carve<MapT>(sbase, p);
  const StagSmem<MapT> X = carve_stag<MapT>(sbase, p);
  const RowDesc D = carve_desc(sbase, p);
  const unsigned sb32 = (unsigned)__cvta_generic_to_shared(sbase);
  const int G = p.G, GG = p.GG, PP = p.P, PS = p.PS;
  const unsigned lt_mask = (1u << lane) - 1u;
  const int T2[2] = {p.n_possible_t[0][0], p.n_possible_t[1][0]};  // first flat id of type 2 per species

  #pragma unroll 1
  for (int i = lane; i < p.init_bytes / 16; i += 32)
    reinterpret_cast<uint4*>(sbase + p.so_map[0])[i] = __ldg(reinterpret_cast<const uint4*>(p.init_image) + i);
  unsigned rowctr = 0;
  EnvLoop L = env_loop(p, SPLIT);
  __syncwarp();

  // owner map of a prey slot's grid channel (STAG:2082-2092)
  auto prey_map = [&](int slot) -> MapT* { return (int)S.id[1][slot] >= T2[1] ? X.map3 : S.map[1]; };

  if (lane == 0) next_ticket(p, L, true);
  for (;;) {
    const int env = __shfl_sync(FULL, L.env_next, 0);
    if (env >= p.B) break;

    int n[2] = {0, 0};
    int births[2] = {0, 0};
    int old_base[2] = {0, 0};
    int new_base[2] = {0, 0};
    int next_live[2] = {0, 0};
    int live[2] = {0, 0};
    int mode = 0;
    unsigned env_flags = 0;
    EnvStats st = {};
    bool over = false, trunc = false, done = false;

    const long long t_env0 = clock64();
    const unsigned t_ns0 = globaltimer_lo();
    // ONE round trip for everything the env needs from HBM/L2 (ppg_base.cu): headers, prefix words, the first entries of
    // both agent lists (speculatively: how many are valid is in the header) and the grass are all requested before any of
    // them is looked at.
    EnvHdr h = p.hdr[env];
    StagHdr sh = p.shdr[env];
    int prow_r[3] = {0, 0, 0};
    double e_r[3] = {0.0, 0.0, 0.0}, trait_r = 0.0;
    unsigned idpos_r[3] = {0, 0, 0}, ageface_r[3] = {0, 0, 0};
#pragma unroll
    for (int q = 0; q < 3; ++q) {  // q = 0: predators 0..31, q = 1, 2: prey 0..63
      const int s = q ? 1 : 0, i = lane + (q == 2 ? 32 : 0);
      if (i < p.cap[s]) {
        const size_t b = (size_t)env * p.cap[s] + i;
        prow_r[q] = p.ag_prow[s][b];
        e_r[q] = p.ag_e[s][b];
        idpos_r[q] = (unsigned)p.ag_id[s][b] | ((unsigned)p.ag_pos[s][b] << 16);
        ageface_r[q] = (unsigned)p.ag_age[s][b];
        if (q == 0) { ageface_r[0] |= (unsigned)p.ag_face[b] << 16; trait_r = p.ag_trait[b]; }
      }
    }
    unsigned gp_r[4] = {0, 0, 0, 0};
    double ge_r[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int g = lane + 32 * q;
      if (g < p.n_grass) { gp_r[q] = p.gr_pos[(size_t)env * p.n_grass + g]; ge_r[q] = p.gr_e[(size_t)env * p.n_grass + g]; }
    }
    mode = env_begin<SPLIT>(p, L, env, h.state, p.n_init, old_base, next_live, lane);
    const unsigned genv = (unsigned)(env + p.env_base);

    if (PPG_UNLIKELY(mode == 1)) {
      // ------------------------------------------------------------------ reset() (STAG:414-430,268-412,2095-2193)
      h.episode += 1;
      h.step = 0;
      h.spawn_draws = 0;
      h.status = 0;
      h.state = 0;
      sh.trait_draws = 0;
      sh.capture_draws = 0;
      sh.facing_draws = (unsigned)p.n_init[0];  // the founders own facing draws 0..n-1 of the episode
#pragma unroll
      for (int k = 0; k < 12; ++k) sh.capture[k] = 0;
      sh.capture_real[0] = sh.capture_real[1] = sh.capture_real[2] = 0.0;
      const int n_f = p.n_init[0] + p.n_init[1], n_total = n_f + p.n_grass, n_pred = p.n_init[0];
      int* cells = reinterpret_cast<int*>(S.vt[0]);
      unsigned* first = reinterpret_cast<unsigned*>(S.E[0]);
      bool from_tape = false;
      if (p.tape_cells != nullptr) {
        if (h.tape_pos + n_total + n_pred <= h.tape_end) {  // the cells, then one facing index per founder predator
          #pragma unroll 1
          for (int i = lane; i < n_total; i += 32) cells[i] = p.tape_cells[h.tape_pos + i];
          #pragma unroll 1
          for (int i = lane; i < n_pred; i += 32) X.face[i] = (uint8_t)p.tape_cells[h.tape_pos + n_total + i];
          h.tape_pos += n_total + n_pred;
          from_tape = true;
        } else {
          h.status |= PPG_STATUS_TAPE_EXHAUSTED;
        }
      }
      if (!from_tape) {
        philox_placement(cells, first, n_total, GG, genv, h.episode, h.seed_key, lane, p.wall_cells, p.n_walls);
        #pragma unroll 1
        for (int i = lane; i < n_pred; i += 32)  // _random_predator_facing (STAG:939-942)
          X.face[i] = (uint8_t)ppg_bounded(ppg_draw_u32(h.seed_key, genv, h.episode, PPG_STREAM_FACING, (unsigned)i), 8u);
      }
      __syncwarp();
      // _sample_initial_predator_trait (STAG:1084-1088)
      if (p.coop_enabled) {
        if (p.tape_reals != nullptr && sh.real_pos + n_pred <= sh.real_end) {
          #pragma unroll 1
          for (int k = lane; k < n_pred; k += 32) {
            const double v = p.tape_reals[sh.real_pos + k];
            X.trait[k] = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
          }
          sh.real_pos += n_pred;
        } else {
          if (p.tape_reals != nullptr) h.status |= PPG_STATUS_TAPE_EXHAUSTED;
          if (p.trait_std > 0) {
            sh.trait_draws = draw_normals_batched(X.trait, n_pred, p.trait_mean, p.trait_std, 0.0, 1.0, h.seed_key, genv, h.episode,
                                                  PPG_STREAM_TRAIT, sh.trait_draws, lane);
          } else {
            const double v = p.trait_mean;
            #pragma unroll 1
            for (int k = lane; k < n_pred; k += 32) X.trait[k] = v < 0.0 ? 0.0 : (v > 1.0 ? 1.0 : v);
          }
        }
      } else {
        #pragma unroll 1
        for (int k = lane; k < n_pred; k += 32) X.trait[k] = 1.0;
      }
      __syncwarp();
      {
        // founders in `self.agents` order: predators type 1, type 2, prey type 1, type 2 (STAG:373-380)
        int k0 = 0;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          #pragma unroll 1
          for (int i = lane; i < p.n_init[s]; i += 32) {
            const int c = cells[k0 + i];
            const int cx = c / G, cy = c % G;
            const int t = i >= p.n_init_t[s][0];
            const int id = t ? T2[s] + (i - p.n_init_t[s][0]) : i;
            S.id[s][i] = (uint16_t)id;
            S.pos[s][i] = (uint16_t)((cx << 8) | cy);
            S.flg[s][i] = F_ALIVE;
            X.age[s][i] = 0;
            MapT* m = s == 0 ? S.map[0] : (t ? X.map3 : S.map[1]);
            m[CELLXY(cx, cy)] = (MapT)(i + 1);
          }
          k0 += p.n_init[s];
          n[s] = p.n_init[s];
        }
        __syncwarp();  // `first` aliases the energy arrays: write the energies only after the placement is read
        #pragma unroll 1
        for (int i = lane; i < p.n_init[0]; i += 32) S.E[0][i] = p.init_e[0];
        #pragma unroll 1
        for (int i = lane; i < p.n_init[1]; i += 32) S.E[1][i] = p.init_e_prey_t[i >= p.n_init_t[1][0]];
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
#pragma unroll
      for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int t = 0; t < 2; ++t) sh.next_idx_t[s][t] = (unsigned short)p.n_init_t[s][t];
      next_live[0] = n[0]; next_live[1] = n[1];
      live[0] = n[0]; live[1] = n[1];
      env_flags = PPG_ENV_RESET;
    } else if (mode == 2) {
      // ------------------------------------------------------------------ step() (STAG:432-718)
      n[0] = h.n_list[0]; n[1] = h.n_list[1];
      // second (and last) dependent round trip: the actions of the rows the agents occupied in the previous output
      int act_r[3] = {0, 0, 0};
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int s = q ? 1 : 0, i = lane + (q == 2 ? 32 : 0);
        if (i < SEL(n)) act_r[q] = p.actions[s][prow_r[q]];
      }
      // meanwhile: grass regrowth (STAG:761-769) from the registers
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int g = lane + 32 * q;
        if (g < p.n_grass) {
          S.gpos[g] = (uint16_t)gp_r[q];
          S.map[2][CELLP(gp_r[q])] = (MapT)(g + 1);
          const double v = ge_r[q] + p.grass_gain;
          S.gE[g] = v < p.grass_cap ? v : p.grass_cap;
        }
      }
      #pragma unroll 1
      for (int g = lane + 128; g < p.n_grass; g += 32) {  // more than 128 patches: the rest the plain way
        const size_t b = (size_t)env * p.n_grass;
        const unsigned gp = p.gr_pos[b + g];
        S.gpos[g] = (uint16_t)gp;
        S.map[2][CELLP(gp)] = (MapT)(g + 1);
        const double v = p.gr_e[b + g] + p.grass_gain;
        S.gE[g] = v < p.grass_cap ? v : p.grass_cap;
      }
      unsigned bad = 0;
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
          // entries 0..31 (predators) / 0..63 (prey) are already in registers, with their actions
          const int q = s == 0 ? (i < 32 ? 0 : 3) : (i < 32 ? 1 : (i < 64 ? 2 : 3));
          int a;
          double e0, trv = 0.0;
          unsigned idpos, ageface;
          if (q < 3) {
            a = q == 0 ? act_r[0] : (q == 1 ? act_r[1] : act_r[2]);
            e0 = q == 0 ? e_r[0] : (q == 1 ? e_r[1] : e_r[2]);
            idpos = q == 0 ? idpos_r[0] : (q == 1 ? idpos_r[1] : idpos_r[2]);
            ageface = q == 0 ? ageface_r[0] : (q == 1 ? ageface_r[1] : ageface_r[2]);
            trv = trait_r;
          } else {
            a = p.actions[s][p.ag_prow[s][b + i]];
            e0 = p.ag_e[s][b + i];
            idpos = (unsigned)p.ag_id[s][b + i] | ((unsigned)p.ag_pos[s][b + i] << 16);
            ageface = (unsigned)p.ag_age[s][b + i];
            if (s == 0) { ageface |= (unsigned)p.ag_face[b + i] << 16; trv = p.ag_trait[b + i]; }
          }
          const int id = (int)(idpos & 0xFFFFu);
          const int t = id >= T2[s];
          const int R = p.type_ar[t];
          int move = a & 0xFF;
          if (R > 0) {  // _generate_action_map (STAG:181-190); the reference raises KeyError on anything else
            if (a < 0 || move >= R * R) { bad = PPG_STATUS_BAD_ACTION; move = (R * R) / 2; }
          } else if (move != 0) {
            bad = PPG_STATUS_BAD_ACTION;
          }
          SEL(S.id)[i] = (uint16_t)id;
          SEL(S.pos)[i] = (uint16_t)(idpos >> 16);
          SEL(S.E)[i] = e0 - (s == 0 ? p.loss[0] : p.loss_prey_t[t]);  // STAG:742
          SEL(X.age)[i] = (uint16_t)((ageface & 0xFFFFu) + 1u);         // STAG:752
          SEL(S.act)[i] = (uint8_t)move;
          SEL(S.flg)[i] = F_ALIVE;
          if (s == 0) {
            X.join[i] = (uint8_t)((a >> PPG_STAG_JOIN_SHIFT) & 1);  // STAG:810-812
            X.face[i] = (uint8_t)(ageface >> 16);
            X.trait[i] = trv;
          }
          if (!use_order) SEL(X.mord)[i] = (uint16_t)i;
        }
      }
      h.status |= (unsigned char)__reduce_or_sync(FULL, bad);
      __syncwarp();
      // owner maps as the grid stands after the decay loop: of agents sharing a cell of one channel the later one in
      // list order wrote last
#pragma unroll 1
      for (int s = 0; s < 2; ++s)
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int i = b0 + lane;
          const bool v = i < SEL(n);
          int cell = 0;
          MapT* m = S.map[0];
          if (v) {
            cell = CELLP((unsigned)SEL(S.pos)[i]);
            if (s == 1) m = prey_map(i);
            m[cell] = (MapT)(i + 1);
          }
          __syncwarp();
          bool need = v && m[cell] < (unsigned)(i + 1);
          while (__any_sync(FULL, need)) {
            if (need) m[cell] = (MapT)(i + 1);
            __syncwarp();
            need = v && m[cell] < (unsigned)(i + 1);
          }
        }
      __syncwarp();

      // movements in action-dict order per species (STAG:801-890)
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int k = b0 + lane;
          int j = 0, oc = 0, tc = 0, nx0 = 0, ny0 = 0;
          const bool v = k < SEL(n);
          MapT* own = S.map[0];
          if (v) {
            j = SEL(X.mord)[k];
            const unsigned ps = SEL(S.pos)[j];
            const int a = SEL(S.act)[j];
            const int t = (int)SEL(S.id)[j] >= T2[s];
            const int R = p.type_ar[t];
            const int x = ps >> 8, y = ps & 255;
            int dx = 0, dy = 0;
            if (R > 0) { const int d = (R - 1) / 2; dx = a / R - d; dy = a % R - d; }
            if (s == 0) {
              if (dx != 0 || dy != 0) {  // _update_predator_facing: from the intended move, even if blocked (STAG:933-937)
                const int q = ((dx > 0) - (dx < 0) + 1) * 3 + ((dy > 0) - (dy < 0) + 1);
                X.face[j] = (uint8_t)(q < 4 ? q : q - 1);
              }
            } else {
              own = t ? X.map3 : S.map[1];
            }
            nx0 = min(max(x + dx, 0), G - 1); ny0 = min(max(y + dy, 0), G - 1);
            oc = CELLXY(x, y); tc = CELLXY(nx0, ny0);
            red_shared_add(reinterpret_cast<unsigned*>(S.scr) + (oc >> 2), 1u << ((oc & 3) * 8));
            if (tc != oc) red_shared_add(reinterpret_cast<unsigned*>(S.scr) + (tc >> 2), 1u << ((tc & 3) * 8));
          }
          __syncwarp();
          const bool dirty = v && (S.scr[oc] > 1 || S.scr[tc] > 1);
          __syncwarp();
          if (v) { S.scr[oc] = 0; S.scr[tc] = 0; }
          if (v && !dirty) {
            const bool blocked = move_blocked<MapT>(S.map[0], S.map[1], X.map3, S.E[0], S.E[1], p, s, oc, tc);
            const int nc = blocked ? oc : tc;
            if (!blocked) SEL(S.pos)[j] = (uint16_t)((nx0 << 8) | ny0);
            own[oc] = 0;              // STAG:819,824
            own[nc] = (MapT)(j + 1);  // STAG:820,825
          }
          __syncwarp();
          unsigned dm = __ballot_sync(FULL, dirty);
          while (dm) {  // warp-uniform replay, in action order, of the agents that may interact
            const int l = __ffs(dm) - 1;
            dm &= dm - 1;
            const int jj = __shfl_sync(FULL, j, l);
            const int tcl = __shfl_sync(FULL, tc, l), ocl = __shfl_sync(FULL, oc, l);
            const int nxl = __shfl_sync(FULL, nx0, l), nyl = __shfl_sync(FULL, ny0, l);
            const bool blocked = move_blocked<MapT>(S.map[0], S.map[1], X.map3, S.E[0], S.E[1], p, s, ocl, tcl);
            MapT* ownl = s == 0 ? S.map[0] : prey_map(jj);
            __syncwarp();
            if (lane == 0) {
              ownl[ocl] = 0;
              ownl[blocked ? ocl : tcl] = (MapT)(jj + 1);
              if (!blocked) SEL(S.pos)[jj] = (uint16_t)((nxl << 8) | nyl);
            }
            __syncwarp();
          }
        }
      }

      // Step 4a: starvation (STAG:448-453,1046-1067).  The loop runs in `agent_energies` order, but every effect is
      // order-free: the cell of the agent's channel is zeroed whoever the grid shows there, counters commute.
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        int c = 0;
        #pragma unroll 1
        for (int i = lane; i < SEL(n); i += 32)
          if (SEL(S.E)[i] <= 0.0) {
            MapT* m = s == 0 ? S.map[0] : prey_map(i);
            m[CELLP((unsigned)SEL(S.pos)[i])] = 0;
            SEL(S.flg)[i] = F_DIED;
            ++c;
          }
        c = __reduce_add_sync(FULL, c);
        if (s == 0) st.starved[0] += c; else st.starved[1] += c;
      }
      __syncwarp();

      // Step 4b: prey engagements in prey_positions order (STAG:456-460,1444-1500).  A prey can only be captured if a
      // live predator stands within Chebyshev distance 1; all other prey just eat grass and cannot interact with a
      // capture (they stand on different cells), so they go first, 32 at a time.
      #pragma unroll 1
      for (int i = lane; i < n[0]; i += 32)
        if (S.flg[0][i] & F_ALIVE) {
          const int c = CELLP((unsigned)S.pos[0][i]);
#pragma unroll
          for (int dx = -1; dx <= 1; ++dx)
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy) S.scr[c + dx * PS + dy] = 1;
        }
      __syncwarp();
      const double bite_cfg[2] = {p.bite_t[0] > 0.0 ? p.bite_t[0] : 0.0, p.bite_t[1] > 0.0 ? p.bite_t[1] : 0.0};  // max(0.0, b)
      // grass bite of one prey (STAG:1450-1478): mammoths leave a rabbit bite behind
      auto graze = [&](int slot, int g) {
        const double ge = S.gE[g - 1];
        const int t = (int)S.id[1][slot] >= T2[1];
        double bite;
        if (t == 0) {
          double allowed = ge - bite_cfg[1];
          if (!(allowed > 0.0)) allowed = 0.0;
          bite = bite_cfg[0];
          if (allowed < bite) bite = allowed;
          if (ge < bite) bite = ge;
        } else {
          bite = bite_cfg[1] < ge ? bite_cfg[1] : ge;
        }
        const double rem = ge - bite;
        S.E[1][slot] = S.E[1][slot] + bite;
        (t ? X.map3 : S.map[1])[CELLP((unsigned)S.pos[1][slot])] = (MapT)(slot + 1);  // STAG:1468
        S.gE[g - 1] = rem > 0.0 ? rem : 0.0;
        S.flg[1][slot] |= F_ATE;
      };
      bool any_hunted = false;
      for (int b0 = 0; b0 < n[1]; b0 += 32) {
        const int slot = b0 + lane;
        int cell = 0, g = 0;
        bool act = false;
        if (slot < n[1]) {
          cell = CELLP((unsigned)S.pos[1][slot]);
          const bool alive = (S.flg[1][slot] & F_ALIVE) != 0;
          const bool hunted = alive && S.scr[cell] != 0;
          any_hunted |= hunted;
          act = alive && !hunted;
          g = S.map[2][cell];
        }
        const bool eat = act && g != 0;
        if (eat) S.gtag[g - 1] = (uint8_t)lane;
        __syncwarp();
        const bool clash = eat && S.gtag[g - 1] != (uint8_t)lane;
        if (!__any_sync(FULL, clash)) {
          if (eat) graze(slot, g);
          st.grass += __popc(__ballot_sync(FULL, eat));
          __syncwarp();
          continue;
        }
        __syncwarp();
        unsigned em = __ballot_sync(FULL, eat);
        while (em) {  // two prey of this chunk share a patch: exact order
          const int l = __ffs(em) - 1;
          em &= em - 1;
          if (lane == l) graze(slot, g);
          st.grass++;
          __syncwarp();
        }
      }
      any_hunted = __any_sync(FULL, any_hunted);
      if (any_hunted) {
        for (int b0 = 0; b0 < n[1]; b0 += 32) {
          const int sl = b0 + lane;
          bool hunted = false;
          if (sl < n[1]) hunted = (S.flg[1][sl] & F_ALIVE) && S.scr[CELLP((unsigned)S.pos[1][sl])] != 0;
          unsigned hm = __ballot_sync(FULL, hunted);
          while (hm) {
            const int prey = b0 + __ffs(hm) - 1;
            hm &= hm - 1;
            // ---- _handle_team_capture (STAG:1152-1442)
            const unsigned pps = S.pos[1][prey];
            const int px = pps >> 8, py = pps & 255;
            const int pcell = CELLXY(px, py);
            const int ptype = (int)S.id[1][prey] >= T2[1];
            int nj = 0, nr = 0;
            for (int c0 = 0; c0 < n[0]; c0 += 32) {  // predator_positions order; Moore neighbourhood (STAG:1069-1078)
              const int k = c0 + lane;
              bool cand = false, isj = false;
              if (k < n[0]) {
                const unsigned f = S.flg[0][k];
                const unsigned q = S.pos[0][k];
                cand = (f & F_ALIVE) && !(f & F_ATE) && abs((int)(q >> 8) - px) <= 1 && abs((int)(q & 255) - py) <= 1;  // STAG:1158
                isj = cand && X.join[k] != 0;
              }
              const unsigned mj = __ballot_sync(FULL, isj), mr = __ballot_sync(FULL, cand && !isj);
              if (isj) X.jl[nj + __popc(mj & lt_mask)] = (uint16_t)k;
              else if (cand) X.rl[nr + __popc(mr & lt_mask)] = (uint16_t)k;
              nj += __popc(mj); nr += __popc(mr);
            }
            __syncwarp();
            bool captured = false;
            if (nj > 0) {  // STAG:1160-1166
              const double prey_energy = S.E[1][prey];
              // _compute_team_capture_success (STAG:1117-1150)
              const double mg = prey_energy + p.cap_margin;
              const double difficulty = mg > 1e-8 ? mg : 1e-8;
              double prob, ratio;
              bool success;
              if (!p.coop_enabled) {
                ratio = py_sum_energies(S.E[0], X.jl, nj) / difficulty;
                success = ratio > 1.0;
                prob = success ? 1.0 : 0.0;
              } else {
                double total = 0.0;
                for (int k = 0; k < nj; ++k) {
                  const int pid = X.jl[k];
                  const double factor = (1.0 - p.nature_w) + p.nature_w * X.trait[pid];
                  total += S.E[0][pid] * factor;
                }
                ratio = total / difficulty;
                const double ex = ratio > 0.0 ? ratio : 0.0;
                const double base_prob = 1.0 - capture_pow(1.0 - p.p0, ex);  // CPython `**` = glibc pow, bit for bit (include/ppg_pow.h)
                prob = base_prob > p.min_prob ? base_prob : p.min_prob;
                if (prob > 1.0) prob = 1.0;
                const bool force = ratio >= p.force_ratio;
                if (p.capture_model == PPG_CAPTURE_DETERMINISTIC) {
                  success = ratio > 1.0;
                  prob = success ? 1.0 : 0.0;
                } else if (p.capture_model == PPG_CAPTURE_PROBABILISTIC || !force) {
                  double u;
                  if (!stag_take_real(p, sh, h, u)) u = ppg_draw_u01(h.seed_key, genv, h.episode, PPG_STREAM_CAPTURE, &sh.capture_draws);
                  success = u < prob;
                } else {
                  success = true;  // hybrid, force_success: no draw (STAG:1148)
                }
              }
              sh.capture_real[0] = prob; sh.capture_real[1] = ratio; sh.capture_real[2] += prob;  // STAG:1176-1179
              sh.capture[8] += 1;
              st.attempts++;
              const double join_cost = p.join_cost;
              if (!success) {
                if (join_cost != 0.0) {  // STAG:1185-1192
                  #pragma unroll 1
                  for (int k = lane; k < nj; k += 32) S.E[0][X.jl[k]] -= join_cost;
                  __syncwarp();
                  if (lane == 0)
                    for (int k = 0; k < nj; ++k) S.map[0][CELLP((unsigned)S.pos[0][X.jl[k]])] = (MapT)(X.jl[k] + 1);
                  __syncwarp();
                }
                sh.capture[1] += 1; sh.capture[ptype ? 7 : 5] += 1;
                if (nj > 1) sh.capture[3] += 1;
              } else {
                sh.capture[0] += 1; sh.capture[ptype ? 6 : 4] += 1;  // STAG:1264-1271
                if (nj > 1) sh.capture[2] += 1;
                sh.capture[9] += nj;
                const double total_helper = py_sum_energies(S.E[0], X.jl, nj);  // STAG:1273-1274
                const double scav_frac = nr ? p.scav_frac : 0.0;
                const double scav_total = prey_energy * scav_frac;
                const double pool = prey_energy - scav_total;
                __syncwarp();
                #pragma unroll 1
                for (int k = lane; k < nj; k += 32) {  // STAG:1279-1297 (a joiner's snapshot energy is its energy right now)
                  const int pid = X.jl[k];
                  double e = S.E[0][pid];
                  double share;
                  if (p.equal_split) share = pool / (double)nj;
                  else share = total_helper > 0 ? pool * (e / total_helper) : 0.0;
                  e += share;
                  if (join_cost != 0.0) e -= join_cost;
                  S.E[0][pid] = e;
                  S.flg[0][pid] |= F_ATE;
                }
                const double scav_share = nr ? scav_total / (double)nr : 0.0;  // STAG:1338-1348
                if (scav_share != 0.0)
                  #pragma unroll 1
                  for (int k = lane; k < nr; k += 32) {
                    const int pid = X.rl[k];
                    S.E[0][pid] += scav_share;
                    S.flg[0][pid] |= F_ATE;
                  }
                __syncwarp();
                if (lane == 0) {
                  for (int k = 0; k < nj; ++k) S.map[0][CELLP((unsigned)S.pos[0][X.jl[k]])] = (MapT)(X.jl[k] + 1);
                  if (scav_share != 0.0)
                    for (int k = 0; k < nr; ++k) S.map[0][CELLP((unsigned)S.pos[0][X.rl[k]])] = (MapT)(X.rl[k] + 1);
                }
                __syncwarp();
                captured = true;
              }
              if (join_cost != 0.0) {  // joiners the cost starved (STAG:1238-1240,1402-1405)
                int c = 0;
                #pragma unroll 1
                for (int k = lane; k < nj; k += 32) {
                  const int pid = X.jl[k];
                  if (S.E[0][pid] <= 0.0 && (S.flg[0][pid] & F_ALIVE)) {
                    S.map[0][CELLP((unsigned)S.pos[0][pid])] = 0;
                    S.flg[0][pid] = (uint8_t)((S.flg[0][pid] & F_ATE) | F_DIED);
                    ++c;
                  }
                }
                st.starved[0] += __reduce_add_sync(FULL, c);
                __syncwarp();
              }
              if (captured) {  // prey termination (STAG:1419-1440)
                if (lane == 0) {
                  (ptype ? X.map3 : S.map[1])[pcell] = 0;
                  S.flg[1][prey] = F_DIED | F_CAUGHT;
                }
                st.eaten++;
                __syncwarp();
              }
            }
            if (!captured) {  // STAG:1450-1498
              const int g = S.map[2][pcell];
              if (g != 0) {
                if (lane == 0) graze(prey, g);
                st.grass++;
              }
              __syncwarp();
            }
          }
        }
      }
      #pragma unroll 1
      for (int i = lane; i < n[0]; i += 32) {  // un-mark (around every loaded predator: the counters are all zero between uses)
        const int c = CELLP((unsigned)S.pos[0][i]);
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx)
#pragma unroll
          for (int dy = -1; dy <= 1; ++dy) S.scr[c + dx * PS + dy] = 0;
      }
      __syncwarp();

      // Step 7: reproduction, predators then prey, snapshot order (STAG:483-496,1502-1684)
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int k = b0 + lane;
          bool elig = false;
          if (k < SEL(n)) {
            const int t = (int)SEL(S.id)[k] >= T2[s];
            elig = (SEL(S.flg)[k] & F_ALIVE) && SEL(S.E)[k] >= (s == 0 ? p.thr[0] : p.thr_prey_t[t]);
          }
          unsigned m = __ballot_sync(FULL, elig);
          while (m) {
            const int ps_slot = b0 + __ffs(m) - 1;
            m &= m - 1;
            const int t = (int)SEL(S.id)[ps_slot] >= T2[s];
            if (sh.next_idx_t[s][t] >= p.n_possible_t[s][t]) { h.status |= PPG_STATUS_ID_POOL_EMPTY; continue; }  // STAG:1510-1523
            if (SEL(n) + SEL(births) >= p.cap[s]) { h.status |= PPG_STATUS_SLOT_OVERFLOW; continue; }
            // _inherit_predator_trait (STAG:1090-1097): the draws precede the spawn search (STAG:1535 before :1555)
            double child_trait = 1.0;
            if (s == 0 && p.coop_enabled) {
              child_trait = X.trait[ps_slot];
              if (p.trait_mut_std > 0.0) {
                double u, d;
                if (!stag_take_real(p, sh, h, u)) u = ppg_draw_u01(h.seed_key, genv, h.episode, PPG_STREAM_TRAIT, &sh.trait_draws);
                if (u < p.trait_mut_rate) {
                  if (!stag_take_real(p, sh, h, d)) d = p.trait_mut_std * ppg_draw_normal(h.seed_key, genv, h.episode, PPG_STREAM_TRAIT, &sh.trait_draws);
                  child_trait += d;
                }
              }
              child_trait = child_trait < 0.0 ? 0.0 : (child_trait > 1.0 ? 1.0 : child_trait);
            }
            const unsigned pp = SEL(S.pos)[ps_slot];
            const int px = pp >> 8, py = pp & 255;
            int nl[2] = {n[0] + births[0], n[1] + births[1]};
            int sx = -1, sy = -1;  // _find_available_spawn_position (STAG:1010-1044)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int cx = px + (c == 0 ? -1 : (c == 1 ? 1 : 0));
              const int cy = py + (c == 2 ? -1 : (c == 3 ? 1 : 0));
              if (sx < 0 && cx >= 0 && cx < G && cy >= 0 && cy < G) {
                if (!(p.n_walls && S.map[0][CELLXY(cx, cy)] == (MapT)p.wall_idx) && !any_agent_at(S, nl, (unsigned)((cx << 8) | cy), lane)) { sx = cx; sy = cy; }  // STAG:1026-1027
              }
            }
            if (sx < 0) {
              if (count_free_cells<MapT>(sbase, p, nl[0], nl[1], lane) == 0) { h.status |= PPG_STATUS_NO_SPAWN_CELL; continue; }  // no draw (STAG:1041-1044)
              st.fallback++;
              int c;
              if (stag_take_int(p, h, c)) { sx = c / G; sy = c % G; }
              else {
                c = philox_free_cell<MapT>(sbase, p, nl[0], nl[1], ppg_draw_u32(h.seed_key, genv, h.episode, PPG_STREAM_SPAWN, h.spawn_draws), lane);
                h.spawn_draws++;
                sx = c >> 8; sy = c & 255;
              }
            }
            const int cs = SEL(n) + SEL(births);
            if (s == 0) births[0]++; else births[1]++;
            const int child_id = (t ? T2[s] : 0) + sh.next_idx_t[s][t]++;  // _alloc_new_id (STAG:2240-2253)
            const double child_e = s == 0 ? p.init_e[0] : p.init_e_prey_t[t];
            const double pe = SEL(S.E)[ps_slot] - child_e;
            int f = 0;
            if (s == 0) {
              if (!stag_take_int(p, h, f)) f = (int)ppg_bounded(ppg_draw_u32(h.seed_key, genv, h.episode, PPG_STREAM_FACING, sh.facing_draws++), 8u);  // STAG:1559
              sh.capture[10] += 1;
            } else {
              sh.capture[11] += 1;
            }
            __syncwarp();
            if (lane == 0) {
              SEL(S.id)[cs] = (uint16_t)child_id;
              SEL(S.pos)[cs] = (uint16_t)((sx << 8) | sy);
              SEL(S.E)[cs] = child_e;
              SEL(S.flg)[cs] = F_ALIVE | F_NEWBORN;
              SEL(X.age)[cs] = 0;
              if (s == 0) { X.trait[cs] = child_trait; X.face[cs] = (uint8_t)f; }
              SEL(S.E)[ps_slot] = pe;
              MapT* m = s == 0 ? S.map[0] : (t ? X.map3 : S.map[1]);
              m[CELLXY(sx, sy)] = (MapT)(cs + 1);       // STAG:1566,1660
              m[CELLXY(px, py)] = (MapT)(ps_slot + 1);  // STAG:1567,1661
              SEL(S.flg)[ps_slot] |= F_REPRO;
            }
            __syncwarp();
          }
        }
      }
      __syncwarp();

      // Step 8: episode end (STAG:584-594), time limit (STAG:657-716)
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        int c = 0;
        #pragma unroll 1
        for (int i = lane; i < n[s] + births[s]; i += 32) c += (S.flg[s][i] & F_ALIVE) ? 1 : 0;
        live[s] = __reduce_add_sync(FULL, c);
      }
      done = live[0] <= 0 || live[1] <= 0;
      h.step += 1;
      trunc = h.step >= p.max_steps;  // overrides: survivors are truncated, "__all__" terminated becomes False
      over = done || trunc;
      env_flags = trunc ? PPG_ENV_TRUNCATED : (done ? PPG_ENV_TERMINATED : 0);
      if (over) {
        if (p.autoreset) { next_live[0] = p.n_init[0]; next_live[1] = p.n_init[1]; }
      } else {
        next_live[0] = live[0]; next_live[1] = live[1];
      }
    } else {
      env_flags = PPG_ENV_IDLE;
    }

    env_publish<SPLIT>(p, L, env, mode, next_live, births, (L.n_old_total[0] + L.n_old_total[1]) / p.B * 5 / 4, true, lane);

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
          if (!SPLIT) newborn_base(p, L, env, lane, new_base);
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
            int row = 0, cellp = 0, ihi = 0, jhi = 0;
            bool alive = false, valid = false;
            unsigned nb_lab = 0;
            if (slot < tot) {
              valid = true;
              const bool newborn = slot >= SEL(n);
              row = newborn ? SEL(new_base) + (slot - SEL(n)) : SEL(old_base) + slot;
              const unsigned f = SEL(S.flg)[slot];
              alive = (f & F_ALIVE) != 0;
              const int t = (int)SEL(S.id)[slot] >= T2[s];
              double rew = 0.0;
              if (mode == 2 && !newborn) {
                if (f & F_DIED) rew = p.strict_out ? (s == 0 ? p.death_pen[0] : p.death_pen[1 + t]) : 0.0;  // STAG:1050-1054,577,609
                else if (f & F_REPRO) rew = p.r_repro_t[s][t];                                               // STAG:1573,1667
              }
              unsigned rf = 0;
              if (f & F_DIED) rf |= PPG_ROW_TERMINATED;
              if (alive && (done || trunc)) rf |= PPG_ROW_TRUNCATED;  // STAG:587-591,659-716
              if (f & F_NEWBORN) rf |= PPG_ROW_NEWBORN;
              if (mode == 1) rf |= PPG_ROW_FOUNDER;
              if (f & F_ATE) rf |= PPG_ROW_ATE;
              if (f & F_REPRO) rf |= PPG_ROW_REPRODUCED;
              if (!(SPLIT && newborn)) {
                p.row_env[s][row] = env;
                p.row_agent[s][row] = SEL(S.id)[slot];
                p.reward[s][row] = (float)rew;
                p.flags[s][row] = (uint8_t)rf;
              }
              nb_lab = (unsigned)SEL(S.id)[slot] | (rf << 16);
              cellp = stag_view(p, s, SEL(S.pos)[slot], s == 0 ? (int)X.face[slot] : 0, PP, PS, ihi, jhi);
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
              if (s == 0) { p.ag_face[sb + dst] = X.face[slot]; p.ag_trait[sb + dst] = X.trait[slot]; }
            }
            if (s == 0) wpos[0] += __popc(ma); else wpos[1] += __popc(ma);
            if (SPLIT) {
              if (valid) {
                SEL(D.dsc)[slot] = (uint16_t)(alive ? (unsigned)cellp : DSC_ZERO);  // ended: all-zero observation (STAG:596-612)
                SEL(D.dsx)[slot] = (unsigned)ihi | ((unsigned)jhi << 8);
                if (pass == 1) p.nb_info[s][sb + (slot - SEL(n))] = (unsigned long long)nb_lab | ((unsigned long long)(unsigned)dst << 32);
              }
              continue;
            }
            unsigned m = __ballot_sync(FULL, valid);
            while (m) {
              const int l = __ffs(m) - 1;
              m &= m - 1;
              const int r = __shfl_sync(FULL, row, l);
              float* dst = obs_s + (size_t)r * elems;
              if (!((ma >> l) & 1u)) { zero_row(dst, elems, lane); continue; }  // ended: all-zero observation (STAG:596-612)
              const int cp = __shfl_sync(FULL, cellp, l);
              const int ih = __shfl_sync(FULL, ihi, l), jh = __shfl_sync(FULL, jhi, l);
              if (ih >= p.R[s] - 1 && jh >= p.R[s] - 1) emit_row<MapT, false, false>(p, sb32, dst, cp, s, rr, rowctr, lane);
              else emit_row_masked<MapT>(p, sb32, dst, cp, s, ih, jh, lane);
            }
          }
        }
      }
      env_rows_done<SPLIT>(p, L, sbase, env, mode, keep, old_base, n, births, new_base, next_live, lane);
      // leave the maps empty for the next env of this warp: every loaded or born slot un-writes its cell in its channel
      #pragma unroll 1
      for (int i = lane; i < n[0] + births[0]; i += 32) S.map[0][CELLP((unsigned)S.pos[0][i])] = 0;
      #pragma unroll 1
      for (int i = lane; i < n[1] + births[1]; i += 32) prey_map(i)[CELLP((unsigned)S.pos[1][i])] = 0;
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
      if (over) h.state = p.autoreset ? ST_NEEDS_RESET : ST_IDLE;
      if (lane == 0) { p.hdr[env] = h; p.shdr[env] = sh; }
      add_stats(p, env, mode, n, births, over, trunc, h.step, st, lane);
    } else {
      env_idle<SPLIT>(p, sbase, env, old_base, lane);
    }
    env_end<SPLIT>(p, L, env, mode, n, births, env_flags, h, t_env0, t_ns0, live, mode != 0, lane);  // an idle env keeps the counts of its last step
  }
  if (SPLIT) queue_push(p, L.pend, L.pend_env, lane);
}

// reals cursor of the replay tape
__global__ void ppg_set_tape_reals_stag_kernel(StagHdr* shdr, int B, const long long* real_off) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  shdr[e].real_pos = real_off ? real_off[e] : 0;
  shdr[e].real_end = real_off ? real_off[e + 1] : 0;
}

// uniform random actions for the rows of the last output: predators MultiDiscrete([n_moves, 2]) packed as
// move | join << 8, prey Discrete(n_moves) (STAG:1802-1816); the move range follows the agent's type
__global__ void ppg_random_actions_stag_kernel(const int32_t* __restrict__ n_rows, const int32_t* __restrict__ row_env0,
                                               const int32_t* __restrict__ row_agent0, const int32_t* __restrict__ row_env1,
                                               const int32_t* __restrict__ row_agent1, int32_t* act0, int32_t* act1,
                                               unsigned long long seed, unsigned call, unsigned env_base, int t2_pred, int t2_prey,
                                               int ar0, int ar1) {
  allow_dependent_launch();       // PDL chain (see ppg_random_actions_kernel)
  wait_for_stream_predecessor();
  // read through a volatile pointer: as a plain load from a `const __restrict__` pointer the compiler hoisted n_rows[0] ABOVE
  // griddepcontrol.wait (SASS: LDG.E.CONSTANT before ACQBULK), i.e. the row count of the step before was read while that
  // step's kernels were still running — with the launch chain on and several steps queued the actions then covered the wrong
  // number of rows (tests/test_gpu_rollout.py)
  const volatile int32_t* const nr = n_rows;
  const int n0 = nr[0] + nr[2], n1 = nr[1] + nr[3];
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n0 + n1; i += gridDim.x * blockDim.x) {
    const int s = i >= n0;
    const int row = s ? i - n0 : i;
    const unsigned env = (unsigned)(s ? row_env1[row] : row_env0[row]) + env_base;
    const unsigned id = (unsigned)(s ? row_agent1[row] : row_agent0[row]);
    const unsigned r = ppg_draw_u32(seed, env, call, PPG_STREAM_ACTION + 8u * (unsigned)s, id);
    const int R = ((int)id >= (s ? t2_prey : t2_pred)) ? ar1 : ar0;
    const unsigned mv = ppg_bounded(r, (unsigned)(R > 0 ? R * R : 1));
    const unsigned jn = s == 0 ? (ppg_draw_u32(seed, env, call, PPG_STREAM_ACTION + 16u, id) & 1u) : 0u;
    (s ? act1 : act0)[row] = (int32_t)(mv | (jn << PPG_STAG_JOIN_SHIFT));
  }
}

template <typename MapT>
static StepKernel stag_kernel(const StepParams& p) {
  return {p.obs_split ? ppg_step_stag_kernel<1, MapT, true> : ppg_step_stag_kernel<1, MapT, false>, 32};
}

StepKernel step_kernel_stag(const StepParams& p) {
  return p.map_bytes == 1 ? stag_kernel<uint8_t>(p) : stag_kernel<uint16_t>(p);
}

cudaError_t launch_set_tape_reals_stag(StagHdr* shdr, int B, const long long* real_off, cudaStream_t s) {
  ppg_set_tape_reals_stag_kernel<<<(B + 255) / 256, 256, 0, s>>>(shdr, B, real_off);
  return cudaGetLastError();
}

cudaError_t launch_random_actions_stag(const int32_t* n_rows, const int32_t* re0, const int32_t* ra0, const int32_t* re1, const int32_t* ra1,
                                       int32_t* a0, int32_t* a1, unsigned long long seed, unsigned call, unsigned env_base, int t2_pred,
                                       int t2_prey, int ar0, int ar1, int blocks, cudaStream_t s) {
  return pdl_launch(ppg_random_actions_stag_kernel, dim3((unsigned)blocks), dim3(256), 0, s, n_rows, re0, ra0, re1, ra1, a0, a1, seed, call, env_base, t2_pred,
                    t2_prey, ar0, ar1);
}

}  // namespace ppg
