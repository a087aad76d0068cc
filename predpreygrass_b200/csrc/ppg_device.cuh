// ppg_device.cuh — device-side data layout shared by the kernels and the C-ABI host code.
//
// Data layout in HBM (one handle = B env instances on one GPU), structure of arrays:
//   per env          EnvHdr (64 B): step counter, list lengths, id counters, RNG/tape cursors, flags
//   per env, species ag_id u16[cap], ag_pos u16[cap] (x<<8|y), ag_energy f64[cap], ag_prow i32[cap]
//                    (+ ag_parent u16[cap], kickback reward only) — a COMPACT list in the reference's
//                    `self.agents` order (BASE:73,468): position in the list = iteration order
//   per env          gr_pos u16[n_grass], gr_energy f64[n_grass]
//   per env          counters u32[16] (PPG_STAT_*)
// The float64 grid of the reference (`grid_world_state`, BASE:124) is NOT stored, neither in HBM nor
// in shared memory: a non-zero cell of the reference grid always holds the current energy of the
// agent that wrote it last, so the kernels keep per-species OWNER maps (cell -> list slot + 1) in
// shared memory and look the value up (see DESIGN.md "owner maps").
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdlib>
#include <utility>

#include "../../include/ppg.h"
#include "../../include/ppg_philox.h"
#include "../../include/ppg_pow.h"

namespace ppg {

#define PPG_MAX_NJ 13  // observation rows of up to 416 floats

struct __align__(16) EnvHdr {
  unsigned long long seed_key;  // Philox key of this env (ppg_reset seeds)
  long long tape_pos, tape_end; // replay-tape cursor into tape_cells
  int step;                     // current_step (BASE:134,471)
  unsigned episode;             // Philox counter word
  unsigned spawn_draws;         // Philox draw index of the spawn-fallback stream
  unsigned short n_list[2];     // live agents per species = list length
  unsigned short next_idx[2];   // _next_predator_idx / _next_prey_idx (BASE:66-67)
  unsigned char state;          // ST_*
  unsigned char status;         // PPG_STATUS_* (sticky until reset)
  unsigned char sortflag;       // bit s: list of species s is not in lexicographic order yet
  unsigned char first_step;     // 1 right after reset(): engagement order is the founders' numeric order
  unsigned short n_sorted[2];   // length of the lexicographically sorted prefix of the list (rest: last step's newborns)
  int pad[2];
};
static_assert(sizeof(EnvHdr) == 64, "EnvHdr must be 64 bytes");

enum : unsigned char { ST_NEEDS_RESET = 1, ST_IDLE = 2 };

// ECO only: second per-env header (32 B)
struct __align__(16) EcoHdr {
  long long real_pos, real_end;  // replay-tape cursor into tape_reals
  int active[2];                 // active_num_predators / active_num_prey (ECO:212-213); the reference lets them drift
  unsigned trait_draws;          // Philox counter of the trait stream
  unsigned next_seq;             // insertion index of the next newborn in self.agents / agent_positions
};
static_assert(sizeof(EcoHdr) == 32, "EcoHdr must be 32 bytes");

// STAG only: second per-env header (112 B)
struct __align__(16) StagHdr {
  long long real_pos, real_end;  // replay-tape cursor into tape_reals
  double capture_real[3];        // last_success_prob, last_effort_ratio, success_prob_sum (STAG:249-251)
  unsigned capture[12];          // team-capture counters in the order of ppg_read_env_stag (STAG:237-254)
  unsigned trait_draws, facing_draws, capture_draws;  // Philox counters of the trait / facing / capture streams
  unsigned short next_idx_t[2][2];                     // head of the per-type id deques (STAG:2259-2291)
  unsigned pad;
};
static_assert(sizeof(StagHdr) == 112, "StagHdr must be 112 bytes");

// per-slot flag bits, shared memory only
enum : unsigned char {
  F_ALIVE = 1,    // in agent_positions
  F_DIED = 2,     // terminated this step
  F_ATE = 4,      // agents_just_ate
  F_REPRO = 8,    // reproduced this step
  F_NEWBORN = 16, // born this step
  F_CAUGHT = 32,  // died by being eaten (reward differs from starvation)
  F_CARC = 64,    // ECO: member of dead_prey (bitten, not fully eaten)
  F_BORNROW = 128 // ECO: the newborn's row was written at birth (kept if the episode ends on this step, ECO:417-420)
};

// header of an env image (ints)
enum { IH_OLD_BASE0 = 0, IH_OLD_BASE1, IH_N0, IH_N1, IH_BIRTHS0, IH_BIRTHS1, IH_MODE, IH_KEEP, IH_INTS = 16 };
#define DSC_SKIP 0xFFFFu  // the row was written by the step kernel (captured at the moment of death / birth)
#define DSC_ZERO 0xFFFEu  // STAG: ended agents are observed as all-zero rows
#define DSC_COPY 0xFFFDu  // ECO: the row was captured at birth into born_obs[env][dsx] (episode ended on this step, ECO:417-420)
#define PPG_EP_STRIDE 12            // doubles per env in StepParams::ep_sums
#define PPG_EP_BLOCKED_CAPACITY 4   // [2] births skipped because the id pool was exhausted (MR:857,943)
#define PPG_EP_BLOCKED_DENSITY 6    // predator births skipped by the density cap (MR:852)
#define PPG_EP_SATIATION_BLOCKED 7  // catches skipped while digesting (MR:739)
#define PPG_EP_DONATED 8            // [2] energy donated = received per species (COOP:585-586)
#define PPG_BORN_K 4      // at-birth rows kept per env and species; further ones take the (blocking) direct path
#define PPG_MAX_GHOSTS 16 // ECO: stale prey-channel cells carried per env (ppg_eco.cu header); more raise PPG_STATUS_GHOST_CELL

// trait variants whose number of founders is drawn per episode (MR:189-192); cadence and ECO have a fixed number
__host__ __device__ inline bool ppg_random_founders(int trait_mode) {
  return trait_mode == PPG_TRAIT_METABOLIC || trait_mode == PPG_TRAIT_INVESTMENT || trait_mode == PPG_TRAIT_COOPERATION;
}

struct StepParams {
  // ---- config ----
  int B, G, GG, C;
  int env_base;           // ppg_config.env_index_base
  int R[2], off[2], elems[2];
  int cap[2], n_init[2], n_possible[2], n_grass, max_steps, reward_mode, autoreset;
  double loss[2], thr[2], init_e[2], grass_cap, grass_gain, init_e_grass;
  double grass_gain_season[2];  // BASE family, seasonal regrowth: grass_gain * season multiplier (high, low); season_len = 0: none
  int season_len;
  double r_catch, r_eat, r_pstep, r_qstep, pen_caught, r_repro[2], r_kick[2];
  // ---- state ----
  EnvHdr* hdr;
  uint16_t* ag_id[2];
  uint16_t* ag_pos[2];
  double* ag_e[2];
  int32_t* ag_prow[2];
  uint16_t* ag_par[2];
  uint16_t* gr_pos;
  double* gr_e;
  const uint16_t* lexrank[2];
  const int32_t* tape_cells;
  uint32_t* counters;  // [B][PPG_N_STATS]
  // ---- dynamic env scheduling + deterministic row allocation (hierarchical counts, see ppg_base.cu) ----
  unsigned long long* ticket;      // env ticket counter (monotonic over launches)
  unsigned long long ticket_base;  // value of *ticket at launch
  int static_first;                // 1: a warp's first env is ticket blockIdx.x (no atomic), the counter hands out tickets >= min(grid, B);
                                   // only where no env ever waits for another one (BASE / STAG two-kernel step)
  unsigned epoch;                  // launch number (1-based); tags every published word
  unsigned* error;                 // device error word (bit0: prefix wait wedged)
  // published per env / per 32-env block / per 1024-env group, ping-pong by epoch parity:
  //   cntA = epoch<<32 | live_pred<<16 | live_prey   (rows the env needs in the NEXT output)
  //   cntB = epoch<<32 | births_pred<<16 | births_prey (newborn rows of THIS output)
  //   sum1/sum2 [.][4] = epoch<<32 | sum of {live_pred, live_prey, births_pred, births_prey}
  unsigned long long* cntA[2];
  unsigned long long* cntB[2];
  unsigned long long* sum1[2];
  unsigned long long* sum2[2];
  // accumulators of the publication (ppg_step_common.cuh): contributors << 56 | first sum << 28 | second sum, [.][0] the
  // live counts, [.][1] the births; cleared by the last contributor of every launch
  unsigned long long* acc1;  // [n_blk][2] per 32-env block
  unsigned long long* acc2;  // [n_grp][2] per 1024-env group
  unsigned long long* acc3;  // [2]
  int32_t* totals;   // [2][4] per parity: total {live_pred, live_prey, births_pred, births_prey}
  int32_t* perm[2];  // [B] per parity: env order of the next launch, big envs first (publish_begin); nullptr: index order
  unsigned* perm_tag;  // [2] epoch that wrote perm[par] (anything else: index order)
  unsigned* perm_cursor;  // [2][2] per parity: entries taken from the front (big envs) / from the back
  const int32_t* order[2];  // optional: rank of each row inside its env+species in the action dict (ppg_step_ordered)
  // ---- io ----
  const int32_t* actions[2];
  float* obs[2];
  int32_t* row_env[2];
  int32_t* row_agent[2];
  float* reward[2];
  uint8_t* flags[2];
  int32_t* old_off[2];
  int32_t* new_off[2];
  int32_t* new_cnt[2];
  int32_t* n_rows;
  uint8_t* env_flags;
  uint8_t* env_status;
  int32_t* env_step;
  int32_t* env_count;
  // ---- shared-memory layout, byte offsets inside one env's region ----
  int so_E[2], so_E0[2], so_gE, so_wt, so_vt[3], so_stage, so_scr, so_id[2], so_pos[2], so_ord[2], so_rnk[2], so_par[2];
  int so_map[4], so_gpos, so_act[2], so_flg[2], so_aux[2], so_gtag;
  int stage_elems;  // floats per staging row buffer (max over species, multiple of 4)
  int smem_per_env;
  // ---- padded map geometry and the observation gather tables (see ppg_base.cu) ----
  int P, PS, CH;        // halo width, row stride, entries per map:  index(x, y) = P + (x + P) * PS + y
  int map_bytes;        // sizeof(map entry): 1 (all capacities <= 253) or 2
  int wall_idx;         // value the predator map holds outside the field (index of the 1.0 entry of the wall table)
  int nj[2];            // per-lane elements of a row per species (see obs_vec)
  int obs_vec[2];       // 1: lane owns float4 groups (row length % 4 == 0, nj = 4 * ceil(elems / 128)); 0: lane owns
                        //    elements lane + 32 j (nj = ceil(elems / 32))
  int emit_kind[2];     // specialised row writer: 1 = (4,7,7), 2 = (4,9,9), 3 = (5,9,9), 4 = (3,7,7), 5 = (3,9,9), 0 = generic
  int obs_bulk;         // 1: rows leave through shared-memory staging + cp.async.bulk; 0: direct streaming stores
  const void* init_image;  // [init_bytes] initial contents of the maps / touch counters / wall table of a warp's slice
  int init_bytes;
  // ---- ECO (ppg_eco.cu) ----
  int variant, action_range, n_actions, genome_enabled, speed_in_obs, max_age[2], carcass_age, slow_dist, fast_dist;
  double move_cost[2], move_exp, bite_cap_grass, bite_cap_prey, f_mean[2], f_std[2], mut_rate, mut_std, sp_lo, sp_hi, sp_thr;
  EcoHdr* ehdr;
  uint16_t* ag_age[2];
  uint16_t* ag_seq[2];
  double* ag_spd[2];
  uint8_t* ag_dead[2];
  // trait variants of ECO (ppg_config.trait_mode): founders ~ U{n_init_min..n_init}, satiation cooldown, meal-sharing radius,
  // gain exponent, density cap (< 0: none)
  int trait_mode, n_init_min[2], sat_cd, coop_range;
  double trait_alpha, repro_ratio;
  // STAG walls (static cells of channel 0, STAG:2107-2160) and line-of-sight test of prey moves (STAG:875-925)
  const int32_t* wall_cells;  // [n_walls] x * G + y
  int n_walls, los_move;
  // ECO lineage survival rewards (ECO:943-984,1422-1470), by agent id: parent id (0xFFFF: founder), live descendants,
  // their count at the previous step, own alive flag; lin_on = any coefficient non-zero
  int lin_on;
  double lin_coeff[2];
  uint16_t* lin_parent[2];  // [B][n_possible[s]]
  int16_t* lin_live[2];
  int16_t* lin_prev[2];
  uint8_t* lin_alive[2];
  // cadence variant: move accumulators (CAD:183-186), slowest cadence, speed-dependent basal cost
  int max_cooldown, so_acc[2];
  double meta_coeff;
  double* ag_acc[2];
  double* ep_sums;     // [B][PPG_EP_STRIDE] optional (ppg_config.track_episode_sums): per-episode distance moved [2], locomotion energy [2],
                       // then the trait variants' event counters at PPG_EP_BLOCKED_CAPACITY ... (ppg_read_episode_events_eco)
  uint8_t* gh_n;       // [B] ghost cells of the env (ppg_eco.cu header)
  uint16_t* gh_cell;   // [B][PPG_MAX_GHOSTS] packed position x << 8 | y
  float* gh_val;       // [B][PPG_MAX_GHOSTS] the stale float32 grid value
  const double* tape_reals;
  int so_spd[2], so_age[2], so_seq[2], so_mord[2];
  const unsigned* obs_self;  // [2][32] per-lane bit mask: element j of the lane lies in the agent's own-speed plane (ECO:707-711)
  // ---- STAG (ppg_stag.cu); ag_age / so_age / so_mord above are shared with ECO ----
  int n_possible_t[2][2], n_init_t[2][2], type_ar[2];
  int equal_split, coop_enabled, capture_model, strict_out;
  int PH;  // high-side halo of the padded maps (forward view: the predator window centre lies up to `off` cells outside)
  double loss_prey_t[2], thr_prey_t[2], init_e_prey_t[2], bite_t[2], r_repro_t[2][2], death_pen[3];
  double cap_margin, join_cost, scav_frac, nature_w, p0, force_ratio, min_prob, trait_mean, trait_std, trait_mut_std, trait_mut_rate;
  StagHdr* shdr;
  uint8_t* ag_face;   // [B][cap0] predator facing, index into _predator_facing_options (STAG:197-206)
  double* ag_trait;   // [B][cap0] predator_cooperation_trait (STAG:230)
  int so_trait, so_face, so_join;
  // ---- two-kernel step (ppg_obs.cu): the step kernel leaves, per env, an IMAGE of what the observation writer needs ----
  //   image = [16-int header][value tables][padded maps][wall table][row descriptors]: one contiguous range of the env's
  //   shared-memory slice [so_img, so_img + img_bytes), dumped to obs_img + env * img_stride and fetched back by the
  //   observation kernel with one bulk asynchronous copy (TMA engine) per env
  int obs_split;            // 1: rows are written by ppg_obs_kernel after the step kernel; 0: by the step kernel itself
  int so_img, img_bytes, img_stride;
  int so_ihdr;              // header ints: IH_* below
  int so_dsc[2];            // u16 [cap]: padded cell index of the window centre of the k-th row of the env, or DSC_SKIP / DSC_ZERO
  int so_dsx[2];            // u32 [cap]: ECO own-speed plane value (float bits); STAG ihi | jhi << 8 (cut-off forward view)
  unsigned char* obs_img;   // [B][img_stride]
  unsigned long long* nb_info[2];  // [B][cap] per newborn of this launch: id | row flags << 16 | list position << 32 (0xFFFF: not kept)
  float* born_obs[2];       // ECO: [B][PPG_BORN_K][elems] at-birth observations of newborns of an episode's last step
  uint4* env_cycles;       // [B] profiling: x = SM cycles the step kernel spent on the env in the last launch, y = mode | births << 8 | agents << 16,
                           //     z = globaltimer (ns, low 32 bits) when the env was taken, w = SM id
  unsigned long long* queue;       // [B] completion queue of the step kernel: epoch << 32 | env, in the order the images reached HBM
  unsigned long long* q_tail;      // entries pushed so far (monotonic over launches); q_base = its value at launch
  unsigned long long q_base;
  unsigned long long* obs_ticket;  // env ticket counter of the observation kernel (monotonic over launches)
  unsigned long long obs_ticket_base;
  const int2* obs_rel;  // [2][PPG_MAX_NJ][32]: x = byte offset of the map entry relative to the agent's own entry in map 0..2
                        //                       (so_map[m] + rel * map_bytes), y = byte offset of the value table; x = INT_MAX: no element
};

// ppg_world_state (ppg_world.cu): grid channel c of env e is table_c[map_c[P + (x + P) * PS + y]] of the env's image.
// Channels >= PPG_WS_SRC share the source of channel PPG_WS_SRC - 1 (STAG's channels past grass: walls table, all zero).
#define PPG_WS_SRC 8
struct WorldStateParams {
  const unsigned char* img;  // StepParams::obs_img
  float* out;                // [n_envs][C][G][G]
  int env_begin, n_envs;
  int img_stride, img_bytes; // image pitch in HBM, bytes brought into shared memory (a multiple of 16)
  int G, C, P, PS;
  int map_off[PPG_WS_SRC];   // byte offset of channel c's owner map inside the image
  int tbl_off[PPG_WS_SRC];   // byte offset of channel c's fp32 value table inside the image
};

// ppg_returns_kernel (ppg_returns.cu): episode returns and agent lifetimes, updated from the rows of the last output
// (include/ppg.h ppg_track_returns).
struct ReturnsParams {
  const int32_t* row_agent[2];
  const float* reward[2];
  const uint8_t* flags[2];
  const int32_t* old_off[2];
  const int32_t* new_off[2];
  const int32_t* new_cnt[2];
  const uint8_t* env_flags;
  const int32_t* env_step;
  double* row_return[2];  // [row_capacity[s]]
  int32_t* row_life[2];
  double* tab_ret[2];     // [B][n_possible[s]]: return so far of the life of (env, id)
  int32_t* tab_life[2];   // [B][n_possible[s]]: rows so far of that life
  double* env_return;     // [B][2]
  uint8_t* env_valid;     // [B]
  double* env_acc;        // [B][PPG_N_EP_STATS]
  int n_possible[2];
  int B;
};

// ppg_agent_state_kernel (ppg_agent_state.cu): the state of the agent behind every row of the last output (include/ppg.h
// ppg_agent_state).  The host resolves each column's source list (nullptr: the column is not written).
struct AgentStateParams {
  ppg_agent_state_args a;
  const EnvHdr* hdr;
  const uint16_t* ag_id[2];
  const uint16_t* ag_pos[2];
  const double* ag_e[2];
  const int32_t* ag_prow[2];
  const uint16_t* ag_age[2];    // ECO family, STAG
  const double* ag_trait[2];    // ECO family: ag_spd[s]; STAG: ag_trait (predators)
  const uint8_t* ag_face;       // STAG predators
  const double* ag_acc[2];      // cadence variant
  const int32_t* row_agent[2];
  const int32_t* old_off[2];
  const int32_t* new_off[2];
  const int32_t* new_cnt[2];
  const uint8_t* env_flags;
  const uint16_t* gr_pos;
  const double* gr_e;
  int cap[2];
  int n_grass, B;
};

// ppg_gae_kernel (ppg_gae.cu): links the rows of a rollout and runs the GAE recursion (include/ppg.h ppg_gae).
struct GaeParams {
  ppg_gae_args a;
  long long cap[2];   // row_capacity[s]: pitch of the row slabs
  int n_possible[2];
  int B;
  int log2_h;         // link table: 1 << log2_h entries per warp and buffer
};

// Launch with programmatic stream serialization (PDL): the grid's CTAs may be scheduled as soon as every CTA of the kernel
// before it in the stream has executed griddepcontrol.launch_dependents (or exited), which hides the launch ramp of the 2960
// one-warp CTAs of a step kernel behind the tail of the observation kernel.  The kernel MUST execute griddepcontrol.wait before
// it reads or writes anything the predecessor touches.  PPG_PDL_CHAIN=0 / ppg_set_pdl_chain(0) turn the chain off (plain stream
// order): a grid waiting in griddepcontrol.wait holds its SM slots, which only hurts when OTHER streams have work for them
// (env groups on their own streams).
#ifdef __CUDACC__
extern int g_pdl_chain;  // ppg_api.cu: -1 = not read yet, 0 = off, 1 = on (ppg_set_pdl_chain)
inline bool pdl_chain_enabled() {
  // OFF by default (include/ppg.h ppg_set_pdl_chain): tests/test_gpu_rollout.py found at the end of round 2 that with the chain
  // on and several steps queued the action kernels read a stale row count (a load hoisted above griddepcontrol.wait); that is
  // fixed and tested, but everything measured in the round after the finding ran with the chain off.
  if (g_pdl_chain < 0) { const char* ev = getenv("PPG_PDL_CHAIN"); g_pdl_chain = ev ? (atoi(ev) != 0) : 0; }
  return g_pdl_chain != 0;
}
template <typename... KArgs, typename... Args>
static inline cudaError_t pdl_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_chain_enabled() ? 1 : 0;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
#endif

}  // namespace ppg
