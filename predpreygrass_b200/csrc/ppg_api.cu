// ppg_api.cu — the C-ABI of include/ppg.h over the CUDA kernels (host side, no torch).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "ppg_device.cuh"

namespace ppg {
cudaError_t launch_step_base(const StepParams& p, int warps_per_cta, int n_cta, size_t smem, cudaStream_t stream);
cudaError_t step_base_occupancy(int warps_per_cta, int map_bytes, bool bulk, bool split, size_t smem, int* blocks_per_sm);
cudaError_t launch_prepare_offsets(const EnvHdr* hdr, int B, int n0, int n1, unsigned long long* cntA, unsigned long long* sum1,
                                   unsigned long long* sum2, int32_t* totals4, unsigned epoch, int hdr_founders, cudaStream_t s);
cudaError_t launch_init_hdr(EnvHdr* hdr, int B, unsigned long long seed, cudaStream_t s);
cudaError_t launch_relabel_rows(const StepParams& p, const unsigned long long* cntA, const unsigned long long* sum1,
                                const unsigned long long* sum2, const int32_t* totals4, cudaStream_t s);
cudaError_t launch_mark_reset(EnvHdr* hdr, int B, const unsigned long long* seeds, const uint8_t* mask, cudaStream_t s);
cudaError_t launch_set_tape(EnvHdr* hdr, int B, const long long* cell_off, cudaStream_t s);
cudaError_t launch_random_actions(const int32_t* n_rows, const int32_t* re0, const int32_t* ra0, const int32_t* re1,
                                  const int32_t* ra1, int32_t* a0, int32_t* a1, unsigned long long seed, unsigned call,
                                  unsigned n_actions, unsigned env_base, int blocks, cudaStream_t s);
cudaError_t launch_stats(const uint32_t* counters, const EnvHdr* hdr, int B, unsigned long long* out, cudaStream_t s);
// ppg_obs.cu
cudaError_t launch_obs(const StepParams& p, int n_cta, bool overlap, cudaStream_t stream);
cudaError_t obs_occupancy(const StepParams& p, int* blocks_per_sm);
// ppg_eco.cu
cudaError_t launch_step_eco(const StepParams& p, int n_cta, size_t smem, cudaStream_t stream);
cudaError_t step_eco_occupancy(int map_bytes, bool split, int kind, size_t smem, int* blocks_per_sm);
cudaError_t launch_set_tape_reals(EcoHdr* ehdr, int B, const long long* real_off, cudaStream_t s);
cudaError_t launch_eco_founders(const StepParams& p, cudaStream_t s);
// ppg_stag.cu
cudaError_t launch_step_stag(const StepParams& p, int n_cta, size_t smem, cudaStream_t stream);
cudaError_t step_stag_occupancy(int map_bytes, bool split, size_t smem, int* blocks_per_sm);
cudaError_t launch_set_tape_reals_stag(StagHdr* shdr, int B, const long long* real_off, cudaStream_t s);
cudaError_t launch_random_actions_stag(const int32_t* n_rows, const int32_t* re0, const int32_t* ra0, const int32_t* re1, const int32_t* ra1,
                                       int32_t* a0, int32_t* a1, unsigned long long seed, unsigned call, unsigned env_base, int t2_pred,
                                       int t2_prey, int ar0, int ar1, int blocks, cudaStream_t s);
// ppg_world.cu
cudaError_t launch_world_state(const WorldStateParams& p, int map_bytes, int n_cta, cudaStream_t stream);
cudaError_t world_state_occupancy(const WorldStateParams& p, int map_bytes, int* blocks_per_sm);
// ppg_returns.cu
cudaError_t launch_returns(const ReturnsParams& p, cudaStream_t stream);
int episode_stats_partials(int B);
cudaError_t launch_episode_stats(const double* env_acc, const uint8_t* env_valid, int B, double* partial, double* out, cudaStream_t stream);
cudaError_t launch_episode_stats_clear(double* env_acc, int B, cudaStream_t stream);
}  // namespace ppg

namespace ppg { int g_pdl_chain = -1; }

using namespace ppg;

// include/ppg_pow.h on the device, argument by argument (ppg_selftest_pow)
__global__ void ppg_pow_selftest_kernel(const double* __restrict__ x, const double* __restrict__ y, double* __restrict__ out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) out[i] = ppg_pow(x[i], y[i]);
}

struct ppg_handle_s {
  ppg_config cfg;
  int B = 0, device = 0;
  StepParams P;
  std::vector<int32_t> walls;  // copy of ppg_config.wall_cells
  int warps_per_cta = 4, n_cta = 0;
  size_t smem_bytes = 0;
  unsigned long long launches_step = 0;  // step-kernel launches so far (epoch)
  unsigned long long ticket_next = 0;    // value the device ticket counter has after all launches so far
  unsigned long long obs_ticket_next = 0;  // same for the observation kernel's counter
  int n_cta_obs = 0;
  bool obs_overlap = true;               // observation kernel launched with programmatic stream serialization
  unsigned long long q_next = 0;         // value the completion-queue tail has after all launches so far
  bool profiling = false;
  std::vector<cudaEvent_t> prof_events;  // triples: before the step kernel, between the kernels, after the observation kernel
  unsigned long long calls = 0;          // ppg_reset(all)/ppg_step calls (ppg_random_actions key)
  // do the env images in obs_img show the world of the last output (ppg_world_state)?
  enum { IMG_NONE, IMG_VALID, IMG_RESTORED, IMG_RESTORED_IDLE } img = IMG_NONE;
  int n_cta_ws = 0;                      // ppg_world_state grid (0: not computed yet)
  // episode returns (ppg_track_returns): allocated at the first switch-on
  bool track_on = false;
  ReturnsParams R;
  bool R_alloc = false;
  double* d_ep_partial = nullptr;        // ppg_episode_stats_device scratch and result
  double* d_ep_stats = nullptr;
  int64_t launch_count = 0;
  std::vector<void*> allocs;
  unsigned long long* d_stats = nullptr;
  int32_t* d_tape_cells = nullptr;
  long long* d_tape_off = nullptr;
  double* d_tape_reals = nullptr;
  long long* d_tape_real_off = nullptr;
  uint8_t* d_mask = nullptr;
  unsigned long long* d_seeds = nullptr;
  int32_t* d_act[2] = {nullptr, nullptr};  // staging for ppg_step_host
  int32_t h_n_rows[4] = {0, 0, 0, 0};
  bool h_n_rows_valid = false;
  ppg_buffers bufs;
  size_t state_bytes = 0;
  std::string err;
};

static thread_local std::string g_err;

#define CK(call)                                                                             \
  do {                                                                                       \
    cudaError_t _e = (call);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      h->err = std::string(#call) + ": " + cudaGetErrorString(_e);                           \
      return PPG_ERR_CUDA;                                                                   \
    }                                                                                        \
  } while (0)

template <typename T>
static cudaError_t dalloc(ppg_handle h, T** p, size_t n) {
  void* q = nullptr;
  cudaError_t e = cudaMalloc(&q, std::max<size_t>(n, 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  e = cudaMemset(q, 0, std::max<size_t>(n, 1) * sizeof(T));
  h->allocs.push_back(q);
  *p = static_cast<T*>(q);
  return e;
}

// Which owner map and which value table show grid channel `ch` (so_* offsets): the observation rows (obs_rel) and
// ppg_world_state both take their sources from here.
//   BASE: 0 walls (predator map: its halo holds the wall entry of the wall table), 1 predators, 2 prey, 3 grass
//   ECO:  0 predators, 1 prey, 2 grass (channel 3, the own-speed plane, is not a gather)
//   STAG (STAG:112-117): 0 walls (wall cells are wall entries of the predator map), 1 predators, 2 mammoths, 3 rabbits,
//         4 grass; further channels read the wall table through the predator map (all zero off the walls)
struct ChannelSource { int map, tbl; };
static ChannelSource channel_source(const StepParams& P, int ch) {
  if (P.variant == PPG_VARIANT_STAG) {
    static const int map_of[5] = {0, 0, 1, 3, 2};
    return {P.so_map[ch < 5 ? map_of[ch] : 0], ch == 1 ? P.so_vt[0] : (ch == 2 || ch == 3) ? P.so_vt[1] : ch == 4 ? P.so_vt[2] : P.so_wt};
  }
  if (P.variant == PPG_VARIANT_ECO) return {P.so_map[ch], P.so_vt[ch]};
  return {P.so_map[ch == 0 ? 0 : ch - 1], ch == 0 ? P.so_wt : P.so_vt[ch - 1]};
}

static int str_cmp_ids(const void* a, const void* b) {
  char sa[16], sb[16];
  snprintf(sa, sizeof sa, "%d", *(const int*)a);
  snprintf(sb, sizeof sb, "%d", *(const int*)b);
  return strcmp(sa, sb);
}

// rank of str(id) among the species' id strings: the order Python's list.sort() gives (BASE:468)
static std::vector<uint16_t> lexrank_table(int n) {
  std::vector<int> ids(n);
  for (int i = 0; i < n; ++i) ids[i] = i;
  qsort(ids.data(), (size_t)n, sizeof(int), str_cmp_ids);
  std::vector<uint16_t> r(std::max(n, 1));
  for (int i = 0; i < n; ++i) r[ids[i]] = (uint16_t)i;
  return r;
}

extern "C" {

int ppg_abi_version(void) { return PPG_ABI_VERSION; }

void ppg_default_config(ppg_config* c) {
  memset(c, 0, sizeof *c);
  c->struct_size = sizeof *c;
  c->variant = PPG_VARIANT_BASE;
  c->reward_mode = PPG_REWARD_SPARSE;
  c->grid_size = 25; c->max_steps = 1000; c->num_obs_channels = 4;
  c->obs_range[0] = 7; c->obs_range[1] = 9;
  c->n_possible[0] = 2000; c->n_possible[1] = 2000;
  c->n_initial[0] = 6; c->n_initial[1] = 8;
  c->n_grass = 100;
  c->cap_live[0] = 64; c->cap_live[1] = 192;
  c->autoreset = 1;
  c->energy_loss[0] = 0.15; c->energy_loss[1] = 0.05;
  c->creation_threshold[0] = 12.0; c->creation_threshold[1] = 8.0;
  c->initial_energy[0] = 5.0; c->initial_energy[1] = 3.0;
  c->initial_energy_grass = 2.0; c->energy_gain_grass = 0.04;
  c->reproduction_reward[0] = 10.0; c->reproduction_reward[1] = 10.0;
  c->kickback_reward[0] = 10.0; c->kickback_reward[1] = 10.0;
  c->seed = 0;
  // ECO fields: neutral values for the BASE family (config.make_config fills the same)
  c->action_range = 3;
  c->max_agent_age[0] = c->max_agent_age[1] = -1;
  c->carcass_only_predator_age = -1;
  c->slow_max_move_distance = c->fast_max_move_distance = 1;
  c->move_speed_cost_exponent = 2.0;
  c->max_energy_grass = c->initial_energy_grass;
  c->max_energy_gain_per_grass = c->max_energy_gain_per_prey = HUGE_VAL;
  c->speed_bounds[0] = 0.5; c->speed_bounds[1] = 2.0;
  c->speed_distance_threshold = 1.5;
  c->season_multiplier[0] = c->season_multiplier[1] = 1.0;  // season_length_steps = 0: no seasons
  // trait-variant fields: neutral values (trait_mode = PPG_TRAIT_SPEED)
  c->n_initial_min[0] = c->n_initial[0]; c->n_initial_min[1] = c->n_initial[1];
  c->trait_alpha = 1.0; c->repro_max_ratio = -1.0;
}

const char* ppg_last_error(ppg_handle h) { return h ? h->err.c_str() : g_err.c_str(); }

static int validate(const ppg_config* c, int32_t n_envs, std::string& err) {
  if (!c || c->struct_size != sizeof(ppg_config)) { err = "ppg_config.struct_size mismatch"; return PPG_ERR_INVALID; }
  if (n_envs <= 0) { err = "n_envs must be positive"; return PPG_ERR_INVALID; }
  if (n_envs > 255 * 1024) { err = "n_envs must be <= 261120 per handle (contributor field of the row-allocation accumulators)"; return PPG_ERR_INVALID; }
  if (c->variant != PPG_VARIANT_BASE && c->variant != PPG_VARIANT_ECO && c->variant != PPG_VARIANT_STAG) { err = "unknown variant"; return PPG_ERR_INVALID; }
  const bool eco = c->variant == PPG_VARIANT_ECO, stag = c->variant == PPG_VARIANT_STAG;
  if (c->reward_mode < 0 || c->reward_mode > PPG_REWARD_SPARSE_KICKBACK) { err = "bad reward_mode"; return PPG_ERR_INVALID; }
  if (c->grid_size < 2 || c->grid_size > 255) { err = "grid_size must be in [2,255]"; return PPG_ERR_INVALID; }
  if (c->season_length_steps < 0 || (c->season_length_steps > 0 && (eco || stag))) { err = "season_length_steps: seasons exist in the BASE family only, >= 0"; return PPG_ERR_INVALID; }
  if (!eco && !stag && c->num_obs_channels != 4) { err = "BASE needs num_obs_channels == 4"; return PPG_ERR_INVALID; }
  if (stag) {
    if (c->num_obs_channels < 5) { err = "STAG needs num_obs_channels >= 5 (walls, predators, mammoths, rabbits, grass)"; return PPG_ERR_INVALID; }
    if (c->reward_mode != PPG_REWARD_SPARSE) { err = "STAG has one reward mode"; return PPG_ERR_INVALID; }
    if (c->max_steps > 65000) { err = "STAG: max_steps must be <= 65000 (16-bit ages)"; return PPG_ERR_INVALID; }
    if (c->cap_live[0] > 32767 || c->cap_live[1] > 32767) { err = "STAG: cap_live must be <= 32767"; return PPG_ERR_INVALID; }
    for (int s = 0; s < 2; ++s) {
      if (c->n_possible_t[s][0] < 0 || c->n_possible_t[s][1] < 0 || c->n_possible_t[s][0] + c->n_possible_t[s][1] != c->n_possible[s]) { err = "STAG: n_possible must be the sum over both types"; return PPG_ERR_INVALID; }
      if (c->n_initial_t[s][0] < 0 || c->n_initial_t[s][1] < 0 || c->n_initial_t[s][0] + c->n_initial_t[s][1] != c->n_initial[s]) { err = "STAG: n_initial must be the sum over both types"; return PPG_ERR_INVALID; }
      if (c->n_initial_t[s][0] > c->n_possible_t[s][0] || c->n_initial_t[s][1] > c->n_possible_t[s][1]) { err = "STAG: more founders than possible agents of a type"; return PPG_ERR_INVALID; }
      if (c->type_action_range[s] < 0 || c->type_action_range[s] > 15 || (c->type_action_range[s] > 0 && (c->type_action_range[s] & 1) == 0)) { err = "STAG: type action range must be odd, <= 15"; return PPG_ERR_INVALID; }
    }
    if (c->team_capture_success_model < 0 || c->team_capture_success_model > PPG_CAPTURE_HYBRID) { err = "bad team_capture_success_model"; return PPG_ERR_INVALID; }
    if (!(c->team_capture_base_success_p0 > 0.0 && c->team_capture_base_success_p0 < 1.0)) { err = "team_capture_base_success_p0 must lie in (0, 1)"; return PPG_ERR_INVALID; }
  }
  if (eco) {
    if (c->num_obs_channels != 3) { err = "ECO needs num_obs_channels == 3 (predators, prey, grass)"; return PPG_ERR_INVALID; }
    if (c->reward_mode != PPG_REWARD_SPARSE) { err = "ECO has one reward mode"; return PPG_ERR_INVALID; }
    if (c->action_range < 1 || (c->action_range & 1) == 0 || c->action_range > 15) { err = "action_range must be odd, <= 15"; return PPG_ERR_INVALID; }
    if (c->n_possible[0] + c->n_possible[1] > 65535) { err = "ECO: n_possible_predators + n_possible_prey must be <= 65535"; return PPG_ERR_INVALID; }
    if (c->max_steps > 65000) { err = "ECO: max_steps must be <= 65000 (16-bit ages)"; return PPG_ERR_INVALID; }
    if (c->cap_live[0] > 32767 || c->cap_live[1] > 32767) { err = "ECO: cap_live must be <= 32767"; return PPG_ERR_INVALID; }
    if (c->slow_max_move_distance < 0 || c->fast_max_move_distance < 0) { err = "max move distance negative"; return PPG_ERR_INVALID; }
    if (!(c->speed_bounds[1] > c->speed_bounds[0])) { err = "speed bounds"; return PPG_ERR_INVALID; }
    if (c->trait_mode < PPG_TRAIT_SPEED || c->trait_mode > PPG_TRAIT_CADENCE) { err = "trait_mode out of range"; return PPG_ERR_INVALID; }
    if (c->trait_mode != PPG_TRAIT_SPEED && (c->lineage_reward_coeff[0] != 0.0 || c->lineage_reward_coeff[1] != 0.0)) { err = "lineage rewards belong to eco_evolutionary (trait_mode speed)"; return PPG_ERR_INVALID; }
    if ((c->lineage_reward_coeff[0] != 0.0 || c->lineage_reward_coeff[1] != 0.0) && (c->cap_live[0] > 32767 || c->n_possible[0] > 65534 || c->n_possible[1] > 65534)) { err = "lineage rewards: n_possible must be <= 65534"; return PPG_ERR_INVALID; }
    if (c->trait_mode == PPG_TRAIT_CADENCE) {
      if (c->max_cooldown < 1) { err = "max_cooldown must be >= 1"; return PPG_ERR_INVALID; }
      if (c->carcass_only_predator_age >= 0) { err = "cadence has no carcass-only predators"; return PPG_ERR_INVALID; }
      if (c->n_initial_min[0] != c->n_initial[0] || c->n_initial_min[1] != c->n_initial[1]) { err = "cadence: the number of founders is fixed"; return PPG_ERR_INVALID; }
    } else if (c->trait_mode != PPG_TRAIT_SPEED) {
      for (int s = 0; s < 2; ++s)
        if (c->n_initial_min[s] < 0 || c->n_initial_min[s] > c->n_initial[s]) { err = "n_initial_min must lie in [0, n_initial]"; return PPG_ERR_INVALID; }
      if (c->satiation_cooldown < 0 || c->satiation_cooldown > 250) { err = "satiation_cooldown must be in [0, 250]"; return PPG_ERR_INVALID; }
      if (c->cooperation_range < 0) { err = "cooperation_range negative"; return PPG_ERR_INVALID; }
      if (c->include_speed_in_obs || c->max_agent_age[0] >= 0 || c->max_agent_age[1] >= 0 || c->carcass_only_predator_age >= 0) { err = "trait variants have no speed plane, age caps or carcass-only predators"; return PPG_ERR_INVALID; }
    }
  } else if (c->trait_mode != 0) { err = "trait_mode belongs to the ECO family"; return PPG_ERR_INVALID; }
  if (c->n_walls != 0 || c->respect_los_for_movement || c->include_visibility_channel) {
    if (!stag) { err = "walls / line of sight belong to the STAG variant"; return PPG_ERR_INVALID; }
    if (c->n_walls < 0 || (c->n_walls > 0 && !c->wall_cells)) { err = "wall_cells missing"; return PPG_ERR_INVALID; }
    for (int k = 0; k < c->n_walls; ++k)
      if (c->wall_cells[k] < 0 || c->wall_cells[k] >= c->grid_size * c->grid_size) { err = "wall cell out of the grid"; return PPG_ERR_INVALID; }
    if (c->n_walls + c->n_initial[0] + c->n_initial[1] + c->n_grass > c->grid_size * c->grid_size) { err = "walls leave too few cells for the reset placement"; return PPG_ERR_INVALID; }
    // the reference's visibility channel is a constant plane of ones (its masks are computed before any wall exists,
    // STAG:408-412); the dict adapter appends it on the host, the batched row layout does not carry it
    if (c->include_visibility_channel) { err = "include_visibility_channel: a constant plane of ones in the reference; appended by the dict adapter (PredPreyGrassStag), not part of the batched rows"; return PPG_ERR_INVALID; }
  }
  if (false) {
  }
  for (int s = 0; s < 2; ++s) {
    if (c->obs_range[s] < 1 || (c->obs_range[s] & 1) == 0 || c->obs_range[s] > 255) { err = "obs_range must be odd"; return PPG_ERR_INVALID; }
    if ((c->num_obs_channels + (eco && c->include_speed_in_obs ? 1 : 0)) * c->obs_range[s] * c->obs_range[s] > 4 * 128) { err = "observation row too large for this build"; return PPG_ERR_INVALID; }
    if (c->n_possible[s] < c->n_initial[s] || c->n_possible[s] > 65535) { err = "n_possible out of range"; return PPG_ERR_INVALID; }
    if (c->cap_live[s] < c->n_initial[s] || c->cap_live[s] <= 0 || c->cap_live[s] > 32768) { err = "cap_live out of range"; return PPG_ERR_INVALID; }
    if (c->n_initial[s] < 0) { err = "n_initial negative"; return PPG_ERR_INVALID; }
  }
  if (c->n_grass < 0 || c->n_grass > 254) { err = "n_grass must be in [0,254]"; return PPG_ERR_INVALID; }
  // "Cannot place more unique positions than grid cells." (BASE:167-168)
  if (c->n_initial[0] + c->n_initial[1] + c->n_grass > c->grid_size * c->grid_size) { err = "Cannot place more unique positions than grid cells."; return PPG_ERR_INVALID; }
  return PPG_OK;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int ppg_create(const ppg_config* cfg, int32_t n_envs, int32_t device, ppg_handle* out) {
  if (!out) return PPG_ERR_INVALID;
  *out = nullptr;
  int rc = validate(cfg, n_envs, g_err);
  if (rc) return rc;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { g_err = "no CUDA device"; return PPG_ERR_NO_DEVICE; }
  if (device < 0 || device >= ndev) { g_err = "bad device index"; return PPG_ERR_INVALID; }
  ppg_handle h = new ppg_handle_s();
  h->cfg = *cfg;
  h->walls.assign(cfg->wall_cells, cfg->wall_cells + (cfg->wall_cells ? cfg->n_walls : 0));  // the caller's list is copied
  h->cfg.wall_cells = h->walls.empty() ? nullptr : h->walls.data();
  h->B = n_envs;
  h->device = device;
  auto fail = [&](int code) { g_err = h->err; ppg_destroy(h); return code; };
#define CKC(call)                                                                            \
  do {                                                                                       \
    cudaError_t _e = (call);                                                                 \
    if (_e != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(_e); return fail(PPG_ERR_CUDA); } \
  } while (0)
  CKC(cudaSetDevice(device));
  const ppg_config& c = h->cfg;
  StepParams& P = h->P;
  memset(&P, 0, sizeof P);
  const int B = n_envs, G = c.grid_size, GG = G * G;
  const bool eco = c.variant == PPG_VARIANT_ECO, stag = c.variant == PPG_VARIANT_STAG;
  const int row_channels = c.num_obs_channels + (eco && c.include_speed_in_obs ? 1 : 0);
  P.B = B; P.G = G; P.GG = GG; P.C = row_channels; P.env_base = c.env_index_base;
  P.variant = c.variant;
  if (eco) {
    P.action_range = c.action_range; P.n_actions = c.action_range * c.action_range; P.genome_enabled = c.genome_enabled != 0;
    P.speed_in_obs = c.include_speed_in_obs != 0; P.max_age[0] = c.max_agent_age[0]; P.max_age[1] = c.max_agent_age[1];
    P.carcass_age = c.carcass_only_predator_age; P.slow_dist = c.slow_max_move_distance; P.fast_dist = c.fast_max_move_distance;
    P.move_cost[0] = c.move_cost_per_cell[0]; P.move_cost[1] = c.move_cost_per_cell[1]; P.move_exp = c.move_speed_cost_exponent;
    P.bite_cap_grass = c.max_energy_gain_per_grass; P.bite_cap_prey = c.max_energy_gain_per_prey;
    for (int s = 0; s < 2; ++s) { P.f_mean[s] = c.founder_speed_mean[s]; P.f_std[s] = c.founder_speed_std[s]; }
    P.mut_rate = c.mutation_rate; P.mut_std = c.mutation_std; P.sp_lo = c.speed_bounds[0]; P.sp_hi = c.speed_bounds[1];
    P.sp_thr = c.speed_distance_threshold;
    P.trait_mode = c.trait_mode; P.n_init_min[0] = c.n_initial_min[0]; P.n_init_min[1] = c.n_initial_min[1];
    P.sat_cd = c.satiation_cooldown; P.coop_range = c.cooperation_range; P.trait_alpha = c.trait_alpha; P.repro_ratio = c.repro_max_ratio;
    P.max_cooldown = c.max_cooldown; P.meta_coeff = c.metabolic_speed_coeff;
    P.lin_coeff[0] = c.lineage_reward_coeff[0]; P.lin_coeff[1] = c.lineage_reward_coeff[1];
    P.lin_on = c.trait_mode == PPG_TRAIT_SPEED && (P.lin_coeff[0] != 0.0 || P.lin_coeff[1] != 0.0);
  } else if (stag) {
    P.action_range = std::max(c.type_action_range[0], c.type_action_range[1]); P.n_actions = P.action_range * P.action_range;
    for (int s = 0; s < 2; ++s)
      for (int t = 0; t < 2; ++t) { P.n_possible_t[s][t] = c.n_possible_t[s][t]; P.n_init_t[s][t] = c.n_initial_t[s][t]; P.r_repro_t[s][t] = c.reproduction_reward_t[s][t]; }
    for (int t = 0; t < 2; ++t) {
      P.type_ar[t] = c.type_action_range[t]; P.loss_prey_t[t] = c.energy_loss_prey_t[t]; P.thr_prey_t[t] = c.creation_threshold_prey_t[t];
      P.init_e_prey_t[t] = c.initial_energy_prey_t[t]; P.bite_t[t] = c.bite_size_prey_t[t];
    }
    for (int k = 0; k < 3; ++k) P.death_pen[k] = c.death_penalty[k];
    P.equal_split = c.team_capture_equal_split != 0; P.coop_enabled = c.coop_trait_enabled != 0; P.capture_model = c.team_capture_success_model;
    P.strict_out = c.strict_rllib_output != 0;
    P.n_walls = (int)h->walls.size(); P.los_move = c.respect_los_for_movement != 0;
    P.cap_margin = c.team_capture_margin; P.join_cost = c.team_capture_join_cost; P.scav_frac = c.team_capture_scavenger_fraction;
    P.nature_w = c.team_capture_nature_weight; P.p0 = c.team_capture_base_success_p0; P.force_ratio = c.team_capture_force_success_ratio;
    P.min_prob = c.team_capture_min_success_prob; P.trait_mean = c.coop_trait_init_mean; P.trait_std = c.coop_trait_init_std;
    P.trait_mut_std = c.coop_trait_mutation_std; P.trait_mut_rate = c.coop_trait_mutation_rate;
  } else {
    P.action_range = 3; P.n_actions = 9;
  }
  for (int s = 0; s < 2; ++s) {
    P.R[s] = c.obs_range[s]; P.off[s] = (c.obs_range[s] - 1) / 2; P.elems[s] = row_channels * c.obs_range[s] * c.obs_range[s];
    P.cap[s] = c.cap_live[s]; P.n_init[s] = c.n_initial[s]; P.n_possible[s] = c.n_possible[s];
    P.loss[s] = c.energy_loss[s]; P.thr[s] = c.creation_threshold[s]; P.init_e[s] = c.initial_energy[s];
    P.r_repro[s] = c.reproduction_reward[s]; P.r_kick[s] = c.kickback_reward[s];
  }
  P.n_grass = c.n_grass; P.max_steps = c.max_steps; P.reward_mode = c.reward_mode; P.autoreset = c.autoreset;
  P.grass_cap = (eco || stag) ? c.max_energy_grass : c.initial_energy_grass; P.grass_gain = c.energy_gain_grass;
  P.season_len = (!eco && !stag) ? c.season_length_steps : 0;
  for (int k = 0; k < 2; ++k) P.grass_gain_season[k] = c.energy_gain_grass * c.season_multiplier[k];  // the reference's fp64 product (SEASON:268)
  P.init_e_grass = c.initial_energy_grass;
  P.r_catch = c.reward_predator_catch_prey; P.r_eat = c.reward_prey_eat_grass; P.r_pstep = c.reward_predator_step;
  P.r_qstep = c.reward_prey_step; P.pen_caught = c.penalty_prey_caught;

  const bool dense = c.reward_mode == PPG_REWARD_DENSE || c.reward_mode == PPG_REWARD_DENSE_ADDITIVE;
  const bool kick = c.reward_mode == PPG_REWARD_SPARSE_KICKBACK;

  P.obs_bulk = 0;
  if (const char* ev = getenv("PPG_OBS_BULK")) P.obs_bulk = atoi(ev) != 0;
  // padded map geometry (ppg_base.cu): halo as wide as the largest observation window
  P.P = std::max(P.off[0], P.off[1]);
  P.PH = P.P;
  if (stag) P.PH = std::max(2 * P.off[0], P.off[1]);  // forward view: the effective window centre lies up to off[0] cells past the far edge
  P.PS = G + P.PH;
  P.CH = (int)align_up((size_t)P.P + (size_t)(G + P.P + P.PH) * P.PS + P.P, 4);
  P.map_bytes = (P.cap[0] <= 253 && P.cap[1] <= 253 && P.n_grass <= 253) ? 1 : 2;
  P.wall_idx = P.cap[0] + 1;
  for (int s = 0; s < 2; ++s) {
    P.obs_vec[s] = P.elems[s] % 4 == 0;
    P.nj[s] = P.obs_vec[s] ? 4 * ((P.elems[s] / 4 + 31) / 32) : (P.elems[s] + 31) / 32;
    P.emit_kind[s] = (P.obs_vec[s] && P.nj[s] == 8) ? 1 : (P.obs_vec[s] && P.nj[s] == 12) ? 2 : (!P.obs_vec[s] && P.nj[s] == 13) ? 3
                     : (!P.obs_vec[s] && P.nj[s] == 5) ? 4 : (!P.obs_vec[s] && P.nj[s] == 8) ? 5 : 0;
  }
  if (P.nj[0] > PPG_MAX_NJ || P.nj[1] > PPG_MAX_NJ) { h->err = "observation row too large for this build"; return fail(PPG_ERR_INVALID); }

  // shared-memory layout of one env (see EnvSmem in ppg_base.cu)
  size_t o = 0;
  auto take = [&](size_t bytes, size_t al) { o = align_up(o, al); size_t r = o; o += bytes; return (int)r; };
  for (int s = 0; s < 2; ++s) { P.so_E[s] = take(8 * (size_t)P.cap[s], 8); P.so_E0[s] = take(dense ? 8 * (size_t)P.cap[s] : 0, 8); }
  P.so_gE = take(8 * (size_t)std::max(1, P.n_grass), 8);
  P.stage_elems = (int)align_up((size_t)std::max(P.elems[0], P.elems[1]), 4);
  // value tables and staging rows are contiguous: reset() stages n_total cells + a GG-entry claim table there
  if (o - (size_t)P.so_E[0] < (size_t)GG * 4) take((size_t)GG * 4 - (o - (size_t)P.so_E[0]), 1);  // reset(): GG-entry claim table over the energy arrays
  P.so_stage = take(P.obs_bulk ? 2 * 4 * (size_t)P.stage_elems : 0, 16);  // row staging only for the bulk-copy writer
  for (int s = 0; s < 2; ++s) {
    P.so_id[s] = take(2 * (size_t)P.cap[s], 2); P.so_pos[s] = take(2 * (size_t)P.cap[s], 2);
    P.so_ord[s] = take(2 * (size_t)P.cap[s], 2); P.so_rnk[s] = take(2 * (size_t)P.cap[s], 2);
    P.so_par[s] = take(kick ? 2 * (size_t)P.cap[s] : 0, 2);
  }
  // ---- the env IMAGE (what the observation kernel needs): header, value tables, row descriptors, maps, wall table ----
  P.so_ihdr = take(4 * (size_t)IH_INTS, 16);
  P.so_img = P.so_ihdr;
  P.so_vt[0] = take(4 * (size_t)(P.cap[0] + 2), 16);
  P.so_vt[1] = take(4 * (size_t)(P.cap[1] + 1), 4);
  P.so_vt[2] = take(4 * (size_t)(P.n_grass + 1), 4);
  for (int s = 0; s < 2; ++s) P.so_dsx[s] = take((eco || stag) ? 4 * (size_t)P.cap[s] : 0, 4);
  for (int s = 0; s < 2; ++s) P.so_dsc[s] = take(2 * (size_t)P.cap[s], 2);
  {
    const size_t need = (size_t)(P.n_init[0] + P.n_init[1] + P.n_grass) * 4;  // reset(): the drawn cells are staged in the value tables (and the descriptors behind them)
    if (o - (size_t)P.so_vt[0] < need) take(need - (o - (size_t)P.so_vt[0]), 1);
  }
  // reset() stages its n_total cells in the value tables and a GG-entry claim table over the energy arrays
  if ((size_t)GG * 4 > (size_t)(P.so_vt[0] - P.so_E[0])) {
    h->err = "internal: reset scratch does not fit (cap_live too small for this grid)"; return fail(PPG_ERR_INVALID);
  }
  // maps, wall table and touch counters are contiguous: their initial contents are one image copied by every warp
  P.so_map[0] = take((size_t)P.map_bytes * P.CH, 16);
  P.so_map[1] = take((size_t)P.map_bytes * P.CH, 4);
  P.so_map[2] = take((size_t)P.map_bytes * P.CH, 4);
  P.so_map[3] = take(stag ? (size_t)P.map_bytes * P.CH : 0, 4);  // STAG: rabbits (grid channel 3)
  P.so_wt = take(4 * (size_t)(P.cap[0] + 2), 4);
  o = align_up(o, 16);
  P.img_bytes = (int)(o - (size_t)P.so_img);
  P.img_stride = (int)align_up((size_t)P.img_bytes, 128);
  P.so_scr = take((size_t)P.CH, 16);
  o = align_up(o, 16);
  P.init_bytes = (int)(o - (size_t)P.so_map[0]);
  P.so_gpos = take(2 * (size_t)std::max(1, P.n_grass), 2);
  for (int s = 0; s < 2; ++s) { P.so_act[s] = take(P.cap[s], 1); P.so_flg[s] = take(P.cap[s], 1); P.so_aux[s] = take(kick ? P.cap[s] : 0, 1); }
  P.so_gtag = take(std::max(1, P.n_grass), 1);
  if (eco) {
    for (int s = 0; s < 2; ++s) {
      P.so_spd[s] = take(8 * (size_t)P.cap[s], 8); P.so_age[s] = take(2 * (size_t)P.cap[s], 2);
      P.so_seq[s] = take(2 * (size_t)P.cap[s], 2); P.so_mord[s] = take(2 * (size_t)P.cap[s], 2);
      P.so_acc[s] = take(P.trait_mode == PPG_TRAIT_CADENCE ? 8 * (size_t)P.cap[s] : 0, 8);
    }
  }
  if (stag) {
    P.so_trait = take(8 * (size_t)P.cap[0], 8);
    for (int s = 0; s < 2; ++s) { P.so_age[s] = take(2 * (size_t)P.cap[s], 2); P.so_mord[s] = take(2 * (size_t)P.cap[s], 2); }
    P.so_face = take(P.cap[0], 1); P.so_join = take(P.cap[0], 1);
  }
  P.smem_per_env = (int)align_up(o, 128);
  const size_t smem_max = 227 * 1024;
  if ((size_t)P.smem_per_env > smem_max) { h->err = "cap_live/grid too large for shared memory"; return fail(PPG_ERR_INVALID); }
  {
    // per-lane gather constants: element q = lane + 32 j of a row is channel c, window cell (i, jj);
    // BASE channels: 0 = outside the grid (predator map halo -> wall table), 1 predators, 2 prey, 3 grass
    {
      std::vector<unsigned char> img((size_t)P.init_bytes, 0);
      for (int i = 0; i < P.CH; ++i) {
        const int xx = i >= P.P ? (i - P.P) / P.PS - P.P : -1, yy = i >= P.P ? (i - P.P) % P.PS : 0;
        const bool field = i >= P.P && xx >= 0 && xx < G && yy < G;
        if (!field && !eco && !stag) {  // ECO has no wall channel; STAG's wall channel is empty (walls are rejected by the config layer): out-of-grid window cells stay 0 (ECO:700-706)
          if (P.map_bytes == 1) img[(size_t)i] = (unsigned char)P.wall_idx;
          else reinterpret_cast<uint16_t*>(img.data())[i] = (uint16_t)P.wall_idx;
        }
      }
      if (!eco && !stag) reinterpret_cast<float*>(img.data() + (P.so_wt - P.so_map[0]))[P.wall_idx] = 1.0f;
      if (stag && !h->walls.empty()) {  // STAG walls (STAG:2152-2159): static WALL entries of the predator map, shown by channel 0
        for (int w : h->walls) {
          const int i = P.P + (w / G + P.P) * P.PS + w % G;
          if (P.map_bytes == 1) img[(size_t)i] = (unsigned char)P.wall_idx;
          else reinterpret_cast<uint16_t*>(img.data())[i] = (uint16_t)P.wall_idx;
        }
        reinterpret_cast<float*>(img.data() + (P.so_wt - P.so_map[0]))[P.wall_idx] = 1.0f;
        int32_t* d_w = nullptr;
        CKC(dalloc(h, &d_w, h->walls.size()));
        CKC(cudaMemcpy(d_w, h->walls.data(), h->walls.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        P.wall_cells = d_w;
      }
      unsigned char* d_img = nullptr;
      CKC(dalloc(h, &d_img, img.size()));
      CKC(cudaMemcpy(d_img, img.data(), img.size(), cudaMemcpyHostToDevice));
      P.init_image = d_img;
    }
    std::vector<int> rel((size_t)2 * PPG_MAX_NJ * 32 * 2, 0);
    std::vector<unsigned> selfm(64, 0u);
    for (int s = 0; s < 2; ++s) {
      const int R = P.R[s], RR = R * R;
      for (int j = 0; j < P.nj[s]; ++j)
        for (int lane = 0; lane < 32; ++lane) {
          const size_t at0 = ((size_t)(s * PPG_MAX_NJ + j) * 32 + lane) * 2;
          rel[at0] = 0; rel[at0 + 1] = P.so_wt;  // lanes past the end of the row: a harmless in-range read, never stored
          const int q = P.obs_vec[s] ? 4 * (lane + 32 * (j / 4)) + (j % 4) : j * 32 + lane;
          if (q >= P.elems[s]) continue;
          const int ch = q / RR, i = (q % RR) / R, jj = q % R;
          const int cellrel = (i - P.off[s]) * P.PS + (jj - P.off[s]);
          const size_t at = ((size_t)(s * PPG_MAX_NJ + j) * 32 + lane) * 2;
          if (eco && ch >= 3) { selfm[(size_t)s * 32 + lane] |= 1u << j; continue; }  // ECO's own-speed plane
          const ChannelSource src = channel_source(P, ch);
          rel[at] = (src.map - P.so_map[0]) + cellrel * P.map_bytes;
          rel[at + 1] = src.tbl;
        }
    }
    int* d_rel = nullptr;
    CKC(dalloc(h, &d_rel, rel.size()));
    CKC(cudaMemcpy(d_rel, rel.data(), rel.size() * sizeof(int), cudaMemcpyHostToDevice));
    P.obs_rel = reinterpret_cast<const int2*>(d_rel);
    if (eco) {
      unsigned* d_self = nullptr;
      CKC(dalloc(h, &d_self, selfm.size()));
      CKC(cudaMemcpy(d_self, selfm.data(), selfm.size() * sizeof(unsigned), cudaMemcpyHostToDevice));
      P.obs_self = d_self;
    }
  }
  int W = 1;
  if (const char* ev = getenv("PPG_WARPS_PER_CTA")) W = atoi(ev);
  if (W != 1 && W != 4 && W != 8) W = 1;
  while (W > 1 && (size_t)W * P.smem_per_env > smem_max) W >>= 1;
  if (eco || stag) W = 1;
  // two-kernel step (default): the step kernel leaves env images, ppg_obs_kernel writes the observation rows
  P.obs_split = 1;
  if (const char* ev = getenv("PPG_OBS_SPLIT")) P.obs_split = atoi(ev) != 0;
  if (W != 1 || P.obs_bulk || P.CH >= (int)DSC_COPY) P.obs_split = 0;
  h->warps_per_cta = W;
  h->smem_bytes = (size_t)W * P.smem_per_env;
  {
    // persistent warps: as many CTAs as fit on the device, never more than there are envs
    int per_sm = 0, n_sm = 0;
    if (eco) CKC(step_eco_occupancy(P.map_bytes, P.obs_split != 0, P.trait_mode != PPG_TRAIT_SPEED ? 1 : (P.lin_on ? 2 : 0), h->smem_bytes, &per_sm));
    else if (stag) CKC(step_stag_occupancy(P.map_bytes, P.obs_split != 0, h->smem_bytes, &per_sm));
    else CKC(step_base_occupancy(W, P.map_bytes, P.obs_bulk != 0, P.obs_split != 0, h->smem_bytes, &per_sm));
    CKC(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
    if (per_sm < 1) { h->err = "step kernel does not fit on an SM"; return fail(PPG_ERR_INVALID); }
    h->n_cta = std::min((B + W - 1) / W, per_sm * n_sm);
    if (const char* ev = getenv("PPG_MAX_CTAS")) h->n_cta = std::max(1, std::min(h->n_cta, atoi(ev)));
  }

  // state
  CKC(dalloc(h, &P.hdr, (size_t)B));
  for (int s = 0; s < 2; ++s) {
    const size_t n = (size_t)B * P.cap[s];
    CKC(dalloc(h, &P.ag_id[s], n)); CKC(dalloc(h, &P.ag_pos[s], n)); CKC(dalloc(h, &P.ag_e[s], n));
    CKC(dalloc(h, &P.ag_prow[s], n)); CKC(dalloc(h, &P.ag_par[s], c.reward_mode == PPG_REWARD_SPARSE_KICKBACK ? n : 1));
    if (eco) {
      CKC(dalloc(h, &P.ag_age[s], n)); CKC(dalloc(h, &P.ag_seq[s], n)); CKC(dalloc(h, &P.ag_spd[s], n)); CKC(dalloc(h, &P.ag_dead[s], n));
      if (P.trait_mode == PPG_TRAIT_CADENCE) CKC(dalloc(h, &P.ag_acc[s], n));
      if (P.lin_on) {
        const size_t m = (size_t)B * P.n_possible[s];
        CKC(dalloc(h, &P.lin_parent[s], m)); CKC(dalloc(h, &P.lin_live[s], m)); CKC(dalloc(h, &P.lin_prev[s], m)); CKC(dalloc(h, &P.lin_alive[s], m));
      }
    }
    if (stag) {
      CKC(dalloc(h, &P.ag_age[s], n));
      if (s == 0) { CKC(dalloc(h, &P.ag_face, n)); CKC(dalloc(h, &P.ag_trait, n)); }
    }
    std::vector<uint16_t> lr = lexrank_table(c.n_possible[s]);
    uint16_t* d = nullptr;
    CKC(dalloc(h, &d, lr.size()));
    CKC(cudaMemcpy(d, lr.data(), lr.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    P.lexrank[s] = d;
  }
  {
    const size_t n_blk = ((size_t)B + 31) / 32, n_grp = ((size_t)B + 1023) / 1024;
    for (int q = 0; q < 2; ++q) {
      CKC(dalloc(h, &P.cntA[q], (size_t)B)); CKC(dalloc(h, &P.cntB[q], (size_t)B));
      CKC(dalloc(h, &P.sum1[q], n_blk * 4)); CKC(dalloc(h, &P.sum2[q], n_grp * 4));
    }
    CKC(dalloc(h, &P.acc1, n_blk * 2)); CKC(dalloc(h, &P.acc2, n_grp * 2)); CKC(dalloc(h, &P.acc3, 2));
    CKC(dalloc(h, &P.totals, 8));
    // big-envs-first order of the next launch: only where no env ever waits for another one (publish_begin)
    bool lpt = !eco && P.obs_split;
    if (const char* ev = getenv("PPG_ENV_ORDER")) lpt = lpt && atoi(ev) != 0;
    if (lpt) { for (int q = 0; q < 2; ++q) CKC(dalloc(h, &P.perm[q], (size_t)B)); CKC(dalloc(h, &P.perm_tag, 2)); CKC(dalloc(h, &P.perm_cursor, 4)); CKC(cudaMemset(P.perm_tag, 0xFF, 2 * sizeof(unsigned))); }  // no epoch carries tag 0xFFFFFFFF
  }
  if (eco) {
    CKC(dalloc(h, &P.ehdr, (size_t)B));
    if (c.track_episode_sums) CKC(dalloc(h, &P.ep_sums, (size_t)B * PPG_EP_STRIDE));
    CKC(dalloc(h, &P.gh_n, (size_t)B)); CKC(dalloc(h, &P.gh_cell, (size_t)B * PPG_MAX_GHOSTS)); CKC(dalloc(h, &P.gh_val, (size_t)B * PPG_MAX_GHOSTS));
  }
  if (stag) CKC(dalloc(h, &P.shdr, (size_t)B));
  CKC(dalloc(h, &P.gr_pos, (size_t)B * std::max(1, P.n_grass)));
  CKC(dalloc(h, &P.gr_e, (size_t)B * std::max(1, P.n_grass)));
  CKC(dalloc(h, &P.counters, (size_t)B * PPG_N_STATS));
  CKC(dalloc(h, &P.ticket, 1));
  CKC(dalloc(h, &P.env_cycles, (size_t)B));
  if (P.obs_split) {
    void* q = nullptr;
    CKC(cudaMalloc(&q, (size_t)B * (size_t)P.img_stride));  // not cleared: every launch writes every env's header
    h->allocs.push_back(q);
    P.obs_img = static_cast<unsigned char*>(q);
    for (int s = 0; s < 2; ++s) CKC(dalloc(h, &P.nb_info[s], (size_t)B * P.cap[s]));
    CKC(dalloc(h, &P.obs_ticket, 1));
    CKC(dalloc(h, &P.queue, (size_t)B));
    CKC(dalloc(h, &P.q_tail, 1));
    if (const char* ev = getenv("PPG_OBS_OVERLAP")) h->obs_overlap = atoi(ev) != 0;
    if (eco)
      for (int s = 0; s < 2; ++s) CKC(dalloc(h, &P.born_obs[s], (size_t)B * PPG_BORN_K * (size_t)P.elems[s]));
    int per_sm = 0, n_sm = 0;
    CKC(obs_occupancy(P, &per_sm));
    CKC(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device));
    if (per_sm < 1) { h->err = "observation kernel does not fit on an SM"; return fail(PPG_ERR_INVALID); }
    h->n_cta_obs = std::min(B, per_sm * n_sm);
    if (const char* ev = getenv("PPG_OBS_CTAS_PER_SM")) h->n_cta_obs = std::max(1, std::min(h->n_cta_obs, atoi(ev) * n_sm));
    // overlap: leave room on every SM for observation CTAs next to the step kernel's persistent warps
    if (const char* ev = getenv("PPG_STEP_CTAS_PER_SM")) h->n_cta = std::max(1, std::min(h->n_cta, atoi(ev) * n_sm));
  }
  CKC(dalloc(h, &P.error, 1));
  CKC(dalloc(h, &h->d_stats, PPG_N_STATS));
  CKC(dalloc(h, &h->d_mask, (size_t)B));
  CKC(dalloc(h, &h->d_seeds, (size_t)B));
  // outputs
  ppg_buffers& b = h->bufs;
  memset(&b, 0, sizeof b);
  for (int s = 0; s < 2; ++s) {
    const size_t rows = (size_t)B * P.cap[s];
    b.row_capacity[s] = (int64_t)rows;
    b.obs_row_elems[s] = P.elems[s];
    void* q = nullptr;
    CKC(cudaMalloc(&q, rows * (size_t)P.elems[s] * sizeof(float)));  // not cleared: only valid rows are ever read
    h->allocs.push_back(q);
    P.obs[s] = b.obs[s] = static_cast<float*>(q);
    CKC(dalloc(h, &P.row_env[s], rows)); CKC(dalloc(h, &P.row_agent[s], rows));
    CKC(dalloc(h, &P.reward[s], rows)); CKC(dalloc(h, &P.flags[s], rows));
    CKC(dalloc(h, &P.old_off[s], (size_t)B + 1)); CKC(dalloc(h, &P.new_off[s], (size_t)B + 1));
    CKC(dalloc(h, &P.new_cnt[s], (size_t)B + 1));
    CKC(dalloc(h, &h->d_act[s], rows));
    b.row_env[s] = P.row_env[s]; b.row_agent[s] = P.row_agent[s]; b.reward[s] = P.reward[s]; b.flags[s] = P.flags[s];
    b.old_off[s] = P.old_off[s]; b.new_off[s] = P.new_off[s]; b.new_cnt[s] = P.new_cnt[s];
  }
  CKC(dalloc(h, &P.n_rows, 4)); CKC(dalloc(h, &P.env_flags, (size_t)B)); CKC(dalloc(h, &P.env_status, (size_t)B));
  CKC(dalloc(h, &P.env_step, (size_t)B)); CKC(dalloc(h, &P.env_count, (size_t)B * 2));
  b.n_rows = P.n_rows; b.env_flags = P.env_flags; b.env_status = P.env_status; b.env_step = P.env_step; b.env_count = P.env_count;
  b.n_envs = B;
  CKC(launch_init_hdr(P.hdr, B, c.seed, 0));
  h->launch_count++;
  CKC(cudaDeviceSynchronize());
  *out = h;
  return PPG_OK;
#undef CKC
}

int ppg_destroy(ppg_handle h) {
  if (!h) return PPG_OK;
  cudaSetDevice(h->device);
  for (void* p : h->allocs) cudaFree(p);
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  if (h->d_tape_cells) cudaFree(h->d_tape_cells);
  if (h->d_tape_off) cudaFree(h->d_tape_off);
  if (h->d_tape_reals) cudaFree(h->d_tape_reals);
  if (h->d_tape_real_off) cudaFree(h->d_tape_real_off);
  delete h;
  return PPG_OK;
}

int ppg_load_tape(ppg_handle h, const ppg_tape* t) {
  if (!h) return PPG_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  if (h->d_tape_cells) { cudaFree(h->d_tape_cells); h->d_tape_cells = nullptr; }
  if (h->d_tape_off) { cudaFree(h->d_tape_off); h->d_tape_off = nullptr; }
  h->P.tape_cells = nullptr;
  if (t && t->cells && t->cell_off) {
    const int64_t total = t->cell_off[h->B];
    CK(cudaMalloc(&h->d_tape_cells, sizeof(int32_t) * (size_t)std::max<int64_t>(total, 1)));
    CK(cudaMalloc(&h->d_tape_off, sizeof(long long) * ((size_t)h->B + 1)));
    CK(cudaMemcpy(h->d_tape_cells, t->cells, sizeof(int32_t) * (size_t)total, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(h->d_tape_off, t->cell_off, sizeof(long long) * ((size_t)h->B + 1), cudaMemcpyHostToDevice));
    h->P.tape_cells = h->d_tape_cells;
  }
  CK(launch_set_tape(h->P.hdr, h->B, h->d_tape_off, 0));
  h->launch_count++;
  if (h->P.variant == PPG_VARIANT_ECO || h->P.variant == PPG_VARIANT_STAG) {
    if (h->d_tape_reals) { cudaFree(h->d_tape_reals); h->d_tape_reals = nullptr; }
    if (h->d_tape_real_off) { cudaFree(h->d_tape_real_off); h->d_tape_real_off = nullptr; }
    h->P.tape_reals = nullptr;
    if (t && t->reals && t->real_off) {
      const int64_t total = t->real_off[h->B];
      CK(cudaMalloc(&h->d_tape_reals, sizeof(double) * (size_t)std::max<int64_t>(total, 1)));
      CK(cudaMalloc(&h->d_tape_real_off, sizeof(long long) * ((size_t)h->B + 1)));
      CK(cudaMemcpy(h->d_tape_reals, t->reals, sizeof(double) * (size_t)total, cudaMemcpyHostToDevice));
      CK(cudaMemcpy(h->d_tape_real_off, t->real_off, sizeof(long long) * ((size_t)h->B + 1), cudaMemcpyHostToDevice));
      h->P.tape_reals = h->d_tape_reals;
    }
    if (h->P.variant == PPG_VARIANT_ECO) CK(launch_set_tape_reals(h->P.ehdr, h->B, h->d_tape_real_off, 0));
    else CK(launch_set_tape_reals_stag(h->P.shdr, h->B, h->d_tape_real_off, 0));
    h->launch_count++;
  }
  CK(cudaDeviceSynchronize());
  return PPG_OK;
}

// publish the rows every env needs in the next output under the tag of the launch that "just ran"
static int prepare_offsets(ppg_handle h, cudaStream_t st) {
  const unsigned prev_epoch = (unsigned)h->launches_step;
  const int q = (int)(prev_epoch & 1u);
  CK(launch_prepare_offsets(h->P.hdr, h->B, h->P.n_init[0], h->P.n_init[1], h->P.cntA[q], h->P.sum1[q], h->P.sum2[q],
                            h->P.totals + 4 * q, prev_epoch, h->P.variant == PPG_VARIANT_ECO && ppg_random_founders(h->P.trait_mode), st));
  h->launch_count++;
  return PPG_OK;
}

static int run_step_kernel(ppg_handle h, const int32_t* a0, const int32_t* a1, const int32_t* o0, const int32_t* o1, cudaStream_t st) {
  StepParams& P = h->P;
  P.actions[0] = a0; P.actions[1] = a1;
  P.order[0] = o0; P.order[1] = o1;
  P.ticket_base = h->ticket_next;
  // tickets: one per env (W == 1) or per group of W envs, plus one terminating draw per warp / CTA.  static_first: a
  // warp's first ticket is its CTA index and every env it works on draws the warp's next one: exactly B draws.
  P.static_first = (h->warps_per_cta == 1 && P.obs_split && P.variant != PPG_VARIANT_ECO) ? 1 : 0;
  if (const char* ev = getenv("PPG_STATIC_FIRST")) P.static_first = P.static_first && atoi(ev) != 0;
  h->ticket_next += P.static_first ? (unsigned long long)h->B
                    : h->warps_per_cta == 1 ? (unsigned long long)h->B + (unsigned long long)h->n_cta
                                          : (unsigned long long)((h->B + h->warps_per_cta - 1) / h->warps_per_cta) + (unsigned long long)h->n_cta;
  P.epoch = (unsigned)(h->launches_step + 1);
  P.q_base = h->q_next;
  if (P.obs_split) h->q_next += (unsigned long long)h->B;  // every env pushes one completion-queue entry per launch
  cudaEvent_t pe[3] = {nullptr, nullptr, nullptr};
  if (h->profiling) {
    for (int k = 0; k < 3; ++k) { CK(cudaEventCreate(&pe[k])); h->prof_events.push_back(pe[k]); }
    CK(cudaEventRecord(pe[0], st));
  }
  if (P.variant == PPG_VARIANT_ECO) CK(launch_step_eco(P, h->n_cta, h->smem_bytes, st));
  else if (P.variant == PPG_VARIANT_STAG) CK(launch_step_stag(P, h->n_cta, h->smem_bytes, st));
  else CK(launch_step_base(P, h->warps_per_cta, h->n_cta, h->smem_bytes, st));
  h->launches_step++;
  h->launch_count++;
  if (h->profiling) CK(cudaEventRecord(pe[1], st));
  if (P.obs_split) {
    // observation rows of this output: one CTA per env at a time, B tickets plus one terminating draw per CTA
    P.obs_ticket_base = h->obs_ticket_next;
    h->obs_ticket_next += (unsigned long long)h->B + (unsigned long long)h->n_cta_obs;
    CK(launch_obs(P, h->n_cta_obs, h->obs_overlap && !h->profiling, st));  // per-kernel timing needs the kernels back to back
    h->launch_count++;
  }
  if (h->profiling) CK(cudaEventRecord(pe[2], st));
  if (h->track_on) {  // after pe[2]: the per-kernel timing of the step is the same with tracking on
    CK(launch_returns(h->R, st));
    h->launch_count++;
  }
  // the images now hold this output's world, except that an env idle since a ppg_restore still has the pre-restore one:
  // after restoring idle envs only a full reset (a0 == NULL, every env dumps its image) makes them valid again
  if (a0 == nullptr || h->img != ppg_handle_s::IMG_RESTORED_IDLE) h->img = ppg_handle_s::IMG_VALID;
  h->calls++;
  h->h_n_rows_valid = false;
  return PPG_OK;
}

int ppg_reset(ppg_handle h, const uint64_t* seeds, const uint8_t* mask, void* cuda_stream) {
  if (!h) return PPG_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaSetDevice(h->device));
  const unsigned long long* dseeds = nullptr;
  if (seeds) { CK(cudaMemcpyAsync(h->d_seeds, seeds, sizeof(uint64_t) * (size_t)h->B, cudaMemcpyHostToDevice, st)); dseeds = h->d_seeds; }
  const uint8_t* dmask = nullptr;
  if (mask) { CK(cudaMemcpyAsync(h->d_mask, mask, (size_t)h->B, cudaMemcpyHostToDevice, st)); dmask = h->d_mask; }
  CK(launch_mark_reset(h->P.hdr, h->B, dseeds, dmask, st));
  h->launch_count++;
  const bool random_founders = h->P.variant == PPG_VARIANT_ECO && ppg_random_founders(h->P.trait_mode);
  if (random_founders) {  // MR:189-192: the number of founders is drawn per episode; the row allocator needs it before the reset runs
    CK(launch_eco_founders(h->P, st));
    h->launch_count++;
  }
  int rc = prepare_offsets(h, st);
  if (rc) return rc;
  if (mask) return PPG_OK;  // partial reset: performed by the next ppg_step
  rc = run_step_kernel(h, nullptr, nullptr, nullptr, nullptr, st);
  if (rc) return rc;
  h->h_n_rows[0] = h->B * h->P.n_init[0]; h->h_n_rows[1] = h->B * h->P.n_init[1];
  h->h_n_rows[2] = h->h_n_rows[3] = 0;
  h->h_n_rows_valid = !random_founders;
  return PPG_OK;
}

int ppg_step(ppg_handle h, const int32_t* actions_pred, const int32_t* actions_prey, void* cuda_stream) {
  if (!h) return PPG_ERR_INVALID;
  if (!actions_pred || !actions_prey) { h->err = "ppg_step: NULL actions"; return PPG_ERR_INVALID; }
  if (h->launches_step == 0) { h->err = "ppg_step before ppg_reset"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  return run_step_kernel(h, actions_pred, actions_prey, nullptr, nullptr, static_cast<cudaStream_t>(cuda_stream));
}

int ppg_step_ordered(ppg_handle h, const int32_t* actions_pred, const int32_t* actions_prey, const int32_t* order_pred,
                     const int32_t* order_prey, void* cuda_stream) {
  if (!h) return PPG_ERR_INVALID;
  if (!actions_pred || !actions_prey) { h->err = "ppg_step_ordered: NULL actions"; return PPG_ERR_INVALID; }
  if (h->launches_step == 0) { h->err = "ppg_step_ordered before ppg_reset"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  return run_step_kernel(h, actions_pred, actions_prey, order_pred, order_prey, static_cast<cudaStream_t>(cuda_stream));
}

int ppg_step_host(ppg_handle h, const int32_t* actions_pred, const int32_t* actions_prey, ppg_buffers* out,
                  int32_t* n_rows_out, void* cuda_stream) {
  if (!h || !out) return PPG_ERR_INVALID;
  if (h->launches_step == 0) { h->err = "ppg_step_host before ppg_reset"; return PPG_ERR_STATE; }
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaSetDevice(h->device));
  if (!h->h_n_rows_valid) {
    CK(cudaMemcpyAsync(h->h_n_rows, h->P.n_rows, sizeof h->h_n_rows, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  const int32_t* src[2] = {actions_pred, actions_prey};
  for (int s = 0; s < 2; ++s) {
    const size_t n = (size_t)h->h_n_rows[s] + (size_t)h->h_n_rows[2 + s];
    if (n) CK(cudaMemcpyAsync(h->d_act[s], src[s], n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  }
  int rc = run_step_kernel(h, h->d_act[0], h->d_act[1], nullptr, nullptr, st);
  if (rc) return rc;
  CK(cudaMemcpyAsync(h->h_n_rows, h->P.n_rows, sizeof h->h_n_rows, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  h->h_n_rows_valid = true;
  for (int s = 0; s < 2; ++s) {
    const size_t n = (size_t)h->h_n_rows[s] + (size_t)h->h_n_rows[2 + s];
    if ((int64_t)n > out->row_capacity[s]) { h->err = "ppg_step_host: host row_capacity too small"; return PPG_ERR_INVALID; }
    if (n) {
      if (out->obs[s]) CK(cudaMemcpyAsync(out->obs[s], h->P.obs[s], n * (size_t)h->P.elems[s] * sizeof(float), cudaMemcpyDeviceToHost, st));
      if (out->row_env[s]) CK(cudaMemcpyAsync(out->row_env[s], h->P.row_env[s], n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      if (out->row_agent[s]) CK(cudaMemcpyAsync(out->row_agent[s], h->P.row_agent[s], n * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      if (out->reward[s]) CK(cudaMemcpyAsync(out->reward[s], h->P.reward[s], n * sizeof(float), cudaMemcpyDeviceToHost, st));
      if (out->flags[s]) CK(cudaMemcpyAsync(out->flags[s], h->P.flags[s], n, cudaMemcpyDeviceToHost, st));
    }
    if (out->old_off[s]) CK(cudaMemcpyAsync(out->old_off[s], h->P.old_off[s], ((size_t)h->B + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (out->new_off[s]) CK(cudaMemcpyAsync(out->new_off[s], h->P.new_off[s], (size_t)h->B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (out->new_cnt[s]) CK(cudaMemcpyAsync(out->new_cnt[s], h->P.new_cnt[s], (size_t)h->B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  }
  if (out->env_flags) CK(cudaMemcpyAsync(out->env_flags, h->P.env_flags, (size_t)h->B, cudaMemcpyDeviceToHost, st));
  if (out->env_status) CK(cudaMemcpyAsync(out->env_status, h->P.env_status, (size_t)h->B, cudaMemcpyDeviceToHost, st));
  if (out->env_step) CK(cudaMemcpyAsync(out->env_step, h->P.env_step, (size_t)h->B * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  if (out->env_count) CK(cudaMemcpyAsync(out->env_count, h->P.env_count, (size_t)h->B * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (n_rows_out) memcpy(n_rows_out, h->h_n_rows, sizeof h->h_n_rows);
  if (out->n_rows) memcpy(out->n_rows, h->h_n_rows, sizeof h->h_n_rows);
  return PPG_OK;
}

int ppg_random_actions(ppg_handle h, uint64_t seed, int32_t* actions_pred, int32_t* actions_prey, void* cuda_stream) {
  if (!h || !actions_pred || !actions_prey) return PPG_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  const StepParams& P = h->P;
  if (P.variant == PPG_VARIANT_STAG)
    CK(launch_random_actions_stag(P.n_rows, P.row_env[0], P.row_agent[0], P.row_env[1], P.row_agent[1], actions_pred, actions_prey, seed,
                                  (unsigned)h->calls, (unsigned)P.env_base, P.n_possible_t[0][0], P.n_possible_t[1][0], P.type_ar[0], P.type_ar[1],
                                  148 * 4, static_cast<cudaStream_t>(cuda_stream)));
  else
  CK(launch_random_actions(P.n_rows, P.row_env[0], P.row_agent[0], P.row_env[1], P.row_agent[1], actions_pred, actions_prey,
                           seed, (unsigned)h->calls, (unsigned)P.n_actions, (unsigned)P.env_base, 148 * 4, static_cast<cudaStream_t>(cuda_stream)));
  h->launch_count++;
  return PPG_OK;
}

int ppg_set_pdl_chain(int32_t on) {
  const int before = pdl_chain_enabled() ? 1 : 0;
  g_pdl_chain = on ? 1 : 0;
  return before;
}

int ppg_rollout_random(ppg_handle* handles, int32_t n_handles, void** cuda_streams, int32_t n_steps, uint64_t seed) {
  if (!handles || n_handles <= 0 || n_steps < 0) return PPG_ERR_INVALID;
  // several handles on their own streams: a step kernel parked in griddepcontrol.wait would hold the slots the other
  // group's kernels are meant to fill, so the launch chain is plain stream order here
  struct ChainOff { int before; bool off; ChainOff(bool o) : before(pdl_chain_enabled()), off(o) { if (off) g_pdl_chain = 0; } ~ChainOff() { if (off) g_pdl_chain = before; } } chain_off(n_handles > 1);
  for (int g = 0; g < n_handles; ++g) {
    if (!handles[g]) return PPG_ERR_INVALID;
    if (handles[g]->launches_step == 0) { handles[g]->err = "ppg_rollout_random before ppg_reset"; return PPG_ERR_STATE; }
  }
  for (int k = 0; k < n_steps; ++k)
    for (int g = 0; g < n_handles; ++g) {
      ppg_handle h = handles[g];
      void* st = cuda_streams ? cuda_streams[g] : nullptr;
      int rc = ppg_random_actions(h, seed, h->d_act[0], h->d_act[1], st);
      if (rc) return rc;
      rc = run_step_kernel(h, h->d_act[0], h->d_act[1], nullptr, nullptr, static_cast<cudaStream_t>(st));
      if (rc) return rc;
    }
  return PPG_OK;
}

int ppg_selftest_pow(const double* x, const double* y, double* out, int64_t n, int32_t device) {
  if (!x || !y || !out || n <= 0) return PPG_ERR_INVALID;
  if (cudaSetDevice(device) != cudaSuccess) { g_err = "ppg_selftest_pow: bad device"; return PPG_ERR_NO_DEVICE; }
  double *dx = nullptr, *dy = nullptr, *dz = nullptr;
  const size_t bytes = (size_t)n * sizeof(double);
  cudaError_t e = cudaMalloc(&dx, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&dy, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&dz, bytes);
  if (e == cudaSuccess) e = cudaMemcpy(dx, x, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dy, y, bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) { ppg_pow_selftest_kernel<<<148 * 8, 256>>>(dx, dy, dz, (long long)n); e = cudaGetLastError(); }
  if (e == cudaSuccess) e = cudaMemcpy(out, dz, bytes, cudaMemcpyDeviceToHost);
  cudaFree(dx); cudaFree(dy); cudaFree(dz);
  if (e != cudaSuccess) { g_err = std::string("ppg_selftest_pow: ") + cudaGetErrorString(e); return PPG_ERR_CUDA; }
  return PPG_OK;
}

int ppg_get_buffers(ppg_handle h, ppg_buffers* out) {
  if (!h || !out) return PPG_ERR_INVALID;
  *out = h->bufs;
  return PPG_OK;
}

// ---- snapshot / restore: the SoA slab as one host blob -----------------------------------------
struct Seg { void* p; size_t bytes; };
static std::vector<Seg> state_segments(ppg_handle h) {
  const StepParams& P = h->P;
  std::vector<Seg> v;
  v.push_back({P.hdr, sizeof(EnvHdr) * (size_t)h->B});
  for (int s = 0; s < 2; ++s) {
    const size_t n = (size_t)h->B * P.cap[s];
    v.push_back({P.ag_id[s], n * 2}); v.push_back({P.ag_pos[s], n * 2}); v.push_back({P.ag_e[s], n * 8});
    v.push_back({P.ag_prow[s], n * 4});
    if (P.reward_mode == PPG_REWARD_SPARSE_KICKBACK) v.push_back({P.ag_par[s], n * 2});
    if (P.variant == PPG_VARIANT_ECO) {
      v.push_back({P.ag_age[s], n * 2}); v.push_back({P.ag_seq[s], n * 2}); v.push_back({P.ag_spd[s], n * 8}); v.push_back({P.ag_dead[s], n});
      if (P.trait_mode == PPG_TRAIT_CADENCE) v.push_back({P.ag_acc[s], n * 8});
      if (P.lin_on) {
        const size_t m = (size_t)h->B * P.n_possible[s];
        v.push_back({P.lin_parent[s], m * 2}); v.push_back({P.lin_live[s], m * 2}); v.push_back({P.lin_prev[s], m * 2}); v.push_back({P.lin_alive[s], m});
      }
    }
    if (P.variant == PPG_VARIANT_STAG) {
      v.push_back({P.ag_age[s], n * 2});
      if (s == 0) { v.push_back({P.ag_face, n}); v.push_back({P.ag_trait, n * 8}); }
    }
  }
  if (P.variant == PPG_VARIANT_STAG) v.push_back({P.shdr, sizeof(StagHdr) * (size_t)h->B});
  if (P.variant == PPG_VARIANT_ECO) {
    v.push_back({P.ehdr, sizeof(EcoHdr) * (size_t)h->B});
    if (P.ep_sums) v.push_back({P.ep_sums, (size_t)h->B * PPG_EP_STRIDE * 8});
    v.push_back({P.gh_n, (size_t)h->B}); v.push_back({P.gh_cell, (size_t)h->B * PPG_MAX_GHOSTS * 2}); v.push_back({P.gh_val, (size_t)h->B * PPG_MAX_GHOSTS * 4});
  }
  v.push_back({P.gr_pos, (size_t)h->B * std::max(1, P.n_grass) * 2});
  v.push_back({P.gr_e, (size_t)h->B * std::max(1, P.n_grass) * 8});
  v.push_back({P.counters, (size_t)h->B * PPG_N_STATS * 4});
  return v;
}

static const size_t SNAP_HEAD = 32;  // calls, magic, total bytes, shape hash

static unsigned long long shape_hash(ppg_handle h) {
  const StepParams& P = h->P;
  const long long v[] = {h->B, P.variant, P.reward_mode, P.G, P.cap[0], P.cap[1], P.n_grass, P.n_possible[0], P.n_possible[1]};
  unsigned long long x = 1469598103934665603ULL;  // FNV-1a
  for (long long w : v)
    for (int k = 0; k < 8; ++k) { x ^= (unsigned long long)((w >> (8 * k)) & 0xFF); x *= 1099511628211ULL; }
  return x;
}

size_t ppg_snapshot_size(ppg_handle h) {
  if (!h) return 0;
  size_t t = SNAP_HEAD;
  for (const Seg& s : state_segments(h)) t += s.bytes;
  return t;
}

int ppg_snapshot(ppg_handle h, void* blob, size_t bytes, void* cuda_stream) {
  if (!h || !blob || bytes < ppg_snapshot_size(h)) return PPG_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaSetDevice(h->device));
  char* q = static_cast<char*>(blob);
  unsigned long long head[4] = {h->calls, 0x50504753ULL, (unsigned long long)ppg_snapshot_size(h), shape_hash(h)};
  memcpy(q, head, SNAP_HEAD);
  q += SNAP_HEAD;
  for (const Seg& s : state_segments(h)) { CK(cudaMemcpyAsync(q, s.p, s.bytes, cudaMemcpyDeviceToHost, st)); q += s.bytes; }
  CK(cudaStreamSynchronize(st));
  return PPG_OK;
}

int ppg_restore(ppg_handle h, const void* blob, size_t bytes, void* cuda_stream) {
  if (!h || !blob || bytes < SNAP_HEAD) return PPG_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaSetDevice(h->device));
  const char* q = static_cast<const char*>(blob);
  unsigned long long head[4];
  memcpy(head, q, SNAP_HEAD);
  if (head[1] != 0x50504753ULL) { h->err = "ppg_restore: not a snapshot blob"; return PPG_ERR_INVALID; }
  if (head[2] != (unsigned long long)ppg_snapshot_size(h) || head[3] != shape_hash(h) || bytes < ppg_snapshot_size(h)) {
    h->err = "ppg_restore: the blob was taken from a handle of another shape (n_envs / variant / grid / cap_live / n_grass)";
    return PPG_ERR_INVALID;
  }
  h->calls = head[0];
  q += SNAP_HEAD;
  {
    // the blob starts with the env headers; an env restored idle is never re-imaged by a step (header-only dump)
    bool idle = false;
    for (int e = 0; e < h->B && !idle; ++e) {
      EnvHdr hd;
      memcpy(&hd, q + (size_t)e * sizeof(EnvHdr), sizeof hd);
      idle = hd.state == ST_IDLE;
    }
    h->img = idle ? ppg_handle_s::IMG_RESTORED_IDLE : ppg_handle_s::IMG_RESTORED;
  }
  for (const Seg& s : state_segments(h)) { CK(cudaMemcpyAsync(s.p, q, s.bytes, cudaMemcpyHostToDevice, st)); q += s.bytes; }
  {
    int rc = prepare_offsets(h, st);
    if (rc) return rc;
    const int q = (int)(h->launches_step & 1ULL);
    CK(launch_relabel_rows(h->P, h->P.cntA[q], h->P.sum1[q], h->P.sum2[q], h->P.totals + 4 * q, st));
    h->launch_count++;
  }
  if (h->track_on) {  // the tracking state is not in the blob: every env is invalid until its next reset
    CK(cudaMemsetAsync(h->R.env_valid, 0, (size_t)h->B, st));
    CK(cudaMemsetAsync(h->R.env_return, 0xFF, (size_t)h->B * 2 * sizeof(double), st));  // all-ones bits: NaN
  }
  CK(cudaStreamSynchronize(st));
  h->h_n_rows_valid = false;
  return PPG_OK;
}

int ppg_track_returns(ppg_handle h, int32_t on, void* cuda_stream) {
  if (!h) return PPG_ERR_INVALID;
  if (!on) { h->track_on = false; return PPG_OK; }
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaSetDevice(h->device));
  ReturnsParams& R = h->R;
  const StepParams& P = h->P;
  if (!h->R_alloc) {
    memset(&R, 0, sizeof R);
    for (int s = 0; s < 2; ++s) {
      R.row_agent[s] = P.row_agent[s]; R.reward[s] = P.reward[s]; R.flags[s] = P.flags[s];
      R.old_off[s] = P.old_off[s]; R.new_off[s] = P.new_off[s]; R.new_cnt[s] = P.new_cnt[s];
      R.n_possible[s] = P.n_possible[s];
      CK(dalloc(h, &R.row_return[s], (size_t)h->bufs.row_capacity[s]));
      CK(dalloc(h, &R.row_life[s], (size_t)h->bufs.row_capacity[s]));
      CK(dalloc(h, &R.tab_ret[s], (size_t)h->B * P.n_possible[s]));
      CK(dalloc(h, &R.tab_life[s], (size_t)h->B * P.n_possible[s]));
    }
    R.env_flags = P.env_flags; R.env_step = P.env_step; R.B = h->B;
    CK(dalloc(h, &R.env_return, (size_t)h->B * 2));
    CK(dalloc(h, &R.env_valid, (size_t)h->B));
    CK(dalloc(h, &R.env_acc, (size_t)h->B * PPG_N_EP_STATS));
    CK(dalloc(h, &h->d_ep_partial, (size_t)episode_stats_partials(h->B) * PPG_N_EP_STATS));
    CK(dalloc(h, &h->d_ep_stats, PPG_N_EP_STATS));
    h->R_alloc = true;
    CK(launch_episode_stats_clear(R.env_acc, h->B, st));
    h->launch_count++;
  }
  if (!h->track_on) {
    CK(cudaMemsetAsync(R.env_valid, 0, (size_t)h->B, st));
    CK(cudaMemsetAsync(R.env_return, 0xFF, (size_t)h->B * 2 * sizeof(double), st));  // all-ones bits: NaN
  }
  h->track_on = true;
  return PPG_OK;
}

int ppg_get_returns(ppg_handle h, ppg_returns* out) {
  if (!h || !out) return PPG_ERR_INVALID;
  if (!h->track_on) { h->err = "ppg_get_returns: tracking is off (ppg_track_returns)"; return PPG_ERR_STATE; }
  for (int s = 0; s < 2; ++s) { out->row_return[s] = h->R.row_return[s]; out->row_life[s] = h->R.row_life[s]; }
  out->env_return = h->R.env_return; out->env_valid = h->R.env_valid; out->env_acc = h->R.env_acc;
  return PPG_OK;
}

int ppg_episode_stats_device(ppg_handle h, double** dev_out, void* cuda_stream) {
  if (!h || !dev_out) return PPG_ERR_INVALID;
  if (!h->R_alloc) { h->err = "ppg_episode_stats_device: tracking was never switched on (ppg_track_returns)"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  CK(launch_episode_stats(h->R.env_acc, h->R.env_valid, h->B, h->d_ep_partial, h->d_ep_stats, static_cast<cudaStream_t>(cuda_stream)));
  h->launch_count += 2;
  *dev_out = h->d_ep_stats;
  return PPG_OK;
}

int ppg_episode_stats_clear(ppg_handle h, void* cuda_stream) {
  if (!h) return PPG_ERR_INVALID;
  if (!h->R_alloc) { h->err = "ppg_episode_stats_clear: tracking was never switched on (ppg_track_returns)"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  CK(launch_episode_stats_clear(h->R.env_acc, h->B, static_cast<cudaStream_t>(cuda_stream)));
  h->launch_count++;
  return PPG_OK;
}

int ppg_world_state(ppg_handle h, int32_t env_begin, int32_t n_envs, float* out, void* cuda_stream) {
  if (!h) return PPG_ERR_INVALID;
  if (env_begin < 0 || n_envs < 1 || env_begin > h->B - n_envs) { h->err = "ppg_world_state: env range outside [0, n_envs)"; return PPG_ERR_INVALID; }
  if (!out) { h->err = "ppg_world_state: NULL out"; return PPG_ERR_INVALID; }
  const StepParams& P = h->P;
  if (!P.obs_split) { h->err = "ppg_world_state: the one-kernel step (PPG_OBS_SPLIT=0) keeps no env images"; return PPG_ERR_STATE; }
  switch (h->img) {
    case ppg_handle_s::IMG_NONE: h->err = "ppg_world_state: no output since ppg_create"; return PPG_ERR_STATE;
    case ppg_handle_s::IMG_RESTORED: h->err = "ppg_world_state: no output since ppg_restore"; return PPG_ERR_STATE;
    case ppg_handle_s::IMG_RESTORED_IDLE: h->err = "ppg_world_state: envs were restored idle; no full ppg_reset since"; return PPG_ERR_STATE;
    default: break;
  }
  CK(cudaSetDevice(h->device));
  WorldStateParams w;
  memset(&w, 0, sizeof w);
  w.img = P.obs_img; w.out = out; w.env_begin = env_begin; w.n_envs = n_envs;
  w.img_stride = P.img_stride; w.img_bytes = P.img_bytes;
  w.G = P.G; w.C = h->cfg.num_obs_channels; w.P = P.P; w.PS = P.PS;
  for (int c = 0; c < PPG_WS_SRC; ++c) {
    const ChannelSource src = channel_source(P, c < w.C ? c : w.C - 1);
    w.map_off[c] = src.map - P.so_img; w.tbl_off[c] = src.tbl - P.so_img;
  }
  for (int c = PPG_WS_SRC; c < w.C; ++c) {
    const ChannelSource src = channel_source(P, c);
    if (src.map - P.so_img != w.map_off[PPG_WS_SRC - 1] || src.tbl - P.so_img != w.tbl_off[PPG_WS_SRC - 1]) {
      h->err = "ppg_world_state: internal: channel sources past PPG_WS_SRC differ"; return PPG_ERR_STATE;
    }
  }
  if (h->n_cta_ws == 0) {
    int per_sm = 0, n_sm = 0;
    CK(world_state_occupancy(w, P.map_bytes, &per_sm));
    CK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, h->device));
    if (per_sm < 1) { h->err = "ppg_world_state: kernel does not fit on an SM"; return PPG_ERR_INVALID; }
    h->n_cta_ws = per_sm * n_sm;
  }
  CK(launch_world_state(w, P.map_bytes, std::min(n_envs, h->n_cta_ws), static_cast<cudaStream_t>(cuda_stream)));
  h->launch_count++;
  return PPG_OK;
}

int ppg_read_env(ppg_handle h, int32_t env, int32_t* n_live, int32_t* ids_pred, int32_t* xy_pred, double* energy_pred,
                 int32_t* ids_prey, int32_t* xy_prey, double* energy_prey, int32_t* xy_grass, double* energy_grass) {
  if (!h || env < 0 || env >= h->B || !n_live) return PPG_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  const StepParams& P = h->P;
  EnvHdr hd;
  CK(cudaMemcpy(&hd, P.hdr + env, sizeof hd, cudaMemcpyDeviceToHost));
  int32_t* ids[2] = {ids_pred, ids_prey};
  int32_t* xy[2] = {xy_pred, xy_prey};
  double* en[2] = {energy_pred, energy_prey};
  for (int s = 0; s < 2; ++s) {
    const int n = hd.n_list[s];
    n_live[s] = n;
    std::vector<uint16_t> id(std::max(n, 1)), pos(std::max(n, 1));
    std::vector<double> e(std::max(n, 1));
    const size_t b = (size_t)env * P.cap[s];
    if (n) {
      CK(cudaMemcpy(id.data(), P.ag_id[s] + b, n * 2, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(pos.data(), P.ag_pos[s] + b, n * 2, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(e.data(), P.ag_e[s] + b, n * 8, cudaMemcpyDeviceToHost));
    }
    // report in agent_positions insertion order = ascending id (BASE:190-200,401)
    std::vector<int> order(n);
    for (int i = 0; i < n; ++i) order[i] = i;
    if (P.variant != PPG_VARIANT_STAG)  // STAG: the device list already is in insertion order (flat ids are not monotonic)
      std::sort(order.begin(), order.end(), [&](int a, int b2) { return id[a] < id[b2]; });
    for (int i = 0; i < n; ++i) {
      const int j = order[i];
      if (ids[s]) ids[s][i] = id[j];
      if (xy[s]) { xy[s][2 * i] = pos[j] >> 8; xy[s][2 * i + 1] = pos[j] & 255; }
      if (en[s]) en[s][i] = e[j];
    }
  }
  const int ng = P.n_grass;
  if (ng) {
    std::vector<uint16_t> gp(ng);
    std::vector<double> ge(ng);
    CK(cudaMemcpy(gp.data(), P.gr_pos + (size_t)env * ng, ng * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ge.data(), P.gr_e + (size_t)env * ng, ng * 8, cudaMemcpyDeviceToHost));
    for (int g = 0; g < ng; ++g) {
      if (xy_grass) { xy_grass[2 * g] = gp[g] >> 8; xy_grass[2 * g + 1] = gp[g] & 255; }
      if (energy_grass) energy_grass[g] = ge[g];
    }
  }
  return PPG_OK;
}

int ppg_read_env_eco(ppg_handle h, int32_t env, int32_t* age_pred, double* speed_pred, int32_t* age_prey, double* speed_prey,
                     uint8_t* dead_prey, int32_t* active_num) {
  if (!h || env < 0 || env >= h->B) return PPG_ERR_INVALID;
  if (h->P.variant != PPG_VARIANT_ECO) { h->err = "ppg_read_env_eco: not an ECO handle"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  const StepParams& P = h->P;
  EnvHdr hd;
  EcoHdr eh;
  CK(cudaMemcpy(&hd, P.hdr + env, sizeof hd, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&eh, P.ehdr + env, sizeof eh, cudaMemcpyDeviceToHost));
  int32_t* age[2] = {age_pred, age_prey};
  double* sp[2] = {speed_pred, speed_prey};
  for (int s = 0; s < 2; ++s) {  // the device list is in ascending id order = the order of ppg_read_env
    const int n = hd.n_list[s];
    if (!n) continue;
    std::vector<uint16_t> a(n);
    std::vector<double> v(n);
    std::vector<uint8_t> d(n);
    const size_t b = (size_t)env * P.cap[s];
    CK(cudaMemcpy(a.data(), P.ag_age[s] + b, n * 2, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(v.data(), P.ag_spd[s] + b, n * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(d.data(), P.ag_dead[s] + b, n, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
      if (age[s]) age[s][i] = a[i];
      if (sp[s]) sp[s][i] = v[i];
      if (s == 1 && dead_prey) dead_prey[i] = d[i];
    }
  }
  if (active_num) { active_num[0] = eh.active[0]; active_num[1] = eh.active[1]; }
  return PPG_OK;
}

int ppg_read_env_acc(ppg_handle h, int32_t env, double* acc_pred, double* acc_prey) {
  if (!h || env < 0 || env >= h->B) return PPG_ERR_INVALID;
  if (h->P.variant != PPG_VARIANT_ECO || h->P.trait_mode != PPG_TRAIT_CADENCE) { h->err = "ppg_read_env_acc: not a cadence handle"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  EnvHdr hd;
  CK(cudaMemcpy(&hd, h->P.hdr + env, sizeof hd, cudaMemcpyDeviceToHost));
  double* out[2] = {acc_pred, acc_prey};
  for (int s = 0; s < 2; ++s)
    if (hd.n_list[s] && out[s]) CK(cudaMemcpy(out[s], h->P.ag_acc[s] + (size_t)env * h->P.cap[s], sizeof(double) * hd.n_list[s], cudaMemcpyDeviceToHost));
  return PPG_OK;
}

int ppg_read_episode_eco(ppg_handle h, int32_t env, double* sums, int32_t* spawned) {
  if (!h || env < 0 || env >= h->B) return PPG_ERR_INVALID;
  if (h->P.variant != PPG_VARIANT_ECO || !h->P.ep_sums) { h->err = "ppg_read_episode_eco: needs an ECO handle created with track_episode_sums"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  EnvHdr hd;
  CK(cudaMemcpy(&hd, h->P.hdr + env, sizeof hd, cudaMemcpyDeviceToHost));
  if (sums) CK(cudaMemcpy(sums, h->P.ep_sums + (size_t)env * PPG_EP_STRIDE, 4 * sizeof(double), cudaMemcpyDeviceToHost));
  // ids are handed out in order and never reused (ECO:260-272): spawned = ids used - founders of the running episode
  const bool rf = ppg_random_founders(h->P.trait_mode);
  if (spawned) for (int s = 0; s < 2; ++s) spawned[s] = (int32_t)hd.next_idx[s] - (rf ? (s == 0 ? (hd.pad[1] & 0xFFFF) : ((hd.pad[1] >> 16) & 0x7FFF)) : h->P.n_init[s]);
  return PPG_OK;
}

int ppg_read_episode_events_eco(ppg_handle h, int32_t env, double* events) {
  if (!h || env < 0 || env >= h->B || !events) return PPG_ERR_INVALID;
  if (h->P.variant != PPG_VARIANT_ECO || !h->P.ep_sums) { h->err = "ppg_read_episode_events_eco: needs an ECO handle created with track_episode_sums"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(events, h->P.ep_sums + (size_t)env * PPG_EP_STRIDE + PPG_EP_BLOCKED_CAPACITY, 6 * sizeof(double), cudaMemcpyDeviceToHost));
  return PPG_OK;
}

int ppg_read_env_stag(ppg_handle h, int32_t env, int32_t* age_pred, int32_t* facing_pred, double* trait_pred, int32_t* age_prey,
                      int64_t* capture, double* capture_real) {
  if (!h || env < 0 || env >= h->B) return PPG_ERR_INVALID;
  if (h->P.variant != PPG_VARIANT_STAG) { h->err = "ppg_read_env_stag: not a STAG handle"; return PPG_ERR_STATE; }
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceSynchronize());
  const StepParams& P = h->P;
  EnvHdr hd;
  StagHdr sh;
  CK(cudaMemcpy(&hd, P.hdr + env, sizeof hd, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(&sh, P.shdr + env, sizeof sh, cudaMemcpyDeviceToHost));
  int32_t* age[2] = {age_pred, age_prey};
  for (int s = 0; s < 2; ++s) {  // the device list is in insertion order = the order of ppg_read_env
    const int n = hd.n_list[s];
    if (!n) continue;
    std::vector<uint16_t> a(n);
    const size_t b = (size_t)env * P.cap[s];
    CK(cudaMemcpy(a.data(), P.ag_age[s] + b, n * 2, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i)
      if (age[s]) age[s][i] = a[i];
    if (s == 0) {
      std::vector<uint8_t> f(n);
      std::vector<double> t(n);
      CK(cudaMemcpy(f.data(), P.ag_face + b, n, cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(t.data(), P.ag_trait + b, n * 8, cudaMemcpyDeviceToHost));
      for (int i = 0; i < n; ++i) {
        if (facing_pred) facing_pred[i] = f[i];
        if (trait_pred) trait_pred[i] = t[i];
      }
    }
  }
  if (capture) for (int k = 0; k < 12; ++k) capture[k] = sh.capture[k];
  if (capture_real) for (int k = 0; k < 3; ++k) capture_real[k] = sh.capture_real[k];
  return PPG_OK;
}

int ppg_stats_device(ppg_handle h, int64_t** dev_out, void* cuda_stream) {
  if (!h || !dev_out) return PPG_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaSetDevice(h->device));
  CK(cudaMemsetAsync(h->d_stats, 0, sizeof(unsigned long long) * PPG_N_STATS, st));
  CK(launch_stats(h->P.counters, h->P.hdr, h->B, h->d_stats, st));
  h->launch_count++;
  *dev_out = reinterpret_cast<int64_t*>(h->d_stats);
  return PPG_OK;
}

int ppg_stats(ppg_handle h, int64_t* out, void* cuda_stream) {
  if (!h || !out) return PPG_ERR_INVALID;
  int64_t* d = nullptr;
  int rc = ppg_stats_device(h, &d, cuda_stream);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaMemcpyAsync(out, d, sizeof(int64_t) * PPG_N_STATS, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  unsigned err = 0;
  CK(cudaMemcpy(&err, h->P.error, sizeof err, cudaMemcpyDeviceToHost));
  if (err) { h->err = "device error word set (row allocation: bit0 prefix wait wedged, bit1 stale counts)"; return PPG_ERR_STATE; }
  return PPG_OK;
}

int ppg_stats_clear(ppg_handle h, void* cuda_stream) {
  if (!h) return PPG_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  CK(cudaMemsetAsync(h->P.counters, 0, (size_t)h->B * PPG_N_STATS * sizeof(uint32_t), static_cast<cudaStream_t>(cuda_stream)));
  return PPG_OK;
}

int64_t ppg_launch_count(ppg_handle h) { return h ? h->launch_count : 0; }

int ppg_profile_env_cycles(ppg_handle h, uint32_t* cycles, uint32_t* info, uint32_t* start_ns, uint32_t* sm, void* cuda_stream) {
  if (!h || !cycles) return PPG_ERR_INVALID;
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CK(cudaSetDevice(h->device));
  std::vector<uint4> tmp((size_t)h->B);
  CK(cudaMemcpyAsync(tmp.data(), h->P.env_cycles, sizeof(uint4) * (size_t)h->B, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int e = 0; e < h->B; ++e) {
    cycles[e] = tmp[(size_t)e].x;
    if (info) info[e] = tmp[(size_t)e].y;
    if (start_ns) start_ns[e] = tmp[(size_t)e].z;
    if (sm) sm[e] = tmp[(size_t)e].w;
  }
  return PPG_OK;
}

int ppg_profile_begin(ppg_handle h) {
  if (!h) return PPG_ERR_INVALID;
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  h->prof_events.clear();
  h->profiling = true;
  return PPG_OK;
}

int ppg_profile_end(ppg_handle h, double* ms_step_kernel, double* ms_obs_kernel, int32_t* n_steps) {
  if (!h) return PPG_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  h->profiling = false;
  double a = 0.0, b = 0.0;
  const size_t n = h->prof_events.size() / 3;
  for (size_t i = 0; i < n; ++i) {
    CK(cudaEventSynchronize(h->prof_events[3 * i + 2]));
    float x = 0.f, y = 0.f;
    CK(cudaEventElapsedTime(&x, h->prof_events[3 * i], h->prof_events[3 * i + 1]));
    CK(cudaEventElapsedTime(&y, h->prof_events[3 * i + 1], h->prof_events[3 * i + 2]));
    a += x; b += y;
  }
  for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
  h->prof_events.clear();
  if (ms_step_kernel) *ms_step_kernel = a;
  if (ms_obs_kernel) *ms_obs_kernel = b;
  if (n_steps) *n_steps = (int32_t)n;
  return PPG_OK;
}

}  // extern "C"
