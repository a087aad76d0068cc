// ppg_base.cu — the BASE-family environment step as one fused, persistent sm_100a kernel (v4).
//
// Reproduces, for B independent env instances in lockstep, `PredPreyGrass.step()` and `reset()` of
//   BASE = predpreygrass/non_evolutionary/base_environment/predpreygrass_rllib_env.py
// and its reward variants (dense_rewards, dense_rewards_additive, sparse_rewards_plus_eating,
// sparse_rewards_plus_kickback; see include/ppg.h PPG_REWARD_*).
//
// Mapping: one warp owns one env for the whole step; warps are persistent and draw env indices
// from a global ticket counter, so envs of very different population sizes balance over the SMs.
// The env's agent lists, grass and three small index MAPS live in the warp's slice of shared
// memory.  The reference's float grid (`grid_world_state`, BASE:124) is never materialised: a
// non-zero grid cell always equals the current energy of the agent that wrote it last, so
// `map[s][cell] = slot + 1` (0 = the reference wrote 0 there) carries the same information in one
// byte per cell, and `map[2][cell] = grass index + 1`.  The maps have a halo as wide as the largest
// observation window (index(x,y) = P + (x+P)*PS + y, the gap after a row doubles as the next row's
// left halo), so a window element is `map[index(agent) + const]` with no bounds test; the halo of
// the predator map holds a WALL index, which makes channel 0 ("outside the grid", BASE:522-523)
// just another table lookup.
//
// Order-dependent phases keep the reference's semantics but run lane-parallel wherever agents
// cannot interact:
//   movement (dict order, BASE:259-273): chunks of 32 agents; an agent whose old or target cell
//     is touched by any other agent of the chunk is replayed sequentially in order, the rest
//     commit in parallel (ordered-claim round with shared-memory touch counters);
//   predators (BASE:279-346): skipped entirely when no predator starved and no prey shares a
//     cell with a predator, else the exact sequential loop;
//   prey (BASE:347-380): 32 prey at a time eat in parallel unless one of them starved or two
//     share a grass patch, else the exact sequential loop for that chunk;
//   births (BASE:389-448): ballot over eligible parents, sequential per birth (rare).
// Observation rows (BASE:511-539): lane l produces elements l, l+32, ... of the [C][R][R] row, each
// by two dependent shared-memory loads (map entry -> fp32 value table) at per-lane constant offsets,
// conflict-free, into a staging row that leaves the SM as ONE bulk asynchronous copy
// (cp.async.bulk shared -> global, 784 / 1296 contiguous bytes), double buffered so gathering row
// r+1 overlaps the store of row r.
//
// Row allocation across envs is deterministic and needs no second kernel: every env publishes
// its live/birth counts; the last finisher of each 32-env block / 1024-env group publishes block
// and group sums (threadfence + counter pattern).  An env derives the first row of its old rows
// from the PREVIOUS launch's sums (complete by construction) and the first row of its newborn
// rows from THIS launch's sums, which it only waits for if it has newborns, after all its other
// work is done.
#include <cuda_runtime.h>

#include "ppg_step_common.cuh"

#ifndef PPG_MIN_CTAS
#define PPG_MIN_CTAS 20  // resident step warps per SM the register allocation is sized for
#endif

namespace ppg {

PHASE_DEFINE(base)
SPAN_DEFINE(base)

// ------------------------------------------------------------------------------------------------
// the step kernel: W persistent warps per CTA, one env per warp at a time
// ------------------------------------------------------------------------------------------------
#define SEL(a) (s == 0 ? a[0] : a[1])

template <int W, typename MapT, bool BULK, bool SPLIT>
__global__ void __launch_bounds__(W * 32, PPG_MIN_CTAS / W) ppg_step_base_kernel(const __grid_constant__ StepParams p) {  // PHASE: kernel prologue
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ int s_env0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  SPAN_MARK(base, 0)
  wait_for_stream_predecessor();  // PDL chain: this grid may have become resident under the tail of the kernel before it
  if (SPLIT) allow_dependent_launch();  // the observation kernel may start filling the SMs' free slots right away
  unsigned char* const sbase = smem_raw + (size_t)warp * p.smem_per_env;
  const EnvSmem<MapT> S = carve<MapT>(sbase, p);
  const RowDesc D = carve_desc(sbase, p);
  const unsigned sb32 = (unsigned)__cvta_generic_to_shared(sbase);
  const int G = p.G, GG = p.GG, PP = p.P, PS = p.PS;
  const int mode_r = p.reward_mode;
  const bool dense = mode_r == PPG_REWARD_DENSE || mode_r == PPG_REWARD_DENSE_ADDITIVE;
  const bool kick = mode_r == PPG_REWARD_SPARSE_KICKBACK;
  const unsigned lt_mask = (1u << lane) - 1u;

  // one-time set-up of this warp's slice: empty maps (predator map: WALL outside the field), zeroed touch
  // counters, wall table — copied from the image ppg_create built.  Every env leaves the maps empty again
  // (it un-writes the cells it wrote).
  {
    const int n16 = p.init_bytes / 16;
    #pragma unroll 1
    for (int i0 = 0; i0 < n16; i0 += 32 * 8) {  // 8 loads in flight per lane: one round trip per 4 KB, not per 512 B
      uint4 v[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) { const int i = i0 + 32 * q + lane; if (i < n16) v[q] = __ldg(reinterpret_cast<const uint4*>(p.init_image) + i); }
#pragma unroll
      for (int q = 0; q < 8; ++q) { const int i = i0 + 32 * q + lane; if (i < n16) reinterpret_cast<uint4*>(sbase + p.so_map[0])[i] = v[q]; }
    }
  }
  unsigned rowctr = 0;
  EnvLoop L = env_loop(p, SPLIT);  // SPLIT exists for W == 1 only
  __syncwarp();

  // W == 1: envs come from the ticket counter (EnvLoop)
  if (W == 1 && lane == 0) next_ticket(p, L, true);
  SPAN_MARK(base, 1)
  for (;;) {
    PHASE_DECL
    int env = 0;  // PHASE: ticket+hdr
    if (W == 1) {
      env = __shfl_sync(FULL, L.env_next, 0);
      if (env >= p.B) break;
    } else {
      // the W warps of a CTA take W consecutive envs and start them together: warps of one CTA then run the
      // same code at about the same time, which keeps the instruction cache warm (the kernel is far larger
      // than the cache and every env walks through most of it once)
      __syncthreads();
      if (threadIdx.x == 0) s_env0 = (int)(atomicAdd(p.ticket, 1ULL) - p.ticket_base) * W;
      __syncthreads();
      if (s_env0 >= p.B) break;
      env = s_env0 + warp;
      if (env >= p.B) continue;
    }

    // per-env registers (warp-uniform)
    int n[2] = {0, 0};  // list length at step start (= old rows)
    int births[2] = {0, 0};
    int old_base[2] = {0, 0};
    int next_live[2] = {0, 0};
    int mode = 0;  // 0 idle, 1 reset, 2 step
    unsigned env_flags = 0;
    EnvStats st = {};
    int cur[2] = {0, 0};
    bool over = false, trunc = false;

    PHASE_MARK(0)
    const long long t_env0 = clock64();
    const unsigned t_ns0 = globaltimer_lo();
    // ONE round trip for everything the env needs from HBM/L2: the header, the prefix words, the first entries of both
    // agent lists (speculatively: how many are valid is in the header) and the grass patches are all requested before any
    // of them is looked at; under the observation kernel's write stream a round trip costs microseconds, so the number of
    // DEPENDENT round trips per env is what the step kernel's duration is made of.
    EnvHdr h = p.hdr[env];
    int prow_r[3] = {0, 0, 0};
    double e_r[3] = {0.0, 0.0, 0.0};
    unsigned idpos_r[3] = {0, 0, 0}, par_r[3] = {0, 0, 0};
#pragma unroll
    for (int q = 0; q < 3; ++q) {  // q = 0: predators 0..31, q = 1, 2: prey 0..63
      const int s = q ? 1 : 0, i = lane + (q == 2 ? 32 : 0);
      if (i < p.cap[s]) {
        const size_t b = (size_t)env * p.cap[s] + i;
        prow_r[q] = p.ag_prow[s][b];
        e_r[q] = p.ag_e[s][b];
        idpos_r[q] = (unsigned)p.ag_id[s][b] | ((unsigned)p.ag_pos[s][b] << 16);
        if (kick) par_r[q] = p.ag_par[s][b];
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
    PHASE_MARK(1)

    if (PPG_UNLIKELY(mode == 1)) {  // PHASE: reset
      // ------------------------------------------------------------------ reset() (BASE:129-217)
      h.episode += 1;
      h.step = 0;
      h.spawn_draws = 0;
      h.status = 0;
      h.sortflag = 0;
      h.first_step = 1;
      h.state = 0;
      const int n_total = p.n_init[0] + p.n_init[1] + p.n_grass;
      // cells in the order predators, prey, grass (BASE:185-187)
      int* cells = reinterpret_cast<int*>(S.vt[0]);          // [n_total], in the value tables (rebuilt before every use)
      unsigned* first = reinterpret_cast<unsigned*>(S.E[0]);  // [GG] draw index that claimed the cell; dead before E is written
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
      if (!from_tape) philox_placement(cells, first, n_total, GG, (unsigned)(env + p.env_base), h.episode, h.seed_key, lane);
      __syncwarp();
      // founders: slots in numeric id order (BASE:143-145,190-200)
      {
        int k0 = 0;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          #pragma unroll 1
          for (int i = lane; i < p.n_init[s]; i += 32) {
            const int c = cells[k0 + i];
            const int cx = c / G, cy = c % G;
            S.id[s][i] = (uint16_t)i;
            S.pos[s][i] = (uint16_t)((cx << 8) | cy);
            S.E[s][i] = p.init_e[s];
            S.flg[s][i] = F_ALIVE;
            if (kick) S.par[s][i] = 0xFFFF;
            S.ord[s][i] = (uint16_t)i;
            S.map[s][CELLXY(cx, cy)] = (MapT)(i + 1);  // BASE:195,200 (cells are unique)
          }
          k0 += p.n_init[s];
          n[s] = p.n_init[s];
          h.n_list[s] = (unsigned short)p.n_init[s];
          h.n_sorted[s] = (unsigned short)p.n_init[s];
          h.next_idx[s] = (unsigned short)p.n_init[s];
        }
        #pragma unroll 1
        for (int g = lane; g < p.n_grass; g += 32) {
          const int c = cells[k0 + g];
          const int cx = c / G, cy = c % G;
          S.gpos[g] = (uint16_t)((cx << 8) | cy);
          S.gE[g] = p.grass_cap;  // BASE:203-208
          S.map[2][CELLXY(cx, cy)] = (MapT)(g + 1);
        }
      }
      __syncwarp();
      cur[0] = n[0]; cur[1] = n[1];
      next_live[0] = n[0]; next_live[1] = n[1];
      env_flags = PPG_ENV_RESET;
      PHASE_MARK(2)
    } else if (mode == 2) {
      // ------------------------------------------------------------------ step() (BASE:219-473)
      n[0] = h.n_list[0]; n[1] = h.n_list[1];  // PHASE: load+decay+maps
      // second (and last) dependent round trip: the actions of the rows the agents occupied in the previous output
      int act_r[3] = {4, 4, 4};
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int s = q ? 1 : 0, i = lane + (q == 2 ? 32 : 0);
        if (i < SEL(n)) act_r[q] = p.actions[s][prow_r[q]];
      }
      // meanwhile: grass regrowth (BASE:252-256) from the registers
      {
        // base_environment_seasonal: square-wave multiplier on the regrowth, phase from the step counter (SEASON:224-234)
        const double grass_gain = p.season_len > 0 ? p.grass_gain_season[(h.step / p.season_len) & 1] : p.grass_gain;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int g = lane + 32 * q;
          if (g < p.n_grass) {
            S.gpos[g] = (uint16_t)gp_r[q];
            const double v = ge_r[q] + grass_gain;
            S.gE[g] = v < p.grass_cap ? v : p.grass_cap;
            S.map[2][CELLP(gp_r[q])] = (MapT)(g + 1);
          }
        }
        #pragma unroll 1
        for (int g = lane + 128; g < p.n_grass; g += 32) {  // more than 128 patches: the rest the plain way
          const size_t b = (size_t)env * p.n_grass;
          const unsigned gp = p.gr_pos[b + g];
          S.gpos[g] = (uint16_t)gp;
          const double v = p.gr_e[b + g] + grass_gain;
          S.gE[g] = v < p.grass_cap ? v : p.grass_cap;
          S.map[2][CELLP(gp)] = (MapT)(g + 1);
        }
      }
      PHASE_MARK(4)
      // the lists; list order = action-dict order (default: row order of the previous output)
      unsigned bad = 0;
      bool resort[2] = {false, false};
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        const size_t b = (size_t)env * p.cap[s];
        const int32_t* ordp = p.order[s];
        bool use_order = ordp != nullptr;
        if (PPG_UNLIKELY(use_order)) {  // must be a permutation of [0, n) (ppg_step_ordered); else fall back to row order
          bool ok = true;
          #pragma unroll 1
          for (int i = lane; i < SEL(n); i += 32) {
            const int d = ordp[p.ag_prow[s][b + i]];
            if ((unsigned)d < (unsigned)SEL(n)) SEL(S.rnk)[d] = (uint16_t)i; else ok = false;
          }
          __syncwarp();
          #pragma unroll 1
          for (int i = lane; i < SEL(n); i += 32) {
            const int d = ordp[p.ag_prow[s][b + i]];
            if ((unsigned)d < (unsigned)SEL(n)) ok &= SEL(S.rnk)[d] == (uint16_t)i;
          }
          use_order = __all_sync(FULL, ok);
          if (!use_order) bad = PPG_STATUS_BAD_ACTION;
          __syncwarp();
        }
        if (s == 0) resort[0] = use_order; else resort[1] = use_order;
        #pragma unroll 1
        for (int i = lane; i < SEL(n); i += 32) {
          // entries 0..31 (predators) / 0..63 (prey) are already in registers, with their actions
          const int q = s == 0 ? (i < 32 ? 0 : 3) : (i < 32 ? 1 : (i < 64 ? 2 : 3));
          int prow, a;
          double e;
          unsigned idpos, par16 = 0;
          if (q < 3) {
            prow = q == 0 ? prow_r[0] : (q == 1 ? prow_r[1] : prow_r[2]);
            e = q == 0 ? e_r[0] : (q == 1 ? e_r[1] : e_r[2]);
            idpos = q == 0 ? idpos_r[0] : (q == 1 ? idpos_r[1] : idpos_r[2]);
            a = q == 0 ? act_r[0] : (q == 1 ? act_r[1] : act_r[2]);
            if (kick) par16 = q == 0 ? par_r[0] : (q == 1 ? par_r[1] : par_r[2]);
          } else {
            prow = p.ag_prow[s][b + i];
            e = p.ag_e[s][b + i];
            idpos = (unsigned)p.ag_id[s][b + i] | ((unsigned)p.ag_pos[s][b + i] << 16);
            a = p.actions[s][prow];
            if (kick) par16 = p.ag_par[s][b + i];
          }
          const int d = use_order ? ordp[prow] : i;
          if ((unsigned)a > 8u) { a = 4; bad = PPG_STATUS_BAD_ACTION; }  // reference: KeyError BASE:502
          SEL(S.id)[d] = (uint16_t)idpos;
          SEL(S.pos)[d] = (uint16_t)(idpos >> 16);
          if (dense) SEL(S.E0)[d] = e;  // energy_before (ADD:256)
          SEL(S.E)[d] = e - p.loss[s];  // Step 1 (BASE:244-250)
          SEL(S.act)[d] = (uint8_t)a;
          SEL(S.flg)[d] = F_ALIVE;
          SEL(S.ord)[d] = (uint16_t)d;
          SEL(S.rnk)[d] = (uint16_t)d;
          if (kick) { SEL(S.par)[d] = (uint16_t)par16; SEL(S.aux)[d] = 0; }
        }
      }
      h.status |= (unsigned char)__reduce_or_sync(FULL, bad);
      PHASE_MARK(3)
      __syncwarp();
      // owner maps as the grid stands after Step 1: of agents sharing a cell the one latest in dict
      // order wrote last (BASE:247,250)
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
      PHASE_MARK(5)

      // Step 2: movements, sequential semantics in dict order per species (BASE:259-273,495-509)  // PHASE: movement
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        MapT* own = SEL(S.map);
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int j = b0 + lane;
          const bool v = j < SEL(n);
          int oc = 0, tc = 0, nx0 = 0, ny0 = 0;
          if (v) {
            const unsigned ps = SEL(S.pos)[j];
            const int a = SEL(S.act)[j];
            const int x = ps >> 8, y = ps & 255;
            const int ax = (a * 11) >> 5;  // a / 3 for 0 <= a <= 8
            nx0 = min(max(x + ax - 1, 0), G - 1); ny0 = min(max(y + (a - 3 * ax) - 1, 0), G - 1);
            oc = CELLXY(x, y); tc = CELLXY(nx0, ny0);
            red_shared_add(reinterpret_cast<unsigned*>(S.scr) + (oc >> 2), 1u << ((oc & 3) * 8));
            if (tc != oc) red_shared_add(reinterpret_cast<unsigned*>(S.scr) + (tc >> 2), 1u << ((tc & 3) * 8));
          }
          __syncwarp();
          const bool dirty = v && (S.scr[oc] > 1 || S.scr[tc] > 1);
          __syncwarp();
          if (v) { S.scr[oc] = 0; S.scr[tc] = 0; }
          if (v && !dirty) {
            // nobody else in this chunk touches my cells: the outcome does not depend on the order
            const unsigned ow = own[tc];
            const bool blocked = ow != 0 && SEL(S.E)[ow - 1] > 0.0;  // own-species channel occupied (BASE:506)
            const int nc = blocked ? oc : tc;
            own[oc] = 0;               // BASE:268,272
            own[nc] = (MapT)(j + 1);   // BASE:269,273
            if (!blocked) SEL(S.pos)[j] = (uint16_t)((nx0 << 8) | ny0);
          }
          __syncwarp();
          unsigned dm = __ballot_sync(FULL, dirty);
          while (dm) {  // warp-uniform replay, in dict order, of the agents that may interact
            const int jj = b0 + __ffs(dm) - 1;
            dm &= dm - 1;
            const unsigned ps = SEL(S.pos)[jj];
            const int a = SEL(S.act)[jj];
            const int xx = ps >> 8, yy = ps & 255;
            const int ax = (a * 11) >> 5;
            const int tx = min(max(xx + ax - 1, 0), G - 1), ty = min(max(yy + (a - 3 * ax) - 1, 0), G - 1);
            const unsigned ow = own[CELLXY(tx, ty)];
            const bool blocked = ow != 0 && SEL(S.E)[ow - 1] > 0.0;
            const int nx = blocked ? xx : tx, ny = blocked ? yy : ty;
            __syncwarp();
            if (lane == 0) {  // one writer: the two map stores may hit the same cell (blocked move) and must keep their order
              own[CELLXY(xx, yy)] = 0;
              own[CELLXY(nx, ny)] = (MapT)(jj + 1);
              SEL(S.pos)[jj] = (uint16_t)((nx << 8) | ny);
            }
            __syncwarp();
          }
        }
      }

      PHASE_MARK(6)
      // deferred `self.agents.sort()` of the previous call (BASE:468): engagement order.  The list is  // PHASE: sort
      // the sorted survivors followed by last step's newborns, so only the newborns have to be ranked in.
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        if (SEL(resort) || (h.sortflag & (1 << s))) {
          const uint16_t* lr = p.lexrank[s];
          const bool by_id = h.first_step != 0;  // right after reset() self.agents is in numeric order (BASE:143-145)
          const int ns = SEL(resort) ? 0 : min((int)(s == 0 ? h.n_sorted[0] : h.n_sorted[1]), SEL(n));
          #pragma unroll 1
          for (int i = lane; i < SEL(n); i += 32) SEL(S.ord)[i] = by_id ? SEL(S.id)[i] : __ldg(lr + SEL(S.id)[i]);
          __syncwarp();
          #pragma unroll 1
          for (int i = lane; i < SEL(n); i += 32) {
            const unsigned key = SEL(S.ord)[i];
            int r = i < ns ? i : 0;
            for (int k = (i < ns ? ns : 0); k < SEL(n); ++k) r += SEL(S.ord)[k] < key;
            SEL(S.rnk)[i] = (uint16_t)r;
          }
          __syncwarp();
          #pragma unroll 1
          for (int i = lane; i < SEL(n); i += 32) SEL(S.ord)[SEL(S.rnk)[i]] = (uint16_t)i;
          __syncwarp();
        }
      }

      PHASE_MARK(7)
      // Step 3a: predators in engagement order (BASE:279-346).  Nothing happens unless a predator  // PHASE: predators
      // starved or some prey (any energy) stands on a live predator's cell.
      // Only predators that starved or share their cell with a prey do anything (the others keep their step reward), and
      // what one predator does can only remove prey from later ones: the candidates are found lane-parallel (prey cells
      // marked in the touch counters) and only they run the sequential loop, in engagement order.
      bool vt_valid = false;  // value tables current (refreshed once, then kept up to date entry by entry)
      #pragma unroll 1
      for (int i = lane; i < n[1]; i += 32) S.scr[CELLP((unsigned)S.pos[1][i])] = 1;
      __syncwarp();
      for (int b0 = 0; b0 < n[0]; b0 += 32) {
        bool evk = false;
        if (b0 + lane < n[0]) {
          const int sl = S.ord[0][b0 + lane];
          evk = S.E[0][sl] <= 0.0 || S.scr[CELLP((unsigned)S.pos[0][sl])] != 0;
        }
        unsigned evm = __ballot_sync(FULL, evk);
        while (evm) {
          const int k = b0 + __ffs(evm) - 1;
          evm &= evm - 1;
          const int slot = S.ord[0][k];
          const unsigned ps = S.pos[0][slot];
          const int cell = CELLP(ps);
          double e = S.E[0][slot];
          if (e <= 0.0) {  // starved (BASE:284-301): observation as of now
            rowctr = emit_row_now<MapT, BULK>(sbase, p, p.obs[0] + (size_t)(old_base[0] + k) * p.elems[0], cell, 0, vt_valid ? -1 : n[0], n[1], rowctr, lane);
            vt_valid = true;
            if (lane == 0) {
              S.map[0][cell] = 0;  // BASE:293
              S.flg[0][slot] = F_DIED;
            }
            st.starved[0]++;
            __syncwarp();
            continue;
          }
          // first prey in agent_positions order (= lowest id) on my cell (BASE:305-312)
          unsigned best = 0xFFFFFFFFu;
          #pragma unroll 1
          for (int i = lane; i < n[1]; i += 32)
            if ((S.flg[1][i] & F_ALIVE) && S.pos[1][i] == ps) best = min(best, ((unsigned)S.id[1][i] << 16) | (unsigned)i);
          best = __reduce_min_sync(FULL, best);
          if (best != 0xFFFFFFFFu) {
            const int q = best & 0xFFFF;
            e += S.E[1][q];  // BASE:324 (also when the prey's energy is <= 0)
            __syncwarp();
            if (lane == 0) {
              S.E[0][slot] = e;
              if (vt_valid) S.vt[0][1 + slot] = (float)e;
              S.map[0][cell] = (MapT)(slot + 1);  // BASE:325
              S.flg[0][slot] |= F_ATE;
            }
            __syncwarp();
            rowctr = emit_row_now<MapT, BULK>(sbase, p, p.obs[1] + (size_t)(old_base[1] + S.rnk[1][q]) * p.elems[1], cell, 1, vt_valid ? -1 : n[0], n[1], rowctr, lane);  // BASE:327
            vt_valid = true;
            if (lane == 0) {
              S.map[1][cell] = 0;  // BASE:335
              S.flg[1][q] = F_DIED | F_CAUGHT;
            }
            st.eaten++;
            __syncwarp();
          }
        }
      }
      __syncwarp();  // every lane's candidate reads of the marks are done
      #pragma unroll 1
      for (int i = lane; i < n[1]; i += 32) S.scr[CELLP((unsigned)S.pos[1][i])] = 0;
      __syncwarp();

      PHASE_MARK(8)
      // Step 3b: prey in engagement order (BASE:347-380)  // PHASE: prey
      for (int b0 = 0; b0 < n[1]; b0 += 32) {
        const int k = b0 + lane;
        int slot = 0, cell = 0, g = 0;
        bool alive = false, starved = false;
        double e = 0.0;
        if (k < n[1]) {
          slot = S.ord[1][k];
          alive = (S.flg[1][slot] & F_ALIVE) != 0;  // not caught above (BASE:281)
          e = S.E[1][slot];
          starved = alive && e <= 0.0;
          cell = CELLP((unsigned)S.pos[1][slot]);
          g = S.map[2][cell];
        }
        const bool eat = alive && !starved && g != 0;
        if (eat) S.gtag[g - 1] = (uint8_t)lane;
        __syncwarp();
        const bool clash = eat && S.gtag[g - 1] != (uint8_t)lane;  // two prey of this chunk on one patch
        if (!__any_sync(FULL, starved || clash)) {
          if (eat) {  // BASE:351-372 (a patch with energy 0 is still "eaten")
            const double en = e + S.gE[g - 1];
            S.E[1][slot] = en;
            S.map[1][cell] = (MapT)(slot + 1);
            S.gE[g - 1] = 0.0;
            S.flg[1][slot] |= F_ATE;
            if (vt_valid) { S.vt[1][1 + slot] = (float)en; S.vt[2][g] = 0.f; }
          }
          st.grass += __popc(__ballot_sync(FULL, eat));
          __syncwarp();
          continue;
        }
        __syncwarp();
        const int kend = min(b0 + 32, n[1]);
        for (int kk = b0; kk < kend; ++kk) {  // exact sequential order for this chunk
          const int sl = S.ord[1][kk];
          if (!(S.flg[1][sl] & F_ALIVE)) continue;
          const int cl = CELLP((unsigned)S.pos[1][sl]);
          const double ee = S.E[1][sl];
          if (ee <= 0.0) {  // BASE:284-301
            rowctr = emit_row_now<MapT, BULK>(sbase, p, p.obs[1] + (size_t)(old_base[1] + kk) * p.elems[1], cl, 1, vt_valid ? -1 : n[0], n[1], rowctr, lane);
            vt_valid = true;
            if (lane == 0) {
              S.map[1][cl] = 0;
              S.flg[1][sl] = F_DIED;
            }
            st.starved[1]++;
            __syncwarp();
            continue;
          }
          const int gg = S.map[2][cl];
          if (gg) {
            const double en = ee + S.gE[gg - 1];
            __syncwarp();
            if (lane == 0) {
              S.E[1][sl] = en;
              S.map[1][cl] = (MapT)(sl + 1);
              S.gE[gg - 1] = 0.0;
              S.flg[1][sl] |= F_ATE;
              if (vt_valid) { S.vt[1][1 + sl] = (float)en; S.vt[2][gg] = 0.f; }
            }
            st.grass++;
            __syncwarp();
          }
        }
      }
      __syncwarp();
      PHASE_MARK(9)

      // Step 5: births in engagement order, predators then prey (BASE:389-448)  // PHASE: births
#pragma unroll 1
      for (int s = 0; s < 2; ++s) {
        for (int b0 = 0; b0 < SEL(n); b0 += 32) {
          const int k = b0 + lane;
          int slot = 0;
          bool elig = false;
          if (k < SEL(n)) {
            slot = SEL(S.ord)[k];
            elig = (SEL(S.flg)[slot] & F_ALIVE) && SEL(S.E)[slot] >= p.thr[s];
          }
          unsigned m = __ballot_sync(FULL, elig);
          while (m) {
            const int l = __ffs(m) - 1;
            m &= m - 1;
            const int ps_slot = __shfl_sync(FULL, slot, l);
            if ((s == 0 ? h.next_idx[0] : h.next_idx[1]) >= p.n_possible[s]) continue;  // id pool empty (BASE:395,424)
            if (SEL(n) + SEL(births) >= p.cap[s]) { h.status |= PPG_STATUS_SLOT_OVERFLOW; continue; }
            const unsigned pp = SEL(S.pos)[ps_slot];
            const int px = pp >> 8, py = pp & 255;
            int nl[2] = {n[0] + births[0], n[1] + births[1]};
            // _find_available_spawn_position (BASE:738-766)
            int sx = -1, sy = -1;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const int cx = px + (c == 0 ? -1 : (c == 1 ? 1 : 0));
              const int cy = py + (c == 2 ? -1 : (c == 3 ? 1 : 0));
              if (sx < 0 && cx >= 0 && cx < G && cy >= 0 && cy < G) {
                if (!any_agent_at(S, nl, (unsigned)((cx << 8) | cy), lane)) { sx = cx; sy = cy; }
              }
            }
            if (PPG_UNLIKELY(sx < 0)) {
              st.fallback++;
              if (p.tape_cells != nullptr && h.tape_pos < h.tape_end) {
                const int c = p.tape_cells[h.tape_pos++];  // recorded np.random.randint choice (BASE:764)
                sx = c / G; sy = c % G;
              } else {
                if (p.tape_cells != nullptr) h.status |= PPG_STATUS_TAPE_EXHAUSTED;
                // uniformly random free cell, ascending cell order, Philox draw
                const int c = philox_free_cell<MapT>(sbase, p, nl[0], nl[1],
                                                     ppg_draw_u32(h.seed_key, (unsigned)(env + p.env_base), h.episode, PPG_STREAM_SPAWN, h.spawn_draws), lane);
                if (c >= 0) { h.spawn_draws++; sx = c >> 8; sy = c & 255; }
              }
              if (sx < 0) { h.status |= PPG_STATUS_NO_SPAWN_CELL; continue; }  // reference raises here
            }
            const int cs = SEL(n) + SEL(births);
            if (s == 0) births[0]++; else births[1]++;
            const int child_id = s == 0 ? h.next_idx[0]++ : h.next_idx[1]++;  // BASE:396-397
            const double pe = SEL(S.E)[ps_slot] - p.init_e[s];  // BASE:404
            __syncwarp();
            if (lane == 0) {  // one writer for the warp-uniform stores
              SEL(S.id)[cs] = (uint16_t)child_id;
              SEL(S.pos)[cs] = (uint16_t)((sx << 8) | sy);
              SEL(S.E)[cs] = p.init_e[s];  // BASE:403
              SEL(S.flg)[cs] = F_ALIVE | F_NEWBORN;
              SEL(S.E)[ps_slot] = pe;
              SEL(S.map)[CELLXY(sx, sy)] = (MapT)(cs + 1);       // BASE:405
              SEL(S.map)[CELLXY(px, py)] = (MapT)(ps_slot + 1);  // BASE:406
              SEL(S.flg)[ps_slot] |= F_REPRO;
            }
            if (kick) {  // KICK:434-449
              const unsigned gp = SEL(S.par)[ps_slot];
              __syncwarp();
              if (lane == 0) {
                SEL(S.aux)[cs] = 0;
                SEL(S.par)[cs] = SEL(S.id)[ps_slot];
                SEL(S.aux)[ps_slot] = 0;  // rewards[agent] = reproduction_reward overwrites earlier kickbacks (BASE:409)
              }
              __syncwarp();
              if (gp != 0xFFFFu) {
                int gs = -1;
                #pragma unroll 1
                for (int i = lane; i < SEL(n) + SEL(births); i += 32)
                  if ((SEL(S.flg)[i] & F_ALIVE) && SEL(S.id)[i] == gp) gs = i;
                gs = __reduce_max_sync(FULL, gs);
                if (gs >= 0) {
                  const uint8_t cnt = SEL(S.aux)[gs];
                  __syncwarp();
                  if (lane == 0) SEL(S.aux)[gs] = (uint8_t)(cnt + 1);
                }
              }
            }
            __syncwarp();
          }
        }
      }
      __syncwarp();
      PHASE_MARK(10)

      // counts, termination, truncation (BASE:456-471)  // PHASE: counts
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        int c = 0;
        #pragma unroll 1
        for (int i = lane; i < n[s] + births[s]; i += 32) c += (S.flg[s][i] & F_ALIVE) ? 1 : 0;
        cur[s] = __reduce_add_sync(FULL, c);
      }
      h.step += 1;
      const bool all_term = cur[1] <= 0 || cur[0] <= 0;
      trunc = !all_term && h.step >= p.max_steps;  // BASE's extra truncation call (BASE:228-238) folded in
      over = all_term || trunc;
      env_flags = (all_term ? PPG_ENV_TERMINATED : 0) | (trunc ? PPG_ENV_TRUNCATED : 0);
      if (over) {
        if (p.autoreset) { next_live[0] = p.n_init[0]; next_live[1] = p.n_init[1]; }
      } else {
        next_live[0] = cur[0]; next_live[1] = cur[1];
      }
    } else {
      env_flags = PPG_ENV_IDLE;
    }

    PHASE_MARK(11)
    // ---------------------------------------------------------------- publish the counts  // PHASE: publish
    env_publish<SPLIT>(p, L, env, mode, next_live, births, (L.n_old_total[0] + L.n_old_total[1]) / p.B * 5 / 4, W == 1, lane);

    PHASE_MARK(12)
    // ------------------------------------------------- rows: metadata, observations, state write-back  // PHASE: rows pass1
    if (lane == 0) {
      p.old_off[0][env] = old_base[0];
      p.old_off[1][env] = old_base[1];
    }
    if (mode != 0) {
      const bool keep = !(over && p.autoreset);  // lists of a finished env are dead when it auto-resets
      refresh_tables(S, p, n[0] + births[0], n[1] + births[1], lane);
      PHASE_MARK(13)
      int wpos[2] = {0, 0};
      int new_base[2] = {0, 0};
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
          const int k = b0 + lane;
          int row = 0, slot = 0, cellp = 0;
          bool alive = false;
          unsigned nb_lab = 0;
          if (k < tot) {
            const bool newborn = k >= SEL(n);
            slot = newborn ? k : SEL(S.ord)[k];
            row = newborn ? SEL(new_base) + (k - SEL(n)) : SEL(old_base) + k;
            const unsigned f = SEL(S.flg)[slot];
            const double e = SEL(S.E)[slot];
            double rew = 0.0;
            if (mode == 2 && !newborn) {
              if (dense) {
                const double e0 = SEL(S.E0)[slot];
                if (f & F_DIED) rew = (f & F_CAUGHT) ? (0.0 - e0) : (e - e0);  // ADD:308,346
                else rew = (e - e0) + ((mode_r == PPG_REWARD_DENSE_ADDITIVE && (f & F_REPRO)) ? p.r_repro[s] : 0.0);  // ADD:468-471
              } else {
                if (f & F_DIED) rew = (f & F_CAUGHT) ? p.pen_caught : 0.0;  // BASE:288,328
                else {
                  rew = s == 0 ? ((f & F_ATE) ? p.r_catch : p.r_pstep) : ((f & F_ATE) ? p.r_eat : p.r_qstep);  // BASE:322,341,365,375
                  if (f & F_REPRO) rew = p.r_repro[s];  // BASE:409,438 overwrites
                  if (kick) for (int q = SEL(S.aux)[slot]; q > 0; --q) rew += p.r_kick[s];  // KICK:446
                }
              }
            }
            unsigned rf = 0;
            if (f & F_DIED) rf |= PPG_ROW_TERMINATED;
            if ((f & F_ALIVE) && trunc) rf |= PPG_ROW_TRUNCATED;
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
            alive = (f & F_ALIVE) != 0;
            const unsigned apos = SEL(S.pos)[slot];
            cellp = CELLP(apos);
          }
          unsigned m = __ballot_sync(FULL, alive);
          // survivors in engagement order (= `self.agents` after the sort), then newborns (BASE:398,468)
          int dst = 0xFFFF;
          if (keep && alive) {
            dst = SEL(wpos) + __popc(m & lt_mask);
            p.ag_id[s][sb + dst] = SEL(S.id)[slot];
            p.ag_pos[s][sb + dst] = SEL(S.pos)[slot];
            p.ag_e[s][sb + dst] = SEL(S.E)[slot];
            p.ag_prow[s][sb + dst] = row;  // SPLIT: newborns get theirs from the observation kernel
            if (kick) p.ag_par[s][sb + dst] = SEL(S.par)[slot];
          }
          if (s == 0) wpos[0] += __popc(m); else wpos[1] += __popc(m);
          // Step 6: observations of everyone still present, from the end-of-step grid (BASE:451-453)
          if (SPLIT) {
            if (k < tot) {
              // agents that died were observed at that moment (emit_row_now); the others by the observation kernel
              SEL(D.dsc)[k] = (uint16_t)(alive ? (unsigned)cellp : DSC_SKIP);
              if (pass == 1) p.nb_info[s][sb + (k - SEL(n))] = (unsigned long long)nb_lab | ((unsigned long long)(unsigned)dst << 32);
            }
          } else {
            while (m) {
              const int l = __ffs(m) - 1;
              m &= m - 1;
              const int cp = __shfl_sync(FULL, cellp, l);
              const int r = __shfl_sync(FULL, row, l);
              emit_row<MapT, BULK>(p, sb32, obs_s + (size_t)r * elems, cp, s, rr, rowctr, lane);
            }
          }
        }
      }
      }
      PHASE_MARK(14)
      env_rows_done<SPLIT>(p, L, sbase, env, mode, keep, old_base, n, births, new_base, next_live, lane);  // PHASE: tail
      PHASE_MARK(15)
      // leave the maps empty for the next env of this warp: un-write every cell that can hold an entry
      // (a non-zero owner entry always has its owner standing on it)
#pragma unroll
      for (int s = 0; s < 2; ++s)
        #pragma unroll 1
        for (int i = lane; i < n[s] + births[s]; i += 32)
          if (S.flg[s][i] & F_ALIVE) S.map[s][CELLP((unsigned)S.pos[s][i])] = 0;
      #pragma unroll 1
      for (int g = lane; g < p.n_grass; g += 32) S.map[2][CELLP((unsigned)S.gpos[g])] = 0;
      if (keep) {
        const int live0 = wpos[0] - births[0], live1 = wpos[1] - births[1];
        h.n_sorted[0] = (unsigned short)live0;
        h.n_sorted[1] = (unsigned short)live1;
        h.n_list[0] = (unsigned short)wpos[0];
        h.n_list[1] = (unsigned short)wpos[1];
        unsigned char sf = 0;
        if (mode == 2) {
          if (births[0] > 0 || h.first_step) sf |= 1;
          if (births[1] > 0 || h.first_step) sf |= 2;
          if (h.first_step) { h.n_sorted[0] = 0; h.n_sorted[1] = 0; }  // founders' numeric order is not the sorted order
          h.first_step = 0;
        }
        h.sortflag = sf;
        const size_t gb = (size_t)env * p.n_grass;
        #pragma unroll 1
        for (int g = lane; g < p.n_grass; g += 32) {
          p.gr_e[gb + g] = S.gE[g];
          if (mode == 1) p.gr_pos[gb + g] = S.gpos[g];
        }
      }
      PHASE_MARK(16)
      if (over) h.state = p.autoreset ? ST_NEEDS_RESET : ST_IDLE;  // idle: final state stays readable
      if (lane == 0) p.hdr[env] = h;
      add_stats(p, env, mode, n, births, over, trunc, h.step, st, lane);
    } else {
      env_idle<SPLIT>(p, sbase, env, old_base, lane);
    }
    const int count[2] = {mode == 0 ? h.n_list[0] : cur[0], mode == 0 ? h.n_list[1] : cur[1]};
    env_end<SPLIT>(p, L, env, mode, n, births, env_flags, h, t_env0, t_ns0, count, true, lane);
    PHASE_MARK(17)
    PHASE_FLUSH(base)
  }
  if (SPLIT) queue_push(p, L.pend, L.pend_env, lane);
  if (lane == 0) bulk_wait_read<0>();  // shared memory must stay valid until the engine has read it
  SPAN_MARK(base, 2)
}

// ------------------------------------------------------------------------------------------------
// small helper kernels
// ------------------------------------------------------------------------------------------------

// Publishes, as if by a launch with tag `epoch`, the rows every env needs in the next output (per-env
// words, block sums, group sums, totals).  Single CTA; used after ppg_create / ppg_reset /
// ppg_restore (the step kernel maintains them itself).
__global__ void ppg_prepare_offsets_kernel(const EnvHdr* __restrict__ hdr, int B, int n_init0, int n_init1, unsigned long long* cntA,
                                           unsigned long long* sum1, unsigned long long* sum2, int32_t* totals4, unsigned epoch, int hdr_founders) {
  const int t = threadIdx.x, T = blockDim.x;
  const int n_blk = (B + 31) >> 5, n_grp = (B + 1023) >> 10;
  for (int e = t; e < B; e += T) {
    const EnvHdr h = hdr[e];
    const bool rs = h.state & ST_NEEDS_RESET, idle = (h.state & ST_IDLE) && !rs;
    // founders of a scheduled reset: constants, or (trait variants of ECO) the per-episode draw kept in the header
    const bool hf = hdr_founders && ((unsigned)h.pad[1] & 0x80000000u);
    const int f0 = hf ? (h.pad[0] & 0xFFFF) : n_init0, f1 = hf ? ((h.pad[0] >> 16) & 0x7FFF) : n_init1;
    const int a0 = idle ? 0 : (rs ? f0 : h.n_list[0]), a1 = idle ? 0 : (rs ? f1 : h.n_list[1]);
    cntA[e] = TAG(epoch, (a0 << 16) | a1);
  }
  __syncthreads();
  for (int b = t; b < n_blk; b += T) {
    int a0 = 0, a1 = 0;
    for (int e = b << 5; e < min(B, (b + 1) << 5); ++e) { a0 += (int)((cntA[e] >> 16) & 0xFFFF); a1 += (int)(cntA[e] & 0xFFFF); }
    sum1[(size_t)b * 4 + 0] = TAG(epoch, a0); sum1[(size_t)b * 4 + 1] = TAG(epoch, a1);
    sum1[(size_t)b * 4 + 2] = TAG(epoch, 0);  sum1[(size_t)b * 4 + 3] = TAG(epoch, 0);
  }
  __syncthreads();
  for (int g = t; g < n_grp; g += T) {
    int a0 = 0, a1 = 0;
    for (int b = g << 5; b < min(n_blk, (g + 1) << 5); ++b) { a0 += (int)(unsigned)sum1[(size_t)b * 4]; a1 += (int)(unsigned)sum1[(size_t)b * 4 + 1]; }
    sum2[(size_t)g * 4 + 0] = TAG(epoch, a0); sum2[(size_t)g * 4 + 1] = TAG(epoch, a1);
    sum2[(size_t)g * 4 + 2] = TAG(epoch, 0);  sum2[(size_t)g * 4 + 3] = TAG(epoch, 0);
  }
  __syncthreads();
  if (t == 0) {
    int a0 = 0, a1 = 0;
    for (int g = 0; g < n_grp; ++g) { a0 += (int)(unsigned)sum2[(size_t)g * 4]; a1 += (int)(unsigned)sum2[(size_t)g * 4 + 1]; }
    totals4[0] = a0; totals4[1] = a1; totals4[2] = 0; totals4[3] = 0;
  }
}

// after ppg_restore: define the "previous output" of the restored state as each env's list laid out
// densely in list order, so that actions for the next step can be indexed by row again
__global__ void ppg_relabel_rows_kernel(StepParams p, const unsigned long long* cntA, const unsigned long long* sum1,
                                        const unsigned long long* sum2, const int32_t* totals4) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.B) return;
  const EnvHdr h = p.hdr[e];
  const bool live = !(h.state & (ST_NEEDS_RESET | ST_IDLE));
  const int blk = e >> 5, grp = e >> 10;
  for (int s = 0; s < 2; ++s) {
    int base = 0;
    for (int i = blk << 5; i < e; ++i) base += (int)((cntA[i] >> (s == 0 ? 16 : 0)) & 0xFFFF);
    for (int b = grp << 5; b < blk; ++b) base += (int)(unsigned)sum1[(size_t)b * 4 + s];
    for (int g = 0; g < grp; ++g) base += (int)(unsigned)sum2[(size_t)g * 4 + s];
    p.old_off[s][e] = base;
    p.new_off[s][e] = 0;
    p.new_cnt[s][e] = 0;
    if (e == 0) {
      p.old_off[s][p.B] = totals4[s];
      p.n_rows[s] = totals4[s];
      p.n_rows[2 + s] = 0;
    }
    if (!live) continue;
    const size_t b = (size_t)e * p.cap[s];
    for (int j = 0; j < h.n_list[s]; ++j) {
      p.ag_prow[s][b + j] = base + j;
      p.row_env[s][base + j] = e;
      p.row_agent[s][base + j] = p.ag_id[s][b + j];
      p.reward[s][base + j] = 0.f;
      p.flags[s][base + j] = 0;
    }
  }
  p.env_flags[e] = 0;
  p.env_status[e] = h.status;
  p.env_step[e] = h.step;
  p.env_count[2 * e] = h.n_list[0];
  p.env_count[2 * e + 1] = h.n_list[1];
}

__global__ void ppg_init_hdr_kernel(EnvHdr* hdr, int B, unsigned long long seed) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  EnvHdr h = {};
  h.seed_key = seed;
  h.state = ST_IDLE;  // not reset yet
  hdr[e] = h;
}

// schedule reset() for the masked envs (mask NULL = all), optionally re-keying the Philox stream
__global__ void ppg_mark_reset_kernel(EnvHdr* hdr, int B, const unsigned long long* seeds, const uint8_t* mask) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  if (mask && !mask[e]) return;
  if (seeds) hdr[e].seed_key = seeds[e];
  hdr[e].state = ST_NEEDS_RESET;
}

__global__ void ppg_set_tape_kernel(EnvHdr* hdr, int B, const long long* cell_off) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B) return;
  hdr[e].tape_pos = cell_off ? cell_off[e] : 0;
  hdr[e].tape_end = cell_off ? cell_off[e + 1] : 0;
}

// uniform random actions for the rows of the last output (synthetic rollouts)
__global__ void ppg_random_actions_kernel(const int32_t* __restrict__ n_rows, const int32_t* __restrict__ row_env0,
                                          const int32_t* __restrict__ row_agent0, const int32_t* __restrict__ row_env1,
                                          const int32_t* __restrict__ row_agent1, int32_t* act0, int32_t* act1,
                                          unsigned long long seed, unsigned call, unsigned n_actions, unsigned env_base) {
  allow_dependent_launch();       // PDL chain: the step kernel behind this one may become resident now ...
  wait_for_stream_predecessor();  // ... and this one waits for the observation kernel (row labels, row counts) before it reads
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
    (s ? act1 : act0)[row] = (int32_t)ppg_bounded(r, n_actions);
  }
}

// sum the per-env counters into int64 totals (block reduce + one atomic per block and counter)
__global__ void ppg_stats_kernel(const uint32_t* __restrict__ counters, const EnvHdr* __restrict__ hdr, int B,
                                 unsigned long long* out) {
  __shared__ unsigned long long s_acc[PPG_N_STATS];
  if (threadIdx.x < PPG_N_STATS) s_acc[threadIdx.x] = 0;
  __syncthreads();
  const int k = threadIdx.x & (PPG_N_STATS - 1);
  unsigned long long a = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)B * PPG_N_STATS; i += (size_t)gridDim.x * blockDim.x) {
    unsigned v = counters[i];
    if (k == PPG_STAT_STATUS_ENVS) v = hdr[i / PPG_N_STATS].status != 0;
    a += v;
  }
  atomicAdd(&s_acc[k], a);
  __syncthreads();
  if (threadIdx.x < PPG_N_STATS && s_acc[threadIdx.x]) atomicAdd(out + threadIdx.x, s_acc[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------
// launch wrappers used by ppg_api.cu
// ------------------------------------------------------------------------------------------------
// SPLIT (two-kernel step) exists for one warp per CTA and direct stores only (ppg_create enforces it)
template <typename MapT>
static StepKernel base_kernel(const StepParams& p, int warps_per_cta) {
  const bool bulk = p.obs_bulk != 0;
  if (p.obs_split) return {ppg_step_base_kernel<1, MapT, false, true>, 32};
  switch (warps_per_cta) {
    case 1: return {bulk ? ppg_step_base_kernel<1, MapT, true, false> : ppg_step_base_kernel<1, MapT, false, false>, 32};
    case 4: return {bulk ? ppg_step_base_kernel<4, MapT, true, false> : ppg_step_base_kernel<4, MapT, false, false>, 4 * 32};
    case 8: return {bulk ? ppg_step_base_kernel<8, MapT, true, false> : ppg_step_base_kernel<8, MapT, false, false>, 8 * 32};
    default: return {nullptr, 0};
  }
}

StepKernel step_kernel_base(const StepParams& p, int warps_per_cta) {
  return p.map_bytes == 1 ? base_kernel<uint8_t>(p, warps_per_cta) : base_kernel<uint16_t>(p, warps_per_cta);
}

cudaError_t launch_prepare_offsets(const EnvHdr* hdr, int B, int n0, int n1, unsigned long long* cntA, unsigned long long* sum1,
                                   unsigned long long* sum2, int32_t* totals4, unsigned epoch, int hdr_founders, cudaStream_t s) {
  ppg_prepare_offsets_kernel<<<1, 1024, 0, s>>>(hdr, B, n0, n1, cntA, sum1, sum2, totals4, epoch, hdr_founders);
  return cudaGetLastError();
}
cudaError_t launch_relabel_rows(const StepParams& p, const unsigned long long* cntA, const unsigned long long* sum1,
                                const unsigned long long* sum2, const int32_t* totals4, cudaStream_t s) {
  ppg_relabel_rows_kernel<<<(p.B + 127) / 128, 128, 0, s>>>(p, cntA, sum1, sum2, totals4);
  return cudaGetLastError();
}
cudaError_t launch_init_hdr(EnvHdr* hdr, int B, unsigned long long seed, cudaStream_t s) {
  ppg_init_hdr_kernel<<<(B + 255) / 256, 256, 0, s>>>(hdr, B, seed);
  return cudaGetLastError();
}
cudaError_t launch_mark_reset(EnvHdr* hdr, int B, const unsigned long long* seeds, const uint8_t* mask, cudaStream_t s) {
  ppg_mark_reset_kernel<<<(B + 255) / 256, 256, 0, s>>>(hdr, B, seeds, mask);
  return cudaGetLastError();
}
cudaError_t launch_set_tape(EnvHdr* hdr, int B, const long long* cell_off, cudaStream_t s) {
  ppg_set_tape_kernel<<<(B + 255) / 256, 256, 0, s>>>(hdr, B, cell_off);
  return cudaGetLastError();
}
cudaError_t launch_random_actions(const int32_t* n_rows, const int32_t* re0, const int32_t* ra0, const int32_t* re1,
                                  const int32_t* ra1, int32_t* a0, int32_t* a1, unsigned long long seed, unsigned call,
                                  unsigned n_actions, unsigned env_base, int blocks, cudaStream_t s) {
  return pdl_launch(ppg_random_actions_kernel, dim3((unsigned)blocks), dim3(256), 0, s, n_rows, re0, ra0, re1, ra1, a0, a1, seed, call, n_actions, env_base);
}
cudaError_t launch_stats(const uint32_t* counters, const EnvHdr* hdr, int B, unsigned long long* out, cudaStream_t s) {
  ppg_stats_kernel<<<148, 256, 0, s>>>(counters, hdr, B, out);
  return cudaGetLastError();
}

}  // namespace ppg
