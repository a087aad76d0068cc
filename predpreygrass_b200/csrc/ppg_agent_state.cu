// ppg_agent_state.cu — the state of the agent behind every row of the last output (include/ppg.h ppg_agent_state).
//
// It reads only what the output left in HBM: the env headers' list lengths, the agent lists (ids, positions, energies, the
// variant's extra columns and ag_prow, the row each entry's action is read from), the grass lists, and the output's row
// offsets, row ids and env flags.  One warp per env (grid-striding): per species the lanes first write the sentinels into the
// env's old and newborn rows, then, after __syncwarp, scatter the list entries into their rows.  An entry k writes row
// r = ag_prow[k] only when r lies in the env's row ranges and row_agent[r] == ag_id[k]: ag_prow is only meaningful for
// entries that have a row in this output (an ECO carcass of an earlier output keeps a stale one), and the ids of one env's
// rows are distinct, so each present row is written by exactly one lane.  Lists of an env whose episode ended in this output
// are not read: an auto-resetting env does not write them back on that step.  The kernel never executes
// griddepcontrol.launch_dependents and is launched without programmatic stream serialization: with the launch chain on, the
// next step's kernels must not rewrite the lists or the rows while it still reads them.
#include <cuda_runtime.h>

#include <cstdint>

#include "ppg_device.cuh"

namespace ppg {

constexpr int AS_WARPS = 8;  // warps per CTA

__device__ __forceinline__ double as_nan() { return __longlong_as_double(0x7FF8000000000000LL); }

__device__ __forceinline__ void blank_row(const ppg_agent_state_args& a, int s, int r) {
  a.present[s][r] = 0;
  if (a.pos[s]) { a.pos[s][2 * (size_t)r] = -1; a.pos[s][2 * (size_t)r + 1] = -1; }
  if (a.energy[s]) a.energy[s][r] = as_nan();
  if (a.trait[s]) a.trait[s][r] = as_nan();
  if (a.acc[s]) a.acc[s][r] = as_nan();
  if (a.age[s]) a.age[s][r] = -1;
  if (a.facing[s]) a.facing[s][r] = -1;
}

__global__ void __launch_bounds__(AS_WARPS * 32) ppg_agent_state_kernel(const __grid_constant__ AgentStateParams p) {
  const ppg_agent_state_args& a = p.a;
  const int lane = threadIdx.x & 31;
  for (int e = blockIdx.x * AS_WARPS + (threadIdx.x >> 5); e < p.B; e += gridDim.x * AS_WARPS) {
    // everything the env's row ranges and list lengths depend on, requested before any of it is used
    const bool ended = (p.env_flags[e] & (PPG_ENV_TERMINATED | PPG_ENV_TRUNCATED)) != 0;
    int o0[2], o1[2], n0[2], nc[2], nl[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      o0[s] = p.old_off[s][e];
      o1[s] = p.old_off[s][e + 1];
      nc[s] = p.new_cnt[s][e];
      n0[s] = p.new_off[s][e];  // defined where new_cnt > 0
      nl[s] = p.hdr[e].n_list[s];
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int n_old = o1[s] - o0[s], n_new = nc[s] > 0 ? nc[s] : 0;
      for (int k = lane; k < n_old + n_new; k += 32) blank_row(a, s, k < n_old ? o0[s] + k : n0[s] + (k - n_old));
    }
    __syncwarp();  // the sentinels are in place before a lane writes a present row over one
    if (!ended) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const size_t b = (size_t)e * p.cap[s];
        const int n_new = nc[s] > 0 ? nc[s] : 0;
        for (int k = lane; k < nl[s]; k += 32) {
          const int r = p.ag_prow[s][b + k];
          const int id = p.ag_id[s][b + k];
          const unsigned xy = p.ag_pos[s][b + k];
          const double en = p.ag_e[s][b + k];
          const bool in_range = (r >= o0[s] && r < o1[s]) || (r >= n0[s] && r < n0[s] + n_new);
          if (!in_range || p.row_agent[s][r] != id) continue;
          a.present[s][r] = 1;
          if (a.pos[s]) { a.pos[s][2 * (size_t)r] = (int32_t)(xy >> 8); a.pos[s][2 * (size_t)r + 1] = (int32_t)(xy & 255u); }
          if (a.energy[s]) a.energy[s][r] = en;
          if (a.trait[s]) a.trait[s][r] = p.ag_trait[s][b + k];
          if (a.acc[s]) a.acc[s][r] = p.ag_acc[s][b + k];
          if (a.age[s]) a.age[s][r] = p.ag_age[s][b + k];
          if (a.facing[s]) a.facing[s][r] = (int8_t)p.ag_face[b + k];
        }
      }
    }
    const size_t gb = (size_t)e * p.n_grass;
    for (int g = lane; g < p.n_grass; g += 32) {
      const unsigned xy = ended ? 0u : p.gr_pos[gb + g];
      if (a.grass_pos) {
        a.grass_pos[2 * (gb + g)] = ended ? -1 : (int32_t)(xy >> 8);
        a.grass_pos[2 * (gb + g) + 1] = ended ? -1 : (int32_t)(xy & 255u);
      }
      if (a.grass_energy) a.grass_energy[gb + g] = ended ? as_nan() : p.gr_e[gb + g];
    }
  }
}

cudaError_t launch_agent_state(const AgentStateParams& p, cudaStream_t stream) {
  ppg_agent_state_kernel<<<(p.B + AS_WARPS - 1) / AS_WARPS, AS_WARPS * 32, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace ppg
