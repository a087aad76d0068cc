// ppg_links.cu — the row of the previous output behind every row of the last output (include/ppg.h ppg_track_links).
//
// ppg_links_kernel runs after the observation kernel of every output while links are on.  One warp per env (grid-striding),
// per species:
//   1. lookup: every old, non-FOUNDER row of an env whose output is not a reset takes its id to the env's link table, which
//      was saved after the previous output, and writes the row found there into prev_row; every other row gets -1;
//   2. save (after __syncwarp, which orders the lookups' reads before the table is rewritten): the table is cleared and
//      refilled from the env's agent lists as the step left them, (ag_id[k], ag_prow[k]) for k < n_list: each agent that
//      acts in the next step and the row of this output its action is read from.
// A table word is id << 16 | j (the link table of ppg_device.cuh), j the position of the row among the env's rows of the
// saved output: old rows o0 + j for j < n_old, newborn rows n0 + (j - n_old) after them.  base[s][e] keeps (o0, n_old, n0) of
// that output, so a lookup needs none of its offsets, which the next step overwrites.  An entry whose ag_prow is not a row of
// this output carrying its id (an ECO carcass of an earlier output keeps a stale ag_prow) is not saved.  The lists of an env
// whose episode ended in this output are not saved either: an auto-resetting env does not write them back on that step, and
// its next output is a reset (all FOUNDER rows) or idle, so nothing looks its table up.
//
// save_only (ppg_track_links switching on, ppg_restore) runs step 2 alone.  No atomics touch prev_row: each row is written by
// one lane, so the result does not depend on the schedule.  The kernel never executes griddepcontrol.launch_dependents and is
// launched without programmatic stream serialization: with the launch chain on, the next step's kernels must not rewrite the
// lists and rows while it still reads them.
#include <cuda_runtime.h>

#include <cstdint>

#include "ppg_device.cuh"

namespace ppg {

constexpr int LK_WARPS = 8;  // warps per CTA

__global__ void __launch_bounds__(LK_WARPS * 32) ppg_links_kernel(const __grid_constant__ LinksParams p) {
  const int lane = threadIdx.x & 31;
  for (int e = blockIdx.x * LK_WARPS + (threadIdx.x >> 5); e < p.B; e += gridDim.x * LK_WARPS) {
    const unsigned ef = p.env_flags[e];
    unsigned err = 0;
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
      const int H = 1 << p.log2_h[s], n_old = o1[s] - o0[s], n_new = nc[s] > 0 ? nc[s] : 0;
      uint32_t* tab = p.tab[s] + (size_t)e * H;
      if (!p.save_only) {
        const bool linked = !(ef & (PPG_ENV_RESET | PPG_ENV_IDLE));
        const int4 bs = p.base[s][e];
        for (int k = lane; k < n_old + n_new; k += 32) {
          const int r = k < n_old ? o0[s] + k : n0[s] + (k - n_old);
          int pr = -1;
          if (k < n_old && linked && !(p.flags[s][r] & PPG_ROW_FOUNDER)) {
            const int id = p.row_agent[s][r];
            if (id >= 0 && id < 0xFFFF) {
              uint32_t q = link_slot(id, p.log2_h[s]);
              for (int probe = 0; probe < H; ++probe) {
                const uint32_t w = tab[q];
                if (w == LINK_EMPTY) break;
                if ((int)(w >> 16) == id) {
                  const int j = (int)(w & 0xFFFFu);
                  pr = j < bs.y ? bs.x + j : bs.z + (j - bs.y);
                  break;
                }
                q = (q + 1) & (H - 1);
              }
            }
            if (pr < 0) err |= PPG_LINK_ERR_MISSING;
          }
          p.prev_row[s][r] = pr;
        }
        __syncwarp();  // every lookup has read the table before it is rewritten
      }
      if (ef & (PPG_ENV_TERMINATED | PPG_ENV_TRUNCATED)) continue;
      for (int k = lane; k < H; k += 32) tab[k] = LINK_EMPTY;
      __syncwarp();
      const size_t b = (size_t)e * p.cap[s];
      for (int k = lane; k < nl[s]; k += 32) {
        const int r = p.ag_prow[s][b + k];
        const int id = p.ag_id[s][b + k];
        const int j = (r >= o0[s] && r < o1[s]) ? r - o0[s] : (r >= n0[s] && r < n0[s] + n_new) ? n_old + (r - n0[s]) : -1;
        if (j < 0 || p.row_agent[s][r] != id) continue;
        const uint32_t w = (uint32_t)id << 16 | (uint32_t)j;
        uint32_t q = link_slot(id, p.log2_h[s]);
        int probe = 0;
        while (atomicCAS(&tab[q], LINK_EMPTY, w) != LINK_EMPTY && ++probe < H) q = (q + 1) & (H - 1);
        if (probe >= H) err |= PPG_LINK_ERR_OVERFLOW;
      }
      if (lane == 0) p.base[s][e] = make_int4(o0[s], n_old, n0[s], 0);
    }
    err = __reduce_or_sync(0xFFFFFFFFu, err);
    if (lane == 0 && err) atomicOr(p.error, err);
  }
}

cudaError_t launch_links(const LinksParams& p, cudaStream_t stream) {
  ppg_links_kernel<<<(p.B + LK_WARPS - 1) / LK_WARPS, LK_WARPS * 32, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace ppg
