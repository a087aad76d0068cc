// ppg_gae.cu — advantages and value targets of a recorded rollout (include/ppg.h ppg_gae).
//
// One warp per (env, species), blockIdx.y = species, grid-striding over the envs.  The warp walks the outputs backward from
// t = T to 0.  At output t it reads the env's rows of t; it looks every live row up, by id, in the link table of output t+1
// and, for a hit, evaluates the recursion from the successor row's reward, flags, value, advantage and link (written by the
// same warp one iteration earlier); and it inserts the old, non-FOUNDER rows of t into the other table, which serves output
// t-1.  A table is an open-addressing hash (linear probing) of (id << 16 | row - old_off) words in the warp's shared-memory
// slice, so its size follows cap_live, never n_possible.  __syncwarp separates the outputs: it orders the warp's global
// writes of output t+1 before the reads of output t.  Every value is one chain of fp32 operations with no reduction, so the
// result does not depend on the schedule.  The kernel never executes griddepcontrol.launch_dependents.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>

#include "ppg_device.cuh"

namespace ppg {

constexpr int GAE_WARPS = 8;  // warps per CTA at most; fewer when a warp's two tables need more than GAE_SMEM_MAX / 8
constexpr int GAE_SMEM_MAX = 227 * 1024;
constexpr uint32_t GAE_EMPTY = 0xFFFFFFFFu;  // id 0xFFFF is never valid (n_possible <= 65535)

__device__ __forceinline__ uint32_t gae_slot(int id, int log2_h) { return ((uint32_t)id * 0x9E3779B1u) >> (32 - log2_h); }

__global__ void __launch_bounds__(GAE_WARPS * 32) ppg_gae_kernel(const __grid_constant__ GaeParams p) {
  extern __shared__ uint32_t gae_smem[];
  const int lane = threadIdx.x & 31, s = blockIdx.y, warps = blockDim.x >> 5;
  const int H = 1 << p.log2_h, T = p.a.T, B = p.B;
  const long long C = p.cap[s];
  uint32_t* const tab = gae_smem + (size_t)(threadIdx.x >> 5) * 2 * H;  // two tables: output t uses tab + (t & 1) * H
  const float gamma = p.a.gamma, gl = __fmul_rn(p.a.gamma, p.a.lam);
  const int32_t* __restrict__ agent = p.a.row_agent[s];
  const uint8_t* __restrict__ flags = p.a.flags[s];
  const float* __restrict__ reward = p.a.reward[s];
  const float* __restrict__ value = p.a.value[s];
  const int32_t* __restrict__ old_off = p.a.old_off[s];
  const int32_t* __restrict__ new_off = p.a.new_off[s];
  const int32_t* __restrict__ new_cnt = p.a.new_cnt[s];
  float* adv = p.a.adv[s];
  float* vtg = p.a.value_target[s];
  int32_t* next_row = p.a.next_row[s];
  const float qnan = __int_as_float(0x7FC00000);

  for (int e = blockIdx.x * warps + (threadIdx.x >> 5); e < B; e += gridDim.x * warps) {
    unsigned err = 0;
    int in_next = 0;       // entries of the table of output t+1
    int old0_next = 0;     // old_off[t+1][e]
    bool next_ok = false;  // the table of output t+1 is complete
    for (int t = T; t >= 0; --t) {
      uint32_t* mine = tab + (t & 1) * H;
      const uint32_t* succ = tab + ((t + 1) & 1) * H;
      for (int k = lane; k < H; k += 32) mine[k] = GAE_EMPTY;
      __syncwarp();
      const int o0 = old_off[(size_t)t * (B + 1) + e], o1 = old_off[(size_t)t * (B + 1) + e + 1];
      const int n0 = new_off[(size_t)t * B + e], nc = new_cnt[(size_t)t * B + e];
      const int n_old = o1 - o0;
      const bool range_ok = 0 <= o0 && o0 <= o1 && o1 <= C && n_old <= H / 2 && n_old < 0xFFFF &&
                            0 <= nc && (nc == 0 || (0 <= n0 && (long long)n0 + nc <= C));
      if (!range_ok) err |= PPG_GAE_ERR_RANGE;
      const int total = range_ok ? n_old + nc : 0;
      const unsigned ef1 = t < T ? p.a.env_flags[(size_t)(t + 1) * B + e] : 0u;
      const bool lookup = t < T && next_ok && !(ef1 & (PPG_ENV_RESET | PPG_ENV_IDLE));
      int inserted = 0, matched = 0;
      for (int j0 = 0; j0 < total; j0 += 32) {
        const int j = j0 + lane;
        const bool live_lane = j < total;
        const long long r = j < n_old ? (long long)o0 + j : (long long)n0 + (j - n_old);
        const size_t ir = (size_t)t * C + r;
        int id = 0;
        unsigned f = 0;
        if (live_lane) {
          id = agent[ir];
          f = flags[ir];
          if (id < 0 || id >= p.n_possible[s]) err |= PPG_GAE_ERR_ID;
        }
        const bool id_ok = live_lane && id >= 0 && id < p.n_possible[s];
        bool ins = t > 0 && id_ok && j < n_old && !(f & (PPG_ROW_FOUNDER | PPG_ROW_NEWBORN));
        if (ins) {
          const uint32_t w = (uint32_t)id << 16 | (uint32_t)j;
          uint32_t k = gae_slot(id, p.log2_h);
          int probe = 0;
          while (atomicCAS(&mine[k], GAE_EMPTY, w) != GAE_EMPTY && ++probe < H) k = (k + 1) & (H - 1);
          if (probe >= H) { err |= PPG_GAE_ERR_RANGE; ins = false; }
        }
        inserted += __popc(__ballot_sync(0xFFFFFFFFu, ins));
        int rn = -1;
        if (lookup && id_ok && !(f & (PPG_ROW_TERMINATED | PPG_ROW_TRUNCATED))) {
          uint32_t k = gae_slot(id, p.log2_h);
          for (int probe = 0; probe < H; ++probe) {
            const uint32_t w = succ[k];
            if (w == GAE_EMPTY) break;
            if ((int)(w >> 16) == id) { rn = old0_next + (int)(w & 0xFFFFu); break; }
            k = (k + 1) & (H - 1);
          }
        }
        matched += __popc(__ballot_sync(0xFFFFFFFFu, rn >= 0));
        if (live_lane && t < T) {
          float a = qnan, vt = qnan;
          if (rn >= 0) {
            const size_t in1 = (size_t)(t + 1) * C + rn;
            const unsigned f1 = flags[in1];
            const bool term = (f1 & PPG_ROW_TERMINATED) || ((ef1 & PPG_ENV_TERMINATED) && !(f1 & PPG_ROW_TRUNCATED));
            const bool trunc = !term && ((f1 & PPG_ROW_TRUNCATED) || (ef1 & PPG_ENV_TRUNCATED));
            const float vn = term ? 0.0f : value[in1];
            const bool cont = t + 1 < T && !term && !trunc && next_row[in1] >= 0;
            const float an = cont ? adv[in1] : 0.0f;
            const float v0 = value[ir];
            const float delta = __fsub_rn(__fadd_rn(reward[in1], __fmul_rn(gamma, vn)), v0);
            a = __fadd_rn(delta, __fmul_rn(gl, an));
            vt = __fadd_rn(a, v0);
          }
          adv[ir] = a;
          vtg[ir] = vt;
          next_row[ir] = rn;
        }
      }
      // every old, non-FOUNDER row of output t+1 must be some live row's successor (the count identity of ppg.h)
      if (lookup && matched != in_next) err |= PPG_GAE_ERR_LINK;
      if (t < T && !lookup && next_ok && in_next != 0) err |= PPG_GAE_ERR_LINK;
      in_next = inserted;
      old0_next = o0;
      next_ok = range_ok;
      __syncwarp();  // this output's table and results are complete before output t-1 reads them
    }
    err = __reduce_or_sync(0xFFFFFFFFu, err);
    if (lane == 0 && err) atomicOr(p.a.error, err);
  }
}

// warps per CTA for a link table of 1 << log2_h entries (0: the two tables of one warp do not fit in shared memory)
int gae_warps(int log2_h) { return (int)std::min<size_t>(GAE_WARPS, GAE_SMEM_MAX / (2 * ((size_t)1 << log2_h) * sizeof(uint32_t))); }

cudaError_t launch_gae(const GaeParams& p, cudaStream_t stream) {
  const int warps = gae_warps(p.log2_h);
  const size_t smem = (size_t)warps * 2 * ((size_t)1 << p.log2_h) * sizeof(uint32_t);
  cudaError_t e = cudaFuncSetAttribute(ppg_gae_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const dim3 grid((unsigned)((p.B + warps - 1) / warps), 2);
  ppg_gae_kernel<<<grid, warps * 32, smem, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace ppg
