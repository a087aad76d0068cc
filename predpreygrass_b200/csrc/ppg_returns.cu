// ppg_returns.cu — episode returns and agent lifetimes on the device (include/ppg.h ppg_track_returns).
//
// ppg_returns_kernel runs after the observation kernel of every output while tracking is on and reads only what the step
// already left in HBM: the rows' ids, rewards and flags, the row offsets and the env flags.  One warp per env
// (grid-striding): per species the old rows first, lanes in parallel, then after __syncwarp the newborn rows, so an id freed
// by a TERMINATED old row and handed to a newborn of the same step is finished before it is restarted.  The per-step sums
// are formed in the fixed order documented in ppg.h (lane-strided partials in row order, then an xor-butterfly), so every
// value is reproducible bit for bit.  The kernel never executes griddepcontrol.launch_dependents and is launched without
// programmatic stream serialization: with the launch chain on, the next step's kernels must not overwrite the rows while
// it still reads them.
//
// ppg_episode_stats_kernel reduces the per-env accumulators [n][PPG_N_EP_STATS] in two passes (blocks of EPS_ROWS rows,
// then one block over the partials), each in a fixed order: bit-identical from run to run.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "ppg_device.cuh"

namespace ppg {

constexpr int RT_WARPS = 8;      // warps per CTA of ppg_returns_kernel
constexpr int EPS_GROUPS = 64;   // row groups per CTA of ppg_episode_stats_kernel (64 x 16 slots = 1024 threads)
constexpr int EPS_ROWS = 256;    // rows per CTA in the first pass

struct LifeSums {
  double step = 0.0;   // sum of this output's rewards of the species
  double ended = 0.0;  // sum of row_return over the lives that ended
  int lives = 0, deaths = 0, rows = 0;
};

__device__ __forceinline__ void update_row(const ReturnsParams& p, int s, int e, int r, bool valid, LifeSums& a) {
  const unsigned f = p.flags[s][r];
  if (!valid) {
    p.row_return[s][r] = __longlong_as_double(0x7FF8000000000000LL);  // NaN
    p.row_life[s][r] = 0;
    return;
  }
  const double rw = (double)p.reward[s][r];
  const size_t k = (size_t)e * p.n_possible[s] + p.row_agent[s][r];
  double ret;
  int life;
  if (f & (PPG_ROW_FOUNDER | PPG_ROW_NEWBORN)) {
    ret = rw;
    life = 1;
  } else {
    ret = p.tab_ret[s][k] + rw;
    life = p.tab_life[s][k] + 1;
  }
  p.tab_ret[s][k] = ret;
  p.tab_life[s][k] = life;
  p.row_return[s][r] = ret;
  p.row_life[s][r] = life;
  a.step += rw;
  if (f & (PPG_ROW_TERMINATED | PPG_ROW_TRUNCATED)) {
    a.lives += 1;
    a.deaths += (f & PPG_ROW_TERMINATED) ? 1 : 0;
    a.ended += ret;
    a.rows += life;
  }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, k);
  return v;  // a + b == b + a in IEEE arithmetic: every lane holds the same bits
}

__global__ void __launch_bounds__(RT_WARPS * 32) ppg_returns_kernel(const __grid_constant__ ReturnsParams p) {
  const int lane = threadIdx.x & 31;
  for (int e = blockIdx.x * RT_WARPS + (threadIdx.x >> 5); e < p.B; e += gridDim.x * RT_WARPS) {
    const unsigned ef = p.env_flags[e];
    if (ef & PPG_ENV_IDLE) continue;
    const bool valid = (ef & PPG_ENV_RESET) || p.env_valid[e];
    LifeSums a[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int o0 = p.old_off[s][e], o1 = p.old_off[s][e + 1];
      for (int r = o0 + lane; r < o1; r += 32) update_row(p, s, e, r, valid, a[s]);
      __syncwarp();  // the old rows' table reads and writes are done before a newborn restarts a reused id
      const int nc = p.new_cnt[s][e];
      if (nc > 0) {
        const int n0 = p.new_off[s][e];
        for (int r = n0 + lane; r < n0 + nc; r += 32) update_row(p, s, e, r, valid, a[s]);
      }
    }
    if (!valid) continue;
    double step[2], ended[2];
    int lives[2], deaths[2], rows[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      step[s] = warp_sum(a[s].step);
      ended[s] = warp_sum(a[s].ended);
      lives[s] = __reduce_add_sync(0xFFFFFFFFu, a[s].lives);
      deaths[s] = __reduce_add_sync(0xFFFFFFFFu, a[s].deaths);
      rows[s] = __reduce_add_sync(0xFFFFFFFFu, a[s].rows);
    }
    if (lane == 0) {
      double* er = p.env_return + 2 * (size_t)e;
      double* acc = p.env_acc + (size_t)e * PPG_N_EP_STATS;
      double ret0 = (ef & PPG_ENV_RESET) ? 0.0 : er[0], ret1 = (ef & PPG_ENV_RESET) ? 0.0 : er[1];
      ret0 += step[0];
      ret1 += step[1];
      er[0] = ret0;
      er[1] = ret1;
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        double* q = acc + PPG_EP_LIVES + PPG_EP_SPECIES_STRIDE * s;
        q[0] += (double)lives[s];
        q[1] += (double)deaths[s];
        q[2] += ended[s];
        q[3] += (double)rows[s];
      }
      if (ef & (PPG_ENV_TERMINATED | PPG_ENV_TRUNCATED)) {
        const double total = ret0 + ret1;
        acc[PPG_EP_EPISODES] += 1.0;
        acc[PPG_EP_LENGTH_SUM] += (double)p.env_step[e];
        acc[PPG_EP_RETURN_SUM] += total;
        acc[PPG_EP_RETURN_SQ_SUM] += total * total;
        acc[PPG_EP_RETURN_PRED] += ret0;
        acc[PPG_EP_RETURN_PREY] += ret1;
        acc[PPG_EP_RETURN_MAX] = fmax(acc[PPG_EP_RETURN_MAX], total);
        acc[PPG_EP_RETURN_NEG_MIN] = fmax(acc[PPG_EP_RETURN_NEG_MIN], -total);
      }
      p.env_valid[e] = 1;
    }
  }
}

__device__ __forceinline__ bool eps_is_max(int slot) { return slot == PPG_EP_RETURN_MAX || slot == PPG_EP_RETURN_NEG_MIN; }

// rows [blockIdx.x * rows_per_cta, ...) of in[n][PPG_N_EP_STATS] -> out[blockIdx.x][PPG_N_EP_STATS].  Thread (g, slot) combines
// rows g, g + 64, ... in order (rows with valid[row] == 0 skipped when valid is given), then the 64 groups are combined by a
// halving tree in shared memory.
__global__ void __launch_bounds__(EPS_GROUPS * PPG_N_EP_STATS) ppg_episode_stats_kernel(const double* __restrict__ in, const uint8_t* __restrict__ valid,
                                                                                       int n, int rows_per_cta, double* __restrict__ out) {
  __shared__ double s_v[EPS_GROUPS][PPG_N_EP_STATS];
  const int slot = threadIdx.x % PPG_N_EP_STATS, g = threadIdx.x / PPG_N_EP_STATS;
  const bool mx = eps_is_max(slot);
  const int lo = blockIdx.x * rows_per_cta, hi = min(n, lo + rows_per_cta);
  double v = mx ? -INFINITY : 0.0;
  for (int r = lo + g; r < hi; r += EPS_GROUPS) {
    if (valid && !valid[r]) continue;
    const double x = in[(size_t)r * PPG_N_EP_STATS + slot];
    v = mx ? fmax(v, x) : v + x;
  }
  s_v[g][slot] = v;
  for (int w = EPS_GROUPS / 2; w > 0; w >>= 1) {
    __syncthreads();
    if (g < w) s_v[g][slot] = mx ? fmax(s_v[g][slot], s_v[g + w][slot]) : s_v[g][slot] + s_v[g + w][slot];
  }
  if (g == 0) out[(size_t)blockIdx.x * PPG_N_EP_STATS + slot] = s_v[0][slot];
}

__global__ void ppg_episode_stats_clear_kernel(double* acc, int B) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * PPG_N_EP_STATS; i += gridDim.x * blockDim.x)
    acc[i] = eps_is_max(i % PPG_N_EP_STATS) ? -INFINITY : 0.0;
}

cudaError_t launch_returns(const ReturnsParams& p, cudaStream_t stream) {
  ppg_returns_kernel<<<(p.B + RT_WARPS - 1) / RT_WARPS, RT_WARPS * 32, 0, stream>>>(p);
  return cudaGetLastError();
}

int episode_stats_partials(int B) { return (B + EPS_ROWS - 1) / EPS_ROWS; }

// partial: [episode_stats_partials(B)][PPG_N_EP_STATS] scratch
cudaError_t launch_episode_stats(const double* env_acc, const uint8_t* env_valid, int B, double* partial, double* out, cudaStream_t stream) {
  const int nb = episode_stats_partials(B);
  ppg_episode_stats_kernel<<<nb, EPS_GROUPS * PPG_N_EP_STATS, 0, stream>>>(env_acc, env_valid, B, EPS_ROWS, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  ppg_episode_stats_kernel<<<1, EPS_GROUPS * PPG_N_EP_STATS, 0, stream>>>(partial, nullptr, nb, nb, out);
  return cudaGetLastError();
}

cudaError_t launch_episode_stats_clear(double* env_acc, int B, cudaStream_t stream) {
  ppg_episode_stats_clear_kernel<<<(B * PPG_N_EP_STATS + 255) / 256, 256, 0, stream>>>(env_acc, B);
  return cudaGetLastError();
}

}  // namespace ppg
