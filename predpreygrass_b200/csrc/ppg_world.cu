// ppg_world.cu — the batched world state (`grid_world_state`, BASE:311 / ECO / STAG) of a range of envs.
//
// The step kernels leave every env's IMAGE in HBM (ppg_obs.cu): padded owner maps, fp32 value tables, wall table — the
// end-of-step grid the observation rows are gathered from.  Gathering the same way at every cell of the field gives the
// reference's grid after step(), rounded to float32 exactly as the rows round it (DESIGN.md §4).
//
// One CTA per env at a time (grid-striding over the range): the image comes into shared memory with coalesced 16-byte
// loads, then the CTA writes the env's C*G*G floats as one contiguous slab with streaming stores (float4 when the slab
// and `out` allow it).  The kernel never executes griddepcontrol.launch_dependents and is launched without programmatic
// stream serialization: with the PDL launch chain on, the next step kernel must not start (and overwrite the images)
// before this kernel has finished reading them.
#include <cuda_runtime.h>

#include <cstdint>

#include "ppg_device.cuh"

namespace ppg {

constexpr int WS_THREADS = 256;

// A field position (channel c, row x, column y).  Every env's slab has the same shape, so a thread's positions are the same
// in every env: they are found by division once and then advanced by additions (dividing by the runtime G and G*G for
// every element made a call 1.5x slower, DESIGN.md §4).
struct WsPos { int c, x, y; };
__device__ __forceinline__ WsPos ws_pos(int q, int G) {
  const int GG = G * G, c = q / GG, r = q - c * GG;
  return {c, r / G, r - (r / G) * G};
}
__device__ __forceinline__ void ws_add(WsPos& a, const WsPos& d, int G) {  // a += d, d.x < G, d.y < G
  a.y += d.y;
  if (a.y >= G) { a.y -= G; ++a.x; }
  a.x += d.x;
  if (a.x >= G) { a.x -= G; ++a.c; }
  a.c += d.c;
}
template <typename MapT>
__device__ __forceinline__ float ws_cell(const WorldStateParams& p, const unsigned char* img, const WsPos& a) {
  const int k = a.c < PPG_WS_SRC ? a.c : PPG_WS_SRC - 1;
  const int idx = p.P + (a.x + p.P) * p.PS + a.y;
  const unsigned m = reinterpret_cast<const MapT*>(img + p.map_off[k])[idx];
  return reinterpret_cast<const float*>(img + p.tbl_off[k])[m];
}

template <typename MapT>
__global__ void __launch_bounds__(WS_THREADS, 6) ppg_world_state_kernel(const __grid_constant__ WorldStateParams p) {
  extern __shared__ __align__(16) unsigned char s_img[];
  const int G = p.G, per_env = p.C * G * G;
  const bool vec = (per_env & 3) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0;
  const int n16 = p.img_bytes >> 4;
  const int lane_q = vec ? 4 * threadIdx.x : threadIdx.x, step_q = vec ? 4 * WS_THREADS : WS_THREADS;
  const WsPos first = ws_pos(lane_q, G), step = ws_pos(step_q, G), one = {0, 0, 1};
  for (int i = blockIdx.x; i < p.n_envs; i += gridDim.x) {
    const uint4* src = reinterpret_cast<const uint4*>(p.img + (size_t)(p.env_begin + i) * p.img_stride);
    uint4* dst = reinterpret_cast<uint4*>(s_img);
    for (int k = threadIdx.x; k < n16; k += WS_THREADS) dst[k] = __ldg(src + k);
    __syncthreads();
    float* out = p.out + (size_t)i * per_env;
    WsPos a = first;
    if (vec) {
      float4* o4 = reinterpret_cast<float4*>(out);
      for (int q = lane_q; q < per_env; q += step_q, ws_add(a, step, G)) {
        WsPos b = a;
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          v[k] = ws_cell<MapT>(p, s_img, b);
          ws_add(b, one, G);
        }
        __stcs(o4 + (q >> 2), make_float4(v[0], v[1], v[2], v[3]));
      }
    } else {
      for (int q = lane_q; q < per_env; q += step_q, ws_add(a, step, G)) __stcs(out + q, ws_cell<MapT>(p, s_img, a));
    }
    __syncthreads();  // every read of the image is done before the next env's copy overwrites it
  }
}

template <typename MapT>
static cudaError_t launch_world_state_t(const WorldStateParams& p, int n_cta, cudaStream_t stream) {
  const size_t smem = (size_t)p.img_bytes;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(ppg_world_state_kernel<MapT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  ppg_world_state_kernel<MapT><<<n_cta, WS_THREADS, smem, stream>>>(p);
  return cudaGetLastError();
}

template <typename MapT>
static cudaError_t world_state_occupancy_t(const WorldStateParams& p, int* blocks_per_sm) {
  const size_t smem = (size_t)p.img_bytes;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(ppg_world_state_kernel<MapT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, ppg_world_state_kernel<MapT>, WS_THREADS, smem);
}

cudaError_t launch_world_state(const WorldStateParams& p, int map_bytes, int n_cta, cudaStream_t stream) {
  return map_bytes == 1 ? launch_world_state_t<uint8_t>(p, n_cta, stream) : launch_world_state_t<uint16_t>(p, n_cta, stream);
}
cudaError_t world_state_occupancy(const WorldStateParams& p, int map_bytes, int* blocks_per_sm) {
  return map_bytes == 1 ? world_state_occupancy_t<uint8_t>(p, blocks_per_sm) : world_state_occupancy_t<uint16_t>(p, blocks_per_sm);
}

}  // namespace ppg
