// ppg_step_common.cuh — device code shared by the step kernels of all env variants (ppg_base.cu, ppg_eco.cu, ppg_stag.cu):
// the per-env shared-memory view, the observation-row writers (two-level gather: padded byte maps -> fp32
// value tables), the deterministic cross-env row allocation (hierarchical epoch-tagged counts), the
// Philox placement / free-cell draws and the env loop around the variants' simulation.  See DESIGN.md §3.
#pragma once
#include <cuda_runtime.h>

#include "ppg_device.cuh"

namespace ppg {

#define FULL 0xffffffffu
// rarely taken branches (reset, replay tapes, explicit action order, fall-backs): kept out of the fall-through path, the step
// kernels are bound by instruction delivery (DESIGN.md §3)
#define PPG_UNLIKELY(x) __builtin_expect(!!(x), 0)

// shared-memory atomics by 32-bit shared address: one ATOMS / RED instruction instead of the generic-pointer atomicAdd's
// address-space dispatch (~15 instructions per call in the SASS of the previous build)
__device__ __forceinline__ void red_shared_add(const void* smem_ptr, unsigned v) {
  asm volatile("red.shared.add.u32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(smem_ptr)), "r"(v) : "memory");
}
__device__ __forceinline__ int atom_shared_add(const void* smem_ptr, int v) {
  int old;
  asm volatile("atom.shared.add.s32 %0, [%1], %2;" : "=r"(old) : "r"((unsigned)__cvta_generic_to_shared(smem_ptr)), "r"(v) : "memory");
  return old;
}

__device__ __forceinline__ unsigned globaltimer_lo() { unsigned v; asm volatile("mov.u32 %0, %%globaltimer_lo;" : "=r"(v)); return v; }
__device__ __forceinline__ unsigned smid() { unsigned v; asm volatile("mov.u32 %0, %%smid;" : "=r"(v)); return v; }

// Per-phase latency profile of the step kernels (experimental builds only: scripts/build_prof.py compiles the library with
// -DPPG_PHASE_PROF; the shipped library has none of this).  PHASE_MARK(k) charges the SM cycles since the previous mark to
// phase k of the env the warp is working on; the per-launch totals are read by `ppg_debug_phase_cycles_<variant>`.
#ifdef PPG_PHASE_PROF
#define PPG_N_PHASES 24
#define PPG_PROF_MAX_ENVS 65536
#define PHASE_DEFINE(name)                                                                                          \
  __device__ unsigned g_phase_cycles_##name[PPG_PROF_MAX_ENVS][PPG_N_PHASES];                                       \
  extern "C" int ppg_debug_phase_cycles_##name(unsigned* out, int n_envs) { /* [n_envs][PPG_N_PHASES] of the last launch */ \
    return cudaMemcpyFromSymbol(out, g_phase_cycles_##name, sizeof(unsigned) * PPG_N_PHASES * (size_t)n_envs) == cudaSuccess ? 0 : -1; \
  }
// kernel span per CTA: globaltimer (ns, low 32 bits) at kernel entry, at the first env's start and at exit
#define SPAN_DEFINE(name)                                                                                           \
  __device__ unsigned g_span_##name[3][8192];                                                                       \
  extern "C" int ppg_debug_span_##name(unsigned* out) { return cudaMemcpyFromSymbol(out, g_span_##name, sizeof(unsigned) * 3 * 8192) == cudaSuccess ? 0 : -1; }
#define SPAN_MARK(name, k) if (lane == 0 && blockIdx.x < 8192) g_span_##name[k][blockIdx.x] = globaltimer_lo();
#define PHASE_DECL long long ph_t = clock64(); unsigned ph_acc[PPG_N_PHASES]; _Pragma("unroll") for (int k_ = 0; k_ < PPG_N_PHASES; ++k_) ph_acc[k_] = 0;
#define PHASE_MARK(k) { const long long t_ = clock64(); ph_acc[k] += (unsigned)(t_ - ph_t); ph_t = t_; }
#define PHASE_FLUSH(name) if (lane == 0 && env < PPG_PROF_MAX_ENVS) { _Pragma("unroll") for (int k_ = 0; k_ < PPG_N_PHASES; k_ += 4) \
    *reinterpret_cast<uint4*>(&g_phase_cycles_##name[env][k_]) = make_uint4(ph_acc[k_], ph_acc[k_ + 1], ph_acc[k_ + 2], ph_acc[k_ + 3]); }
#else
#define PHASE_DEFINE(name)
#define SPAN_DEFINE(name)
#define SPAN_MARK(name, k)
#define PHASE_DECL
#define PHASE_MARK(k)
#define PHASE_FLUSH(name)
#endif

// ------------------------------------------------------------------------------------------------
// shared-memory view of one env
// ------------------------------------------------------------------------------------------------
template <typename MapT>
struct EnvSmem {
  double* E[2];
  double* E0[2];
  double* gE;
  float* wt;       // wall table: 1.0 at wall_idx, else 0 (constant)
  float* vt[3];    // fp32 value tables: predators [cap0+2], prey [cap1+1], grass [n_grass+1]; entry 0 = 0
  float* stage;    // 2 row buffers of stage_elems floats
  uint8_t* scr;    // [CH] touch counters / predator marks; all zero between uses
  uint16_t* id[2];
  uint16_t* pos[2];
  uint16_t* ord[2];  // ord[k] = slot of the k-th agent in engagement order
  uint16_t* rnk[2];  // inverse of ord
  uint16_t* par[2];
  MapT* map[3];      // padded: [0],[1] owner maps (slot + 1 of the agent the reference grid shows, 0 = empty), [2] grass index + 1
  uint16_t* gpos;
  uint8_t* act[2];
  uint8_t* flg[2];
  uint8_t* aux[2];  // kickback count
  uint8_t* gtag;    // [n_grass] scratch for the prey chunk conflict test
};

template <typename MapT>
__device__ __forceinline__ EnvSmem<MapT> carve(unsigned char* base, const StepParams& p) {
  EnvSmem<MapT> s;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    s.E[k] = reinterpret_cast<double*>(base + p.so_E[k]);
    s.E0[k] = reinterpret_cast<double*>(base + p.so_E0[k]);
    s.id[k] = reinterpret_cast<uint16_t*>(base + p.so_id[k]);
    s.pos[k] = reinterpret_cast<uint16_t*>(base + p.so_pos[k]);
    s.ord[k] = reinterpret_cast<uint16_t*>(base + p.so_ord[k]);
    s.rnk[k] = reinterpret_cast<uint16_t*>(base + p.so_rnk[k]);
    s.par[k] = reinterpret_cast<uint16_t*>(base + p.so_par[k]);
    s.act[k] = base + p.so_act[k];
    s.flg[k] = base + p.so_flg[k];
    s.aux[k] = base + p.so_aux[k];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    s.map[k] = reinterpret_cast<MapT*>(base + p.so_map[k]);
    s.vt[k] = reinterpret_cast<float*>(base + p.so_vt[k]);
  }
  s.gE = reinterpret_cast<double*>(base + p.so_gE);
  s.wt = reinterpret_cast<float*>(base + p.so_wt);
  s.stage = reinterpret_cast<float*>(base + p.so_stage);
  s.scr = base + p.so_scr;
  s.gpos = reinterpret_cast<uint16_t*>(base + p.so_gpos);
  s.gtag = base + p.so_gtag;
  return s;
}

// ------------------------------------------------------------------------------------------------
// PTX helpers
// ------------------------------------------------------------------------------------------------
// bulk asynchronous shared -> global copy (TMA engine, SASS UBLKCP)
__device__ __forceinline__ void bulk_store(void* gdst, unsigned ssrc32, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(__cvta_generic_to_global(gdst)), "r"(ssrc32), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ unsigned long long ld_volatile(const unsigned long long* p) {
  return *reinterpret_cast<const volatile unsigned long long*>(p);
}
__device__ __forceinline__ void st_volatile(unsigned long long* p, unsigned long long v) {
  *reinterpret_cast<volatile unsigned long long*>(p) = v;
}
#define TAG(epoch, val) (((unsigned long long)(epoch) << 32) | (unsigned long long)(unsigned)(val))

// padded map index of a packed position (x << 8 | y)
#define CELLP(ps) (PP + ((int)((ps) >> 8) + PP) * PS + (int)((ps)&255u))
#define CELLXY(x, y) (PP + ((x) + PP) * PS + (y))

// two-kernel step: row descriptors inside the env image (DESIGN.md §3.3) and the image dump
struct RowDesc {
  uint16_t* dsc[2];  // padded cell index of the window centre of the k-th row (k < n: rows of the agents that acted, in
                     // output order; k >= n: newborns in birth order), or DSC_SKIP / DSC_ZERO
  unsigned* dsx[2];  // ECO: own-speed plane value (float bits); STAG: ihi | jhi << 8
};
__device__ __forceinline__ RowDesc carve_desc(unsigned char* base, const StepParams& p) {
  RowDesc d;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    d.dsc[k] = reinterpret_cast<uint16_t*>(base + p.so_dsc[k]);
    d.dsx[k] = reinterpret_cast<unsigned*>(base + p.so_dsx[k]);
  }
  return d;
}

// Writes the image header and copies the image range of the env's shared-memory slice to HBM (coalesced 16-byte
// stores, default caching: the observation kernel reads it back from L2 a few microseconds later).  mode 0 (idle
// env): header only, zero rows.  Only the copy: finish_env() signals the env.
__device__ __forceinline__ void dump_image(unsigned char* sbase, const StepParams& p, int env, int mode, bool keep, const int old_base[2],
                                           const int n[2], const int births[2], int lane) {
  int* ih = reinterpret_cast<int*>(sbase + p.so_ihdr);
  if (lane < IH_INTS) {
    int v = 0;
    switch (lane) {
      case IH_OLD_BASE0: v = old_base[0]; break;
      case IH_OLD_BASE1: v = old_base[1]; break;
      case IH_N0: v = mode ? n[0] : 0; break;
      case IH_N1: v = mode ? n[1] : 0; break;
      case IH_BIRTHS0: v = mode ? births[0] : 0; break;
      case IH_BIRTHS1: v = mode ? births[1] : 0; break;
      case IH_MODE: v = mode; break;
      case IH_KEEP: v = keep ? 1 : 0; break;
      default: break;
    }
    ih[lane] = v;
  }
  __syncwarp();
  const uint4* src = reinterpret_cast<const uint4*>(sbase + p.so_img);
  uint4* dst = reinterpret_cast<uint4*>(p.obs_img + (size_t)env * p.img_stride);
  const int n16 = mode ? p.img_bytes >> 4 : (IH_INTS * 4) >> 4;
  #pragma unroll 1
  for (int i = lane; i < n16; i += 32) dst[i] = src[i];
  __syncwarp();
  // the env is handed to the observation kernel by finish_env(), after the env's remaining stores: one fence for all of them
}

// lets a kernel launched with programmatic stream serialization (the observation kernel) start while this one runs
__device__ __forceinline__ void allow_dependent_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// A kernel launched with programmatic stream serialization (pdl_launch below) may become resident while the kernel before it
// in the stream is still running; this is where it waits for that kernel to have completed and flushed its writes.  A no-op
// for a kernel launched without the attribute.  Every step / action kernel executes it before touching global memory.
__device__ __forceinline__ void wait_for_stream_predecessor() { asm volatile("griddepcontrol.wait;" ::: "memory"); }


// ------------------------------------------------------------------------------------------------
// observation rows
// ------------------------------------------------------------------------------------------------
// per-lane gather constants of one species (obs_rel table of the host)
struct RowRel {
  int relb[PPG_MAX_NJ];      // byte offset of the map entry from the agent's own map-0 entry
  unsigned tbl[PPG_MAX_NJ];  // shared address of the value table
  unsigned self;             // bit j: element j is the agent's own trait plane (ECO speed plane), not a gather
};

__device__ __forceinline__ RowRel load_rel(const StepParams& p, int s, unsigned sb32, int lane) {
  RowRel r;
  r.self = p.obs_self ? __ldg(p.obs_self + s * 32 + lane) : 0u;
#pragma unroll
  for (int j = 0; j < PPG_MAX_NJ; ++j) {
    r.relb[j] = 0; r.tbl[j] = 0;
    if (j < p.nj[s]) {
      const int2 v = __ldg(p.obs_rel + (s * PPG_MAX_NJ + j) * 32 + lane);
      r.relb[j] = v.x; r.tbl[j] = sb32 + (unsigned)v.y;  // lanes past the end of the row (last iteration only) get a harmless in-range pair
    }
  }
  return r;
}

// fp32 copies of the energies the observation channels show (float64 state -> float32 row values)
template <typename MapT>
__device__ __forceinline__ void refresh_tables(const EnvSmem<MapT>& S, const StepParams& p, int nt0, int nt1, int lane) {
  #pragma unroll 1
  for (int i = lane; i < nt0; i += 32) S.vt[0][1 + i] = (float)S.E[0][i];
  #pragma unroll 1
  for (int i = lane; i < nt1; i += 32) S.vt[1][1 + i] = (float)S.E[1][i];
  #pragma unroll 1
  for (int g = lane; g < p.n_grass; g += 32) S.vt[2][1 + g] = (float)S.gE[g];
  if (lane == 0) S.vt[0][0] = 0.f;
  if (lane == 1) S.vt[1][0] = 0.f;
  if (lane == 2) S.vt[2][0] = 0.f;
  if (lane == 3) S.vt[0][p.wall_idx] = 0.f;
  __syncwarp();
}

// shared-memory accesses by 32-bit shared address (PTX keeps them in the order written: all map loads of a
// row, then all table loads, then all stores, so the hardware sees 2 dependent latencies per row)
template <typename MapT>
__device__ __forceinline__ unsigned lds_map(unsigned a);
template <>
__device__ __forceinline__ unsigned lds_map<uint8_t>(unsigned a) {
  unsigned v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
template <>
__device__ __forceinline__ unsigned lds_map<uint16_t>(unsigned a) {
  unsigned short v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds_f32(unsigned a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_f32(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }

// _get_observation (BASE:511-539) of the agent whose padded cell index is `cellp` into global row `dst`.
// Every lane produces N elements of the row, element = table[map[cell + const]]:
//   VEC  (row length a multiple of 4): lane l owns the float4 groups l, l+32, ... (4 consecutive elements each;
//        with byte maps the 32 lanes of one load still hit 32 different banks) and stores them with STG.128;
//   !VEC: lane l owns elements l, l+32, ... and stores 32-bit words, 128 contiguous bytes per warp instruction.
// BULK stages the row in shared memory and hands it to the bulk-copy engine instead (cp.async.bulk, one
// 784/1296/1620-byte copy per row, double buffered); measured slower than direct streaming stores for rows this
// small (see DESIGN.md), kept selectable with PPG_OBS_BULK=1.
template <typename MapT, int N, bool VEC, bool BULK, bool SELF = false>
__device__ __forceinline__ void emit_row_t(const StepParams& p, unsigned sb32, float* dst, int cellp, int s, const RowRel& r,
                                           unsigned& rowctr, int lane, float selfv = 0.f) {
  const unsigned a0 = sb32 + (unsigned)(p.so_map[0] + cellp * (int)sizeof(MapT));
  unsigned idx[N];
  float val[N];
#pragma unroll
  for (int j = 0; j < N; ++j) idx[j] = lds_map<MapT>(a0 + (unsigned)r.relb[j]);
#pragma unroll
  for (int j = 0; j < N; ++j) val[j] = lds_f32(r.tbl[j] + 4u * idx[j]);
  if (SELF) {
#pragma unroll
    for (int j = 0; j < N; ++j)
      if ((r.self >> j) & 1u) val[j] = selfv;
  }
  const int elems = p.elems[s];
  if (BULK) {
    const unsigned buf = sb32 + (unsigned)p.so_stage + (rowctr & 1u) * (unsigned)(p.stage_elems * 4);
    ++rowctr;
    if (lane == 0) bulk_wait_read<1>();  // the copy issued two rows ago has finished reading `buf`
    __syncwarp();
    if (VEC) {
#pragma unroll
      for (int v = 0; v < N / 4; ++v)
        if (4 * (lane + 32 * v) < elems) {
#pragma unroll
          for (int k = 0; k < 4; ++k) sts_f32(buf + 16u * (lane + 32 * v) + 4u * k, val[4 * v + k]);
        }
    } else {
#pragma unroll
      for (int j = 0; j < N; ++j)
        if (lane + 32 * j < elems) sts_f32(buf + 4u * (lane + 32 * j), val[j]);
    }
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      bulk_store(dst, buf, (unsigned)elems * 4u);
      bulk_commit();
    }
  } else {
    if (VEC) {
      float4* d = reinterpret_cast<float4*>(dst) + lane;
#pragma unroll
      for (int v = 0; v < N / 4; ++v)
        if (4 * (lane + 32 * v) < elems) __stcs(d + 32 * v, make_float4(val[4 * v], val[4 * v + 1], val[4 * v + 2], val[4 * v + 3]));
    } else {
      float* d = dst + lane;
#pragma unroll
      for (int j = 0; j < N; ++j)
        if (lane + 32 * j < elems) __stcs(d + 32 * j, val[j]);
    }
  }
}

// any row shape: one element at a time
template <typename MapT, bool BULK>
__device__ __noinline__ unsigned emit_row_generic(const StepParams& p, unsigned sb32, float* dst, int cellp, int s, unsigned rowctr, int lane,
                                                  unsigned selfmask = 0u, float selfv = 0.f) {
  const unsigned a0 = sb32 + (unsigned)(p.so_map[0] + cellp * (int)sizeof(MapT));
  const bool vec = p.obs_vec[s] != 0;
  unsigned buf = 0;
  if (BULK) {
    buf = sb32 + (unsigned)p.so_stage + (rowctr & 1u) * (unsigned)(p.stage_elems * 4);
    ++rowctr;
    if (lane == 0) bulk_wait_read<1>();
    __syncwarp();
  }
#pragma unroll 1
  for (int j = 0; j < p.nj[s]; ++j) {
    const int q = vec ? 4 * (lane + 32 * (j >> 2)) + (j & 3) : lane + 32 * j;
    if (q < p.elems[s]) {
      const int2 v = __ldg(p.obs_rel + (s * PPG_MAX_NJ + j) * 32 + lane);
      float x = lds_f32(sb32 + (unsigned)v.y + 4u * lds_map<MapT>(a0 + (unsigned)v.x));
      if ((selfmask >> j) & 1u) x = selfv;
      if (BULK) sts_f32(buf + 4u * q, x); else __stcs(dst + q, x);
    }
  }
  if (BULK) {
    fence_async_smem();
    __syncwarp();
    if (lane == 0) {
      bulk_store(dst, buf, (unsigned)p.elems[s] * 4u);
      bulk_commit();
    }
  }
  return rowctr;
}

// TWO rows of the same species at once (direct stores only): all 2N map loads are issued back to back, then all 2N table
// loads, then the stores — the same two dependent shared-memory latencies as one row, paid once for two rows
// (short_scoreboard was the observation kernel's top stall, profiles/r01_final_summary.md)
template <typename MapT, int N, bool VEC, bool SELF>
__device__ __forceinline__ void emit_row2_t(const StepParams& p, unsigned sb32, float* dst0, float* dst1, int cellp0, int cellp1, int s,
                                            const RowRel& r, int lane, float selfv0, float selfv1) {
  const unsigned a0 = sb32 + (unsigned)(p.so_map[0] + cellp0 * (int)sizeof(MapT));
  const unsigned a1 = sb32 + (unsigned)(p.so_map[0] + cellp1 * (int)sizeof(MapT));
  unsigned idx0[N], idx1[N];
  float val0[N], val1[N];
#pragma unroll
  for (int j = 0; j < N; ++j) idx0[j] = lds_map<MapT>(a0 + (unsigned)r.relb[j]);
#pragma unroll
  for (int j = 0; j < N; ++j) idx1[j] = lds_map<MapT>(a1 + (unsigned)r.relb[j]);
#pragma unroll
  for (int j = 0; j < N; ++j) val0[j] = lds_f32(r.tbl[j] + 4u * idx0[j]);
#pragma unroll
  for (int j = 0; j < N; ++j) val1[j] = lds_f32(r.tbl[j] + 4u * idx1[j]);
  if (SELF) {
#pragma unroll
    for (int j = 0; j < N; ++j)
      if ((r.self >> j) & 1u) { val0[j] = selfv0; val1[j] = selfv1; }
  }
  const int elems = p.elems[s];
  if (VEC) {
    float4* d0 = reinterpret_cast<float4*>(dst0) + lane;
    float4* d1 = reinterpret_cast<float4*>(dst1) + lane;
#pragma unroll
    for (int v = 0; v < N / 4; ++v)
      if (4 * (lane + 32 * v) < elems) {
        __stcs(d0 + 32 * v, make_float4(val0[4 * v], val0[4 * v + 1], val0[4 * v + 2], val0[4 * v + 3]));
        __stcs(d1 + 32 * v, make_float4(val1[4 * v], val1[4 * v + 1], val1[4 * v + 2], val1[4 * v + 3]));
      }
  } else {
    float* d0 = dst0 + lane;
    float* d1 = dst1 + lane;
#pragma unroll
    for (int j = 0; j < N; ++j)
      if (lane + 32 * j < elems) { __stcs(d0 + 32 * j, val0[j]); __stcs(d1 + 32 * j, val1[j]); }
  }
}

// true if the species' row shape has a two-row writer (else the caller writes the rows one by one)
template <typename MapT, bool SELF>
__device__ __forceinline__ bool emit_row2(const StepParams& p, unsigned sb32, float* dst0, float* dst1, int cellp0, int cellp1, int s,
                                          const RowRel& r, int lane, float selfv0 = 0.f, float selfv1 = 0.f) {
  switch (p.emit_kind[s]) {
    case 1: emit_row2_t<MapT, 8, true, SELF>(p, sb32, dst0, dst1, cellp0, cellp1, s, r, lane, selfv0, selfv1); return true;
    case 2: emit_row2_t<MapT, 12, true, SELF>(p, sb32, dst0, dst1, cellp0, cellp1, s, r, lane, selfv0, selfv1); return true;
    case 3: emit_row2_t<MapT, 13, false, SELF>(p, sb32, dst0, dst1, cellp0, cellp1, s, r, lane, selfv0, selfv1); return true;
    case 4: emit_row2_t<MapT, 5, false, SELF>(p, sb32, dst0, dst1, cellp0, cellp1, s, r, lane, selfv0, selfv1); return true;
    case 5: emit_row2_t<MapT, 8, false, SELF>(p, sb32, dst0, dst1, cellp0, cellp1, s, r, lane, selfv0, selfv1); return true;
    default: return false;
  }
}

template <typename MapT, bool BULK, bool SELF = false>
__device__ __forceinline__ void emit_row(const StepParams& p, unsigned sb32, float* dst, int cellp, int s, const RowRel& r,
                                         unsigned& rowctr, int lane, float selfv = 0.f) {
  switch (p.emit_kind[s]) {  // warp-uniform; the row shapes of the reference's env family get straight-line code
    case 1: emit_row_t<MapT, 8, true, BULK, SELF>(p, sb32, dst, cellp, s, r, rowctr, lane, selfv); break;    // (4,7,7): 49 float4
    case 2: emit_row_t<MapT, 12, true, BULK, SELF>(p, sb32, dst, cellp, s, r, rowctr, lane, selfv); break;   // (4,9,9): 81 float4
    case 3: emit_row_t<MapT, 13, false, BULK, SELF>(p, sb32, dst, cellp, s, r, rowctr, lane, selfv); break;  // (5,9,9): 405 floats
    case 4: emit_row_t<MapT, 5, false, BULK, SELF>(p, sb32, dst, cellp, s, r, rowctr, lane, selfv); break;   // (3,7,7): 147 floats (trait variants without a trait plane)
    case 5: emit_row_t<MapT, 8, false, BULK, SELF>(p, sb32, dst, cellp, s, r, rowctr, lane, selfv); break;   // (3,9,9): 243 floats
    default: rowctr = emit_row_generic<MapT, BULK>(p, sb32, dst, cellp, s, rowctr, lane, SELF ? r.self : 0u, selfv);
  }
}

// a row whose window is cut off (saturated forward view): element (c, i, j) is zero unless i <= ihi and j <= jhi
template <typename MapT>
__device__ __noinline__ void emit_row_masked(const StepParams& p, unsigned sb32, float* dst, int cellp, int s, int ihi, int jhi, int lane) {
  const unsigned a0 = sb32 + (unsigned)(p.so_map[0] + cellp * (int)sizeof(MapT));
  const bool vec = p.obs_vec[s] != 0;
  const int R = p.R[s], RR = R * R;
#pragma unroll 1
  for (int j = 0; j < p.nj[s]; ++j) {
    const int q = vec ? 4 * (lane + 32 * (j >> 2)) + (j & 3) : lane + 32 * j;
    if (q < p.elems[s]) {
      const int2 v = __ldg(p.obs_rel + (s * PPG_MAX_NJ + j) * 32 + lane);
      float x = lds_f32(sb32 + (unsigned)v.y + 4u * lds_map<MapT>(a0 + (unsigned)v.x));
      const int r = q % RR;
      if (r / R > ihi || r % R > jhi) x = 0.f;
      __stcs(dst + q, x);
    }
  }
}

// ended agents are observed as all-zero rows (STAG:596-612)
__device__ __forceinline__ void zero_row(float* dst, int elems, int lane) {
  #pragma unroll 1
  for (int q = lane; q < elems; q += 32) __stcs(dst + q, 0.f);
}

// rows of agents that die mid-step: the reference captures them at that moment (BASE:287,327)
template <typename MapT, bool BULK, bool SELF = false>
__device__ __noinline__ unsigned emit_row_now(unsigned char* base, const StepParams& p, float* dst, int cellp, int s, int nt0, int nt1,
                                              unsigned rowctr, int lane, float selfv = 0.f) {
  if (nt0 >= 0) {  // nt0 < 0: the caller keeps the value tables current itself (ppg_base.cu)
    const EnvSmem<MapT> S = carve<MapT>(base, p);
    refresh_tables(S, p, nt0, nt1, lane);
  }
  const unsigned sb32 = (unsigned)__cvta_generic_to_shared(base);
  const RowRel r = load_rel(p, s, sb32, lane);
  emit_row<MapT, BULK, SELF>(p, sb32, dst, cellp, s, r, rowctr, lane, selfv);
  __syncwarp();  // every lane's map / table reads are done before the caller un-writes the dying agent's cell
  return rowctr;
}

// any live agent (either species, newborns included) on cell `pos`?  = `pos in set(agent_positions.values())` (BASE:399,754)
template <typename MapT>
__device__ __forceinline__ bool any_agent_at(const EnvSmem<MapT>& S, const int nl[2], unsigned pos, int lane) {
  bool hit = false;
#pragma unroll
  for (int s = 0; s < 2; ++s)
    #pragma unroll 1
    for (int i = lane; i < nl[s]; i += 32) hit |= (S.flg[s][i] & F_ALIVE) && S.pos[s][i] == pos;
  return __any_sync(FULL, hit);
}

// exclusive prefix, over the envs before `env`, of two 16-bit-packed per-env counts.
//   cnt : per-env words (value pair in bits 31..16 / 15..0), sum1/sum2: per-block / per-group sums at [.][4] + v0, + v0 + 1
// `epoch` = tag the words must carry; wait = poll until they do (this launch's counts) or trust them (previous launch's).
__device__ __forceinline__ bool prefix_before(const unsigned long long* cnt, const unsigned long long* sum1, const unsigned long long* sum2,
                                              int v0, int env, unsigned epoch, bool wait, int lane, int& out0, int& out1) {
  const int blk = env >> 5, grp = env >> 10;
  unsigned spins = 0;
  for (;;) {
    int a0 = 0, a1 = 0;
    bool ok = true;
    if (lane < (env & 31)) {
      const unsigned long long w = ld_volatile(cnt + (blk << 5) + lane);
      ok &= (unsigned)(w >> 32) == epoch;
      a0 += (int)((w >> 16) & 0xFFFFu);
      a1 += (int)(w & 0xFFFFu);
    }
    if (lane < (blk & 31)) {
      const unsigned long long* q = sum1 + (size_t)((grp << 5) + lane) * 4 + v0;
      const unsigned long long w0 = ld_volatile(q), w1 = ld_volatile(q + 1);
      ok &= (unsigned)(w0 >> 32) == epoch && (unsigned)(w1 >> 32) == epoch;
      a0 += (int)(unsigned)w0;
      a1 += (int)(unsigned)w1;
    }
    #pragma unroll 1
    for (int g = lane; g < grp; g += 32) {
      const unsigned long long* q = sum2 + (size_t)g * 4 + v0;
      const unsigned long long w0 = ld_volatile(q), w1 = ld_volatile(q + 1);
      ok &= (unsigned)(w0 >> 32) == epoch && (unsigned)(w1 >> 32) == epoch;
      a0 += (int)(unsigned)w0;
      a1 += (int)(unsigned)w1;
    }
    if (__all_sync(FULL, ok) || !wait) {
      out0 = __reduce_add_sync(FULL, a0);
      out1 = __reduce_add_sync(FULL, a1);
      return __all_sync(FULL, ok);
    }
    // predecessors hold lower tickets, so they are running or done: this terminates.  The cap only
    // protects the box from a wedged launch.
    if (++spins > (1u << 22)) return false;
    __nanosleep(200);
  }
}

// `count` draws of clip(mean + std * N(0,1), lo, hi) into out[0..count), bit-identical to `count` sequential
// ppg_draw_normal calls on the stream (one Philox counter per polar attempt, accepted attempts go to the draws in
// counter order), but with the 32 lanes evaluating 32 consecutive attempts at once.  Returns the advanced counter.
static __device__ __noinline__ unsigned draw_normals_batched(double* out, int count, double mean, double std, double lo, double hi,
                                                             unsigned long long seed_key, unsigned env, unsigned episode, unsigned stream,
                                                             unsigned ctr, int lane) {
  const unsigned lt = (1u << lane) - 1u;
  int got = 0;
  while (got < count) {
    const ppg_u32x4 r = ppg_philox4x32(env, episode, ctr + (unsigned)lane, stream, (unsigned)seed_key, (unsigned)(seed_key >> 32));
    const double a = 2.0 * ppg_u01(r.v[0], r.v[1]) - 1.0, b = 2.0 * ppg_u01(r.v[2], r.v[3]) - 1.0;
    const double q = a * a + b * b;
    const bool acc = q < 1.0 && q > 1e-300;
    const unsigned m = __ballot_sync(FULL, acc);
    const int k = got + __popc(m & lt);
    if (acc && k < count) {
      const double v = mean + std * (a * PPG_SQRT(-2.0 * ppg_log(q) / q));
      out[k] = v < lo ? lo : (v > hi ? hi : v);
    }
    const int cnt = __popc(m);
    if (got + cnt >= count) {
      ctr += __fns(m, 0, count - got) + 1u;  // position after the attempt that produced the last draw
      got = count;
    } else {
      got += cnt;
      ctr += 32u;
    }
  }
  __syncwarp();
  return ctr;
}

// reset(): n_total unique cells in draw order (law of BASE:156-177) from the env's Philox placement stream
// `first[cell]` = 1 + index of the first draw that hit the cell; wall cells (STAG:2138 `free_non_wall_indices`) are
// pre-claimed with 0, which no draw equals: a draw that hits a wall is skipped like a duplicate.
static __device__ __noinline__ void philox_placement(int* cells, unsigned* first, int n_total, int GG, unsigned env, unsigned episode,
                                              unsigned long long seed_key, int lane, const int32_t* walls = nullptr, int n_walls = 0) {
  #pragma unroll 1
  for (int i = lane; i < GG; i += 32) first[i] = 0xFFFFFFFFu;
  __syncwarp();
  #pragma unroll 1
  for (int i = lane; i < n_walls; i += 32) first[walls[i]] = 0u;
  __syncwarp();
  int accepted = 0;
  for (unsigned batch = 0; accepted < n_total; ++batch) {
    const unsigned idx0 = batch * 128u + 4u * lane;
    const ppg_u32x4 r = ppg_philox4x32(env, episode, idx0 >> 2, PPG_STREAM_PLACEMENT, (unsigned)seed_key, (unsigned)(seed_key >> 32));
    unsigned cell[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      cell[k] = ppg_bounded(r.v[k], (unsigned)GG);
      atomicMin(&first[cell[k]], idx0 + k + 1u);
    }
    __syncwarp();
    int mine = 0;
    bool ok[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { ok[k] = first[cell[k]] == idx0 + k + 1u; mine += ok[k]; }
    int incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { int t = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += t; }
    int posn = accepted + incl - mine;
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (ok[k]) { if (posn < n_total) cells[posn] = (int)cell[k]; ++posn; }
    accepted += __shfl_sync(FULL, incl, 31);
    __syncwarp();
  }
}

// Occupancy marks for the free-cell scans below: scr[cell] = 1 under every live agent (O(n / 32) per warp instead of
// testing every cell against every agent).  scr is all zero outside its users; unmark_agents restores that.
template <typename MapT>
__device__ __forceinline__ void mark_agents(const EnvSmem<MapT>& S, const StepParams& p, const int nl[2], uint8_t v, int lane) {
  const int PP = p.P, PS = p.PS;
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2)
    #pragma unroll 1
    for (int i = lane; i < nl[s2]; i += 32)
      if (S.flg[s2][i] & F_ALIVE) S.scr[CELLP((unsigned)S.pos[s2][i])] = v;
  const int G = p.G;
  #pragma unroll 1
  for (int i = lane; i < p.n_walls; i += 32) S.scr[CELLXY(p.wall_cells[i] / G, p.wall_cells[i] % G)] = v;  // walls are never free (STAG:1033-1037)
  __syncwarp();
}

// number of cells no live agent stands on (`all_positions - occupied_positions`, STAG:1037-1039)
template <typename MapT>
__device__ __noinline__ int count_free_cells(unsigned char* base, const StepParams& p, int nl0, int nl1, int lane) {
  const EnvSmem<MapT> S = carve<MapT>(base, p);
  const int G = p.G, GG = p.GG, PP = p.P, PS = p.PS;
  const int nl[2] = {nl0, nl1};
  mark_agents(S, p, nl, 1, lane);
  int n_free = 0;
  for (int c0 = 0; c0 < GG; c0 += 32) {
    const int c = c0 + lane;
    const bool fr = c < GG && S.scr[CELLXY(c / G, c % G)] == 0;
    n_free += __popc(__ballot_sync(FULL, fr));
  }
  __syncwarp();
  mark_agents(S, p, nl, 0, lane);
  return n_free;
}

// spawn fallback (BASE:760-764): the k-th free cell in ascending cell order, k from the env's Philox spawn stream.
// Returns x << 8 | y, or -1 if no cell is free.
template <typename MapT>
__device__ __noinline__ int philox_free_cell(unsigned char* base, const StepParams& p, int nl0, int nl1, unsigned draw, int lane) {
  const EnvSmem<MapT> S = carve<MapT>(base, p);
  const int G = p.G, GG = p.GG, PP = p.P, PS = p.PS;
  const int nl[2] = {nl0, nl1};
  mark_agents(S, p, nl, 1, lane);
  int n_free = 0;
  for (int c0 = 0; c0 < GG; c0 += 32) {
    const int c = c0 + lane;
    const bool fr = c < GG && S.scr[CELLXY(c / G, c % G)] == 0;
    n_free += __popc(__ballot_sync(FULL, fr));
  }
  int found = -1;
  if (n_free > 0) {
    int kth = (int)ppg_bounded(draw, (unsigned)n_free);
    for (int c0 = 0; c0 < GG; c0 += 32) {
      const int c = c0 + lane;
      const bool fr = c < GG && S.scr[CELLXY(c / G, c % G)] == 0;
      const unsigned fm = __ballot_sync(FULL, fr);
      const int cnt = __popc(fm);
      if (kth < cnt) {
        const int cc = c0 + (int)__fns(fm, 0, kth + 1);
        found = ((cc / G) << 8) | (cc % G);
        break;
      }
      kth -= cnt;
    }
  }
  __syncwarp();
  mark_agents(S, p, nl, 0, lane);
  return found;
}


// ------------------------------------------------------------------------------------------------
// deterministic row allocation: publication of an env's (live, births) counts (DESIGN.md §3.4)
// ------------------------------------------------------------------------------------------------
// Every env stores its two epoch-tagged words (cntA: rows it needs in the NEXT output, cntB: newborn rows of THIS
// output) and adds the same pairs to the accumulator of its 32-env block with ONE 64-bit atomic per pair:
//   acc = contributors << 56 | first << 28 | second.
// The atomic's return value tells the env whether it was the block's last contributor; the last one knows the block sum
// (returned value + its own), publishes it as tagged words (sum1), clears the accumulator for the next launch and adds the
// sum to the accumulator of the 1024-env group, and so on up to the totals.  Readers validate every word by its tag, so no
// fence is needed anywhere, and the two atomics are issued long before their results are looked at (publish_begin right
// after the env's counts are known, publish_end after its rows are written): nobody waits on this path.
#define ACC_ONE (1ULL << 56)
#define ACC_M28 0xFFFFFFFULL
#define ACC_M56 ((1ULL << 56) - 1ULL)

//
// Big envs first: env-steps differ 4x in duration (mostly with the number of agents) and a launch has only 1.4 - 7 envs per
// resident warp, so in index order the kernel's last third is a handful of warps finishing big envs they happened to get
// late.  Every env therefore also enters itself into the ORDER of the next launch (perm[par], ticket -> env): envs with
// more agents than `big` (5/4 of the mean) fill it from the front, the others from the back, each through one cursor
// atomic.  The launch's last publisher tags the order with the epoch and clears the other parity's cursors.  Results never
// depend on the order envs are worked on (rows are allocated by env index).  Only for kernels in which no env ever waits
// for another one (BASE / STAG two-kernel step; p.perm == nullptr elsewhere): a waiting env relies on ticket order = env order.
__device__ __forceinline__ void publish_begin(const StepParams& p, int env, int par, unsigned epoch, const int next_live[2],
                                              const int births[2], int lane, unsigned long long& rA, unsigned long long& rB, int big) {
  if (lane == 0) {
    st_volatile(p.cntA[par] + env, TAG(epoch, (next_live[0] << 16) | next_live[1]));
    st_volatile(p.cntB[par] + env, TAG(epoch, (births[0] << 16) | births[1]));
    unsigned long long* acc = p.acc1 + 2 * (size_t)(env >> 5);
    rA = atomicAdd(acc, ACC_ONE | ((unsigned long long)next_live[0] << 28) | (unsigned long long)next_live[1]);
    rB = atomicAdd(acc + 1, ACC_ONE | ((unsigned long long)births[0] << 28) | (unsigned long long)births[1]);
    if (p.perm[par] != nullptr) {
      const bool front = next_live[0] + next_live[1] > big;
      const unsigned pos = atomicAdd(p.perm_cursor + 2 * par + (front ? 0 : 1), 1u);
      p.perm[par][front ? (int)pos : p.B - 1 - (int)pos] = env;
    }
  }
}

// one chain (c = 0: live counts, c = 1: births) from the block level upwards; lane 0 only
static __device__ __noinline__ bool publish_chain(const StepParams& p, int env, int par, unsigned epoch, int c, unsigned long long r, unsigned long long mine,
                                           int n_blk, int n_grp, int n_old0, int n_old1) {
  const int blk = env >> 5, grp = env >> 10;
  if ((int)(r >> 56) + 1 != min(32, p.B - (blk << 5))) return false;
  unsigned long long tot = (r + mine) & ACC_M56;  // this env was the last of its block
  p.acc1[2 * (size_t)blk + c] = 0ULL;
  st_volatile(p.sum1[par] + (size_t)blk * 4 + 2 * c, TAG(epoch, (unsigned)(tot >> 28)));
  st_volatile(p.sum1[par] + (size_t)blk * 4 + 2 * c + 1, TAG(epoch, (unsigned)(tot & ACC_M28)));
  unsigned long long r2 = atomicAdd(p.acc2 + 2 * (size_t)grp + c, ACC_ONE | tot);
  if ((int)(r2 >> 56) + 1 != min(32, n_blk - (grp << 5))) return false;
  tot = (r2 + tot) & ACC_M56;  // last block of its group
  p.acc2[2 * (size_t)grp + c] = 0ULL;
  st_volatile(p.sum2[par] + (size_t)grp * 4 + 2 * c, TAG(epoch, (unsigned)(tot >> 28)));
  st_volatile(p.sum2[par] + (size_t)grp * 4 + 2 * c + 1, TAG(epoch, (unsigned)(tot & ACC_M28)));
  r2 = atomicAdd(p.acc3 + c, ACC_ONE | tot);
  if ((int)(r2 >> 56) + 1 != n_grp) return false;
  tot = (r2 + tot) & ACC_M56;  // last group: totals of this output (births) / of the next one (live)
  p.acc3[c] = 0ULL;
  p.totals[par * 4 + 2 * c] = (int)(tot >> 28);
  p.totals[par * 4 + 2 * c + 1] = (int)(tot & ACC_M28);
  if (c == 0) {
    p.n_rows[0] = n_old0; p.n_rows[1] = n_old1;
    p.old_off[0][p.B] = n_old0; p.old_off[1][p.B] = n_old1;
    if (p.perm[par] != nullptr) {  // every env has entered itself into the next launch's order
      p.perm_tag[par] = epoch;
      p.perm_cursor[2 * (par ^ 1)] = 0u; p.perm_cursor[2 * (par ^ 1) + 1] = 0u;  // idle during this launch, used by the next one
    }
  } else {
    p.n_rows[2] = (int)(tot >> 28); p.n_rows[3] = (int)(tot & ACC_M28);
  }
  return true;
}

// returns (lane 0) whether this env published the last live count of the launch: every env's cntA word is then in place
__device__ __forceinline__ bool publish_end(const StepParams& p, int env, int par, unsigned epoch, const int next_live[2], const int births[2],
                                            int n_blk, int n_grp, const int n_old_total[2], int lane, unsigned long long rA, unsigned long long rB) {
  bool all_live = false;
  if (lane == 0) {
    const int bsz = min(32, p.B - ((env >> 5) << 5));
    if ((int)(rA >> 56) + 1 == bsz)
      all_live = publish_chain(p, env, par, epoch, 0, rA, ACC_ONE | ((unsigned long long)next_live[0] << 28) | (unsigned long long)next_live[1], n_blk, n_grp,
                               n_old_total[0], n_old_total[1]);
    if ((int)(rB >> 56) + 1 == bsz)
      publish_chain(p, env, par, epoch, 1, rB, ACC_ONE | ((unsigned long long)births[0] << 28) | (unsigned long long)births[1], n_blk, n_grp,
                    n_old_total[0], n_old_total[1]);
  }
  return all_live;
}

__device__ __forceinline__ void publish_counts(const StepParams& p, int env, int par, unsigned epoch, const int next_live[2],
                                               const int births[2], int n_blk, int n_grp, const int n_old_total[2], int lane) {
  unsigned long long rA = 0, rB = 0;
  publish_begin(p, env, par, epoch, next_live, births, lane, rA, rB, (n_old_total[0] + n_old_total[1]) / p.B * 5 / 4);
  publish_end(p, env, par, epoch, next_live, births, n_blk, n_grp, n_old_total, lane, rA, rB);
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------
// hand-over of a finished env to the observation kernel (completion queue, DESIGN.md §3.5)
// ------------------------------------------------------------------------------------------------
// The queue slot is drawn early (queue_reserve, together with the publication atomics: one round trip for all three);
// the entry itself may only appear after the env's image and labels are visible, i.e. after a fence that follows those
// stores.  The fence is NOT executed at the end of the env: the warp first issues the global loads of its NEXT env and
// then fences (queue_push from the top of the loop), so that the wait for the store acknowledgements and the wait for the
// loads are one wait instead of two.  `pend` = slot + 1 of the env waiting to be pushed (0: none), lane 0 only.
__device__ __forceinline__ unsigned long long queue_reserve(const StepParams& p, int lane) {
  unsigned long long slot = 0;
  if (lane == 0) slot = atomicAdd(p.q_tail, 1ULL) - p.q_base;
  return slot;
}
__device__ __forceinline__ void queue_push(const StepParams& p, unsigned long long& pend, int& pend_env, int lane) {
  __syncwarp();
  if (lane == 0 && pend != 0ULL) {
    __threadfence();
    st_volatile(p.queue + (pend - 1ULL), TAG(p.epoch, pend_env));
    pend = 0ULL;
  }
}

// ------------------------------------------------------------------------------------------------
// the env loop of a persistent step warp (DESIGN.md §3.4-3.5); the variant's simulation runs between env_begin and
// env_publish, its rows between env_publish and env_rows_done
// ------------------------------------------------------------------------------------------------
// Envs come from the ticket counter; after the first one lane 0 draws the warp's next ticket while the current env is still
// being finished (env_publish: late enough that the schedule stays dynamic, early enough that the atomic's round trip is never
// waited for).  Tickets are handed out in env order to warps that are running, so an env that waits for the publication of a
// lower env (ECO's episode-end rows, the one-kernel step) always waits for a running warp.
struct EnvLoop {
  unsigned epoch;
  int par;                  // epoch & 1: the parity of the count words this launch publishes
  int n_blk, n_grp;         // 32-env blocks, 1024-env groups
  int n_old_total[2];       // rows of the previous output
  bool order;               // the kernel may take its envs out of index order (perm, static_first)
  const int32_t* perm;      // ticket -> env: big envs first when the previous launch left an order (publish_begin), else index order
  int env_next;             // lane 0: the warp's next env
  unsigned long long q_slot, pubA, pubB;  // lane 0: the env's completion-queue slot and row-allocation atomics (env_publish)
  unsigned long long pend;  // lane 0: completion-queue slot + 1 of the env whose hand-over is still owed (queue_push)
  int pend_env;
};

// order: only for kernels in which no env ever waits for another one (publish_begin)
__device__ __forceinline__ EnvLoop env_loop(const StepParams& p, bool order) {
  EnvLoop L;
  L.order = order;
  L.epoch = p.epoch;
  L.par = (int)(L.epoch & 1u);
  L.n_blk = (p.B + 31) >> 5;
  L.n_grp = (p.B + 1023) >> 10;
  L.n_old_total[0] = p.totals[(L.par ^ 1) * 4 + 0];
  L.n_old_total[1] = p.totals[(L.par ^ 1) * 4 + 1];
  L.perm = (order && p.perm[L.par ^ 1] != nullptr && p.perm_tag[L.par ^ 1] == L.epoch - 1u) ? p.perm[L.par ^ 1] : nullptr;
  L.env_next = 0;
  L.pend = 0ULL;
  L.pend_env = 0;
  return L;
}

// lane 0: draws the warp's next env (first: the warp's first one).  static_first: the first ticket of a warp is its CTA index —
// 2960 atomics on one address at kernel start cost the last warp ~7 us; the counter then hands out the tickets from min(grid, B) on.
__device__ __forceinline__ void next_ticket(const StepParams& p, EnvLoop& L, bool first) {
  const int t = !(L.order && p.static_first) ? (int)(atomicAdd(p.ticket, 1ULL) - p.ticket_base)
                : first ? min((int)blockIdx.x, p.B) : min((int)gridDim.x, p.B) + (int)(atomicAdd(p.ticket, 1ULL) - p.ticket_base);
  L.env_next = L.perm != nullptr && t < p.B ? L.perm[t] : t;
}

// Start of an env whose header and first list entries have been requested: its first old row (the previous launch published
// how many rows every env needs now), the hand-over of the warp's previous env (its stores were issued a round trip ago, the
// fence finds them acknowledged) and the mode (0 idle, 1 reset, 2 step).  Reset / idle envs know their counts up front
// (`founders`, no births) and publish them before doing any work, so that later envs waiting for their newborn-row prefix
// never wait for a reset.
template <bool SPLIT>
__device__ __forceinline__ int env_begin(const StepParams& p, EnvLoop& L, int env, unsigned state, const int founders[2], int old_base[2],
                                         int next_live[2], int lane) {
  if (!prefix_before(p.cntA[L.par ^ 1], p.sum1[L.par ^ 1], p.sum2[L.par ^ 1], 0, env, L.epoch - 1u, false, lane, old_base[0], old_base[1])) {
    if (lane == 0) atomicOr(p.error, 2u);  // the host did not prepare the counts of the previous output
  }
  if (SPLIT) queue_push(p, L.pend, L.pend_env, lane);
  const int mode = (state & ST_NEEDS_RESET) ? 1 : ((state & ST_IDLE) ? 0 : 2);
  if (mode != 2) {
    const int births[2] = {0, 0};
    if (mode == 1) { next_live[0] = founders[0]; next_live[1] = founders[1]; }
    publish_counts(p, env, L.par, L.epoch, next_live, births, L.n_blk, L.n_grp, L.n_old_total, lane);
  }
  return mode;
}

// After the simulation: four atomics back to back, nobody waits for them here — the warp's next env (`tickets`), this env's
// slot in the completion queue and the two accumulators of the row allocation (results looked at in env_rows_done).
// `big`: the big-env bound of publish_begin.
template <bool SPLIT>
__device__ __forceinline__ void env_publish(const StepParams& p, EnvLoop& L, int env, int mode, const int next_live[2], const int births[2],
                                            int big, bool tickets, int lane) {
  if (tickets && lane == 0) next_ticket(p, L, false);
  L.q_slot = L.pubA = L.pubB = 0ULL;
  if (SPLIT) L.q_slot = queue_reserve(p, lane);
  if (mode == 2) publish_begin(p, env, L.par, L.epoch, next_live, births, lane, L.pubA, L.pubB, big);
}

// one-kernel step: the first newborn row of the env depends on the births of every env before it; by now (all other work of
// the env is done) the predecessors have normally published theirs.  The two-kernel step never waits: the observation kernel
// places the newborn rows (nb_info).
__device__ __forceinline__ void newborn_base(const StepParams& p, const EnvLoop& L, int env, int lane, int new_base[2]) {
  int nb0 = 0, nb1 = 0;
  if (!prefix_before(p.cntB[L.par], p.sum1[L.par], p.sum2[L.par], 2, env, L.epoch, true, lane, nb0, nb1)) {
    if (lane == 0) atomicOr(p.error, 1u);
  }
  new_base[0] = L.n_old_total[0] + nb0;
  new_base[1] = L.n_old_total[1] + nb1;
}

// After the rows of a reset or stepped env: the rest of its publication, its newborn-row range and (two-kernel step) its image,
// dumped before the caller un-writes the maps.
template <bool SPLIT>
__device__ __forceinline__ void env_rows_done(const StepParams& p, const EnvLoop& L, unsigned char* sbase, int env, int mode, bool keep,
                                              const int old_base[2], const int n[2], const int births[2], const int new_base[2],
                                              const int next_live[2], int lane) {
  if (mode == 2) publish_end(p, env, L.par, L.epoch, next_live, births, L.n_blk, L.n_grp, L.n_old_total, lane, L.pubA, L.pubB);
  if (lane < 2) {
    const int nb = lane == 0 ? births[0] : births[1];
    if (!SPLIT) p.new_off[lane][env] = nb > 0 ? (lane == 0 ? new_base[0] : new_base[1]) : 0;
    p.new_cnt[lane][env] = nb;
  }
  if (SPLIT) dump_image(sbase, p, env, mode, keep, old_base, n, births, lane);
}

// an idle env: no rows, a header-only image
template <bool SPLIT>
__device__ __forceinline__ void env_idle(const StepParams& p, unsigned char* sbase, int env, const int old_base[2], int lane) {
  if (lane < 2) {
    p.new_off[lane][env] = 0;
    p.new_cnt[lane][env] = 0;
  }
  const int none[2] = {0, 0};
  if (SPLIT) dump_image(sbase, p, env, 0, false, old_base, none, none, lane);
}

// counters of one env-step behind PPG_STAT_*
struct EnvStats {
  unsigned starved[2], eaten, grass, fallback;
  unsigned attempts;  // STAG's capture attempts, 0 elsewhere
};

// lane k adds statistic k (selects, no divergent switch)
__device__ __forceinline__ void add_stats(const StepParams& p, int env, int mode, const int n[2], const int births[2], bool over, bool trunc,
                                          unsigned step, const EnvStats& st, int lane) {
  if (lane < PPG_N_STATS) {
    unsigned add = 0;
    if (mode == 2) {
      add = lane == PPG_STAT_ENV_STEPS ? 1u : add;
      add = lane == PPG_STAT_AGENT_STEPS ? (unsigned)(n[0] + n[1]) : add;
      add = lane == PPG_STAT_EPISODES ? (unsigned)over : add;
      add = lane == PPG_STAT_EPISODE_STEPS ? (over ? step : 0u) : add;
      add = lane == PPG_STAT_BIRTHS_PRED ? (unsigned)births[0] : add;
      add = lane == PPG_STAT_BIRTHS_PREY ? (unsigned)births[1] : add;
      add = lane == PPG_STAT_STARVED_PRED ? st.starved[0] : add;
      add = lane == PPG_STAT_STARVED_PREY ? st.starved[1] : add;
      add = lane == PPG_STAT_EATEN_PREY ? st.eaten : add;
      add = lane == PPG_STAT_GRASS_EATEN ? st.grass : add;
      add = lane == PPG_STAT_TRUNCATED ? (unsigned)trunc : add;
      add = lane == PPG_STAT_SPAWN_FALLBACK ? st.fallback : add;
      add = lane == PPG_STAT_CAPTURE_ATTEMPTS ? st.attempts : add;
    }
    if (lane == PPG_STAT_ROWS_PRED) add = n[0] + births[0];
    if (lane == PPG_STAT_ROWS_PREY) add = n[1] + births[1];
    if (add) atomicAdd(p.counters + (size_t)env * PPG_N_STATS + lane, add);  // RED: nobody waits for the old value
  }
}

// End of an env: its per-env outputs, then its hand-over to the observation kernel is owed (made from the top of the warp's next
// env or after the loop, queue_push).  `count`: the agent counts the env reports, written unless `write_count` is false.
template <bool SPLIT>
__device__ __forceinline__ void env_end(const StepParams& p, EnvLoop& L, int env, int mode, const int n[2], const int births[2],
                                        unsigned env_flags, const EnvHdr& h, long long t_env0, unsigned t_ns0, const int count[2],
                                        bool write_count, int lane) {
  if (lane == 0) {
    p.env_cycles[env] = make_uint4((unsigned)(clock64() - t_env0), (unsigned)mode | ((unsigned)(births[0] + births[1]) << 8) | ((unsigned)(n[0] + n[1]) << 16), t_ns0, smid());
    p.env_flags[env] = (uint8_t)env_flags;
    p.env_status[env] = h.status;
    p.env_step[env] = h.step;
    if (write_count) {
      p.env_count[2 * env] = count[0];
      p.env_count[2 * env + 1] = count[1];
    }
  }
  if (SPLIT && lane == 0) { L.pend = L.q_slot + 1ULL; L.pend_env = env; }
  __syncwarp();
}

}  // namespace ppg
