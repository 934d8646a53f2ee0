/**
 * \file update_kernels.cu
 * \brief K_update: the GPU-resident server's push handler, fused (sm_100a).
 *
 * The reference aggregates on the CPU with `store[key] += val`
 * (include/ps/kv_app.h:441-447) and leaves the optimizer to the consumer. Here
 * one memory-bound pass per parameter shard does everything the server owes its
 * workers for a round:
 *     g      = grad_scale * sum_w dequant(slot_w)      (bf16 | fp8-block | f32 slots, or ONE
 *              multimem.ld_reduce stream: the NVSwitch sums the W workers' symmetric buffers)
 *     m,v,p  = AdamW / SGD-momentum on fp32 state
 *     out_k  = bf16(p)  for every destination k       (<= 9: local + W workers)
 * The destinations may be peer-mapped worker parameter buffers, so the update
 * is also the pull reply: parameters leave the SM once and fan out over NVLink
 * as plain 16-byte stores — there is no intermediate shard copy to re-read.
 *
 * Roofline: per element it must read W*g + 12 B (master, m, v) and write 12 B +
 * 2 B per destination; no reuse, so the target is HBM / NVLink bandwidth.
 * Each thread-iteration handles 8 elements: 16-byte loads for bf16 grads, 8-byte
 * for fp8, 2 x 16-byte for each fp32 state array, 16-byte bf16 stores.
 */
#include <cuda_runtime.h>

#include <atomic>

#include <cstdint>
#include <cstdlib>

#include "kernels/ps_kernels.h"
#include "kernels/update_math.cuh"

namespace ps_kernels_internal {
void CountLaunch(int n);
int NumSMs();
int CurrentDevice();
}

namespace {

constexpr int kThreads = 256;
constexpr int kMaxDevices = 16;  // as in NumSMs(): per-device caches (CurrentDevice() maps others to 0)

struct UpdateDev {
  size_t n;
  int num_grads;
  int num_outs;
  const void* grads[PS_MAX_FANIN];
  float* master;
  float* m;
  float* v;
  void* outs[PS_MAX_FANOUT];
  void* mc_out;     // NVLS multicast destination (bf16), or null
  int body_outs;    // unicast outputs written in the vector body
};

/*! one store, replicated by the NVSwitch to every GPU bound to the multicast object */
__device__ __forceinline__ void multimem_st16(void* p, const int4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p),
               "f"(__int_as_float(v.x)), "f"(__int_as_float(v.y)), "f"(__int_as_float(v.z)),
               "f"(__int_as_float(v.w))
               : "memory");
}
/*! sum over every GPU bound to the multicast object, reduced by the NVSwitch in fp32 */
__device__ __forceinline__ int4 multimem_ld_reduce16(const void* p) {
  int4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.v4.bf16x2 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p)
               : "memory");
  return r;
}
__device__ __forceinline__ uint32_t multimem_ld_reduce4(const void* p) {
  uint32_t r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.acc::f32.bf16x2 %0, [%1];"
               : "=r"(r)
               : "l"(p)
               : "memory");
  return r;
}
/*! \brief sum of 8 consecutive gradient elements starting at 8*i over all W slots */
template <int FMT>
__device__ __forceinline__ void gather_grads(const UpdateDev& a, size_t i, float* g) {
#pragma unroll
  for (int j = 0; j < 8; ++j) g[j] = 0.f;
  if (FMT == PS_GRAD_MC_BF16) {
    const int4 q = multimem_ld_reduce16(static_cast<const unsigned char*>(a.grads[0]) + i * 16);
    float2 f;
    f = bf2(q.x); g[0] = f.x; g[1] = f.y;
    f = bf2(q.y); g[2] = f.x; g[3] = f.y;
    f = bf2(q.z); g[4] = f.x; g[5] = f.y;
    f = bf2(q.w); g[6] = f.x; g[7] = f.y;
    return;
  }
  const size_t npad = (a.n + 31) / 32 * 32;
#pragma unroll 1
  for (int w = 0; w < a.num_grads; ++w) {
    const unsigned char* base = static_cast<const unsigned char*>(a.grads[w]);
    if (FMT == PS_GRAD_BF16) {
      const int4 q = ldg16(base + i * 16);
      float2 f;
      f = bf2(q.x); g[0] += f.x; g[1] += f.y;
      f = bf2(q.y); g[2] += f.x; g[3] += f.y;
      f = bf2(q.z); g[4] += f.x; g[5] += f.y;
      f = bf2(q.w); g[6] += f.x; g[7] += f.y;
    } else if (FMT == PS_GRAD_FP8BLOCK) {
      const uint2 q = ldg8(base + i * 8);
      const float s = e8m0(base[npad + (i >> 2)]);
      float t[8];
      fp8x4_to_f32(q.x, s, t);
      fp8x4_to_f32(q.y, s, t + 4);
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] += t[j];
    } else {
      const int4 q0 = ldg16(base + i * 32), q1 = ldg16(base + i * 32 + 16);
      g[0] += __int_as_float(q0.x); g[1] += __int_as_float(q0.y);
      g[2] += __int_as_float(q0.z); g[3] += __int_as_float(q0.w);
      g[4] += __int_as_float(q1.x); g[5] += __int_as_float(q1.y);
      g[6] += __int_as_float(q1.z); g[7] += __int_as_float(q1.w);
    }
  }
}

template <int FMT>
__device__ __forceinline__ float gather_one(const UpdateDev& a, size_t e) {
  float g = 0.f;
  if (FMT == PS_GRAD_MC_BF16) {
    const float2 f = bf2(multimem_ld_reduce4(static_cast<const unsigned char*>(a.grads[0]) + (e & ~size_t(1)) * 2));
    return (e & 1) ? f.y : f.x;
  }
  const size_t npad = (a.n + 31) / 32 * 32;
  for (int w = 0; w < a.num_grads; ++w) {
    const unsigned char* base = static_cast<const unsigned char*>(a.grads[w]);
    if (FMT == PS_GRAD_BF16) {
      g += __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[e]);
    } else if (FMT == PS_GRAD_FP8BLOCK) {
      const __half_raw h = __nv_cvt_fp8_to_halfraw(base[e], __NV_E4M3);
      g += __half2float(__half(h)) * e8m0(base[npad + (e >> 5)]);
    } else {
      g += reinterpret_cast<const float*>(base)[e];
    }
  }
  return g;
}

template <int FMT, int OPT, bool OUT_F32>
__global__ void __launch_bounds__(kThreads)
k_update(const UpdateDev a, const ps_opt_params o) {
  const size_t n8 = a.n / 8;
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  for (size_t i = static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x; i < n8; i += stride) {
    // issue the state loads first so they overlap the W gradient loads
    float4 p0 = ldf4(a.master + i * 8), p1 = ldf4(a.master + i * 8 + 4);
    float4 m0 = ldf4(a.m + i * 8), m1 = ldf4(a.m + i * 8 + 4);
    float4 v0 = make_float4(0, 0, 0, 0), v1 = v0;
    if (OPT == PS_OPT_ADAMW) {
      v0 = ldf4(a.v + i * 8);
      v1 = ldf4(a.v + i * 8 + 4);
    }
    float g[8];
    gather_grads<FMT>(a, i, g);
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] *= o.grad_scale;
    step<OPT>(p0.x, m0.x, v0.x, g[0], o); step<OPT>(p0.y, m0.y, v0.y, g[1], o);
    step<OPT>(p0.z, m0.z, v0.z, g[2], o); step<OPT>(p0.w, m0.w, v0.w, g[3], o);
    step<OPT>(p1.x, m1.x, v1.x, g[4], o); step<OPT>(p1.y, m1.y, v1.y, g[5], o);
    step<OPT>(p1.z, m1.z, v1.z, g[6], o); step<OPT>(p1.w, m1.w, v1.w, g[7], o);
    stf4(a.master + i * 8, p0); stf4(a.master + i * 8 + 4, p1);
    stf4(a.m + i * 8, m0); stf4(a.m + i * 8 + 4, m1);
    if (OPT == PS_OPT_ADAMW) {
      stf4(a.v + i * 8, v0);
      stf4(a.v + i * 8 + 4, v1);
    }
    if (OUT_F32) {
#pragma unroll 1
      for (int k = 0; k < a.body_outs; ++k) {
        stf4(static_cast<float*>(a.outs[k]) + i * 8, p0);
        stf4(static_cast<float*>(a.outs[k]) + i * 8 + 4, p1);
      }
    } else {
      int4 out;
      out.x = pk(p0.x, p0.y); out.y = pk(p0.z, p0.w);
      out.z = pk(p1.x, p1.y); out.w = pk(p1.z, p1.w);
#pragma unroll 1
      for (int k = 0; k < a.body_outs; ++k) st16(static_cast<char*>(a.outs[k]) + i * 16, out);
      if (a.mc_out) multimem_st16(static_cast<char*>(a.mc_out) + i * 16, out);
    }
  }
  // ragged tail (< 8 elements) handled by the first threads of block 0
  if (blockIdx.x == 0) {
    const size_t e = n8 * 8 + threadIdx.x;
    if (e < a.n) {
      float p = a.master[e], m = a.m[e], v = OPT == PS_OPT_ADAMW ? a.v[e] : 0.f;
      const float g = gather_one<FMT>(a, e) * o.grad_scale;
      step<OPT>(p, m, v, g, o);
      a.master[e] = p;
      a.m[e] = m;
      if (OPT == PS_OPT_ADAMW) a.v[e] = v;
      for (int k = 0; k < a.num_outs; ++k) {
        if (OUT_F32) static_cast<float*>(a.outs[k])[e] = p;
        else static_cast<__nv_bfloat16*>(a.outs[k])[e] = __float2bfloat16_rn(p);
      }
    }
  }
}


// ---------------------------------------------------------------------------
// K_update, TMA flavour (PS_UPDATE_TMA=1, experimental until it has run on hardware)
//
// The register-file version above can keep ~28 KB of loads in flight per SM (4 CTAs x 256 threads
// x one 8-element group); its remaining stall is the first use of a load. Here one elected
// thread per CTA streams whole tiles — fp32 master / m / v and the W gradient slots — into shared
// memory with cp.async.bulk behind mbarriers, kTmaStages - 1 tiles (up to ~110 KB) ahead of the
// 256 consumer threads, which compute from shared memory and write results with plain vector
// stores (stores do not stall). One persistent CTA per SM.
//   tile   = 2048 elements; thread t owns elements [4t, 4t+4) and [1024+4t, 1024+4t+4) of it,
//            so every shared-memory access of a warp is contiguous (no bank conflicts)
//   stage  = 24 KB of state + W x (4 KB bf16 | 2 KB fp8 | 8 KB f32) of gradients
//   tail   = the elements after the last full tile are done by CTA 0 with the scalar path
// ---------------------------------------------------------------------------
constexpr int kTile = 2048;
constexpr int kTmaStagesU = 3;

__device__ __forceinline__ uint32_t smem_addr(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init_u(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_u(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait_u(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(smem_addr(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void bulk_load_u(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_addr(smem_dst)),
      "l"(gsrc), "r"(bytes), "r"(smem_addr(bar))
      : "memory");
}
__device__ __forceinline__ void st8(void* p, uint32_t a, uint32_t b) {
  asm volatile("st.global.L1::no_allocate.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void multimem_st8(void* p, uint32_t a, uint32_t b) {
  asm volatile("multimem.st.relaxed.sys.global.v2.f32 [%0], {%1,%2};" ::"l"(p), "f"(__uint_as_float(a)),
               "f"(__uint_as_float(b))
               : "memory");
}

template <int FMT>
__host__ __device__ constexpr int GradTileBytes() {
  return FMT == PS_GRAD_BF16 ? kTile * 2 : (FMT == PS_GRAD_FP8BLOCK ? kTile : kTile * 4);
}

template <int FMT, int OPT>
__global__ void __launch_bounds__(kThreads, 1)
k_update_tma(const UpdateDev a, const ps_opt_params o) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t full[kTmaStagesU];
  constexpr int kStateBytes = kTile * 4;
  constexpr int kGradBytes = GradTileBytes<FMT>();
  const int W = a.num_grads;
  const int stage_bytes = 3 * kStateBytes + W * kGradBytes;
  const size_t n_tiles = a.n / kTile;
  const size_t first = blockIdx.x, stride = gridDim.x;
  const size_t mine = first < n_tiles ? (n_tiles - first + stride - 1) / stride : 0;
  const int tid = threadIdx.x;
  if (tid == 0) {
    for (int s = 0; s < kTmaStagesU; ++s) mbar_init_u(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // producer (thread 0): all loads of my k-th tile into its stage
  auto issue = [&](size_t k) {
    const int s = static_cast<int>(k % kTmaStagesU);
    const size_t e0 = (first + k * stride) * static_cast<size_t>(kTile);
    unsigned char* st = smem + static_cast<size_t>(s) * stage_bytes;
    mbar_expect_u(&full[s], static_cast<uint32_t>(OPT == PS_OPT_ADAMW ? stage_bytes : stage_bytes - kStateBytes));
    bulk_load_u(st, a.master + e0, kStateBytes, &full[s]);
    bulk_load_u(st + kStateBytes, a.m + e0, kStateBytes, &full[s]);
    if (OPT == PS_OPT_ADAMW) bulk_load_u(st + 2 * kStateBytes, a.v + e0, kStateBytes, &full[s]);
    for (int w = 0; w < W; ++w) {
      const unsigned char* g = static_cast<const unsigned char*>(a.grads[w]);
      const size_t goff = FMT == PS_GRAD_BF16 ? e0 * 2 : (FMT == PS_GRAD_FP8BLOCK ? e0 : e0 * 4);
      bulk_load_u(st + 3 * kStateBytes + w * kGradBytes, g + goff, kGradBytes, &full[s]);
    }
  };
  if (tid == 0) {
    for (size_t k = 0; k < mine && k < static_cast<size_t>(kTmaStagesU - 1); ++k) issue(k);
  }

  const size_t npad = (a.n + 31) / 32 * 32;
  for (size_t j = 0; j < mine; ++j) {
    const int s = static_cast<int>(j % kTmaStagesU);
    const unsigned char* st = smem + static_cast<size_t>(s) * stage_bytes;
    mbar_wait_u(&full[s], static_cast<uint32_t>((j / kTmaStagesU) & 1));
    const size_t e0 = (first + j * stride) * static_cast<size_t>(kTile);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int le = h * (kTile / 2) + 4 * tid;  // first of my 4 elements inside the tile
      float4 p = *reinterpret_cast<const float4*>(st + le * 4);
      float4 m = *reinterpret_cast<const float4*>(st + kStateBytes + le * 4);
      float4 v = make_float4(0, 0, 0, 0);
      if (OPT == PS_OPT_ADAMW) v = *reinterpret_cast<const float4*>(st + 2 * kStateBytes + le * 4);
      float g[4] = {0.f, 0.f, 0.f, 0.f};
      for (int w = 0; w < W; ++w) {
        const unsigned char* gs = st + 3 * kStateBytes + w * kGradBytes;
        if (FMT == PS_GRAD_BF16) {
          const uint2 q = *reinterpret_cast<const uint2*>(gs + le * 2);
          float2 f;
          f = bf2(q.x); g[0] += f.x; g[1] += f.y;
          f = bf2(q.y); g[2] += f.x; g[3] += f.y;
        } else if (FMT == PS_GRAD_FP8BLOCK) {
          const uint32_t q = *reinterpret_cast<const uint32_t*>(gs + le);
          const unsigned char* base = static_cast<const unsigned char*>(a.grads[w]);
          const float sc = e8m0(base[npad + ((e0 + le) >> 5)]);  // scales are tiny: straight from global
          float t[4];
          fp8x4_to_f32(q, sc, t);
          g[0] += t[0]; g[1] += t[1]; g[2] += t[2]; g[3] += t[3];
        } else {
          const float4 q = *reinterpret_cast<const float4*>(gs + le * 4);
          g[0] += q.x; g[1] += q.y; g[2] += q.z; g[3] += q.w;
        }
      }
      step<OPT>(p.x, m.x, v.x, g[0] * o.grad_scale, o); step<OPT>(p.y, m.y, v.y, g[1] * o.grad_scale, o);
      step<OPT>(p.z, m.z, v.z, g[2] * o.grad_scale, o); step<OPT>(p.w, m.w, v.w, g[3] * o.grad_scale, o);
      const size_t e = e0 + le;
      stf4(a.master + e, p);
      stf4(a.m + e, m);
      if (OPT == PS_OPT_ADAMW) stf4(a.v + e, v);
      const uint32_t lo = pk(p.x, p.y), hi = pk(p.z, p.w);
#pragma unroll 1
      for (int k = 0; k < a.body_outs; ++k) st8(static_cast<char*>(a.outs[k]) + e * 2, lo, hi);
      if (a.mc_out) multimem_st8(static_cast<char*>(a.mc_out) + e * 2, lo, hi);
    }
    __syncthreads();  // every thread has read stage s (and the stage of tile j-1 long before)
    if (tid == 0 && j + kTmaStagesU - 1 < mine) issue(j + kTmaStagesU - 1);
  }

  // elements after the last full tile: scalar path, CTA 0
  if (blockIdx.x == 0) {
    for (size_t e = n_tiles * kTile + tid; e < a.n; e += kThreads) {
      float p = a.master[e], m = a.m[e], v = OPT == PS_OPT_ADAMW ? a.v[e] : 0.f;
      const float g = gather_one<FMT>(a, e) * o.grad_scale;
      step<OPT>(p, m, v, g, o);
      a.master[e] = p;
      a.m[e] = m;
      if (OPT == PS_OPT_ADAMW) a.v[e] = v;
      for (int k = 0; k < a.num_outs; ++k) static_cast<__nv_bfloat16*>(a.outs[k])[e] = __float2bfloat16_rn(p);
    }
  }
}

template <int FMT>
__global__ void __launch_bounds__(kThreads)
k_sum(float* __restrict__ out, const UpdateDev a, float scale, int accumulate) {
  const size_t n8 = a.n / 8;
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  for (size_t i = static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x; i < n8; i += stride) {
    float g[8];
    gather_grads<FMT>(a, i, g);
    float4 o0 = make_float4(0, 0, 0, 0), o1 = o0;
    if (accumulate) {
      o0 = ldf4(out + i * 8);
      o1 = ldf4(out + i * 8 + 4);
    }
    o0.x += g[0] * scale; o0.y += g[1] * scale; o0.z += g[2] * scale; o0.w += g[3] * scale;
    o1.x += g[4] * scale; o1.y += g[5] * scale; o1.z += g[6] * scale; o1.w += g[7] * scale;
    stf4(out + i * 8, o0);
    stf4(out + i * 8 + 4, o1);
  }
  if (blockIdx.x == 0) {
    const size_t e = n8 * 8 + threadIdx.x;
    if (e < a.n) out[e] = (accumulate ? out[e] : 0.f) + gather_one<FMT>(a, e) * scale;
  }
}

int GridFor(size_t items, int max_ctas, int per_sm) {
  size_t want = (items + kThreads - 1) / kThreads;
  size_t cap = max_ctas > 0 ? static_cast<size_t>(max_ctas) : static_cast<size_t>(ps_kernels_internal::NumSMs()) * per_sm;
  if (want > cap) want = cap;
  return want < 1 ? 1 : static_cast<int>(want);
}

/*!
 * \brief which flavour runs a shard, decided by measurement on B200 (profiles/r2/r2_kernel_bench_*.txt,
 *        fraction of the 6571 GB/s copy roofline, 64 M elements, W = 1..4, fan-out 1..5):
 *          bf16 / f32 gradient slots   LDG 0.82-0.95   TMA-staged 0.93-1.01   -> TMA
 *          fp8-block gradient slots    LDG 0.82-0.90   TMA-staged 0.66-0.72   -> LDG (byte-wise decode out of
 *                                                                                shared memory bank-conflicts)
 *        A third flavour (two groups per thread, "x2") lost at W = 4 (0.72-0.76) and was removed.
 *        PS_UPDATE_TMA=0 / 1 forces one flavour for every format.
 */
template <int FMT>
bool UseTma() {
  static const int forced = [] {
    const char* v = getenv("PS_UPDATE_TMA");
    return v == nullptr ? -1 : (atoi(v) != 0 ? 1 : 0);
  }();
  if (forced >= 0) return forced == 1;
  return FMT == PS_GRAD_BF16 || FMT == PS_GRAD_F32;
}

template <int FMT, int OPT>
bool LaunchUpdateTmaImpl(const UpdateDev& d, const ps_opt_params& o, bool out_f32, int max_ctas, cudaStream_t st) {
  if (!UseTma<FMT>() || out_f32) return false;
  const size_t tiles = d.n / kTile;
  const int stage = 3 * kTile * 4 + d.num_grads * GradTileBytes<FMT>();
  const int smem = kTmaStagesU * stage;
  if (tiles < 4 || smem > 220 * 1024) return false;
  // (cp.async.bulk needs 16-byte aligned sources: ps_launch_update has refused anything else)
  // the attribute belongs to the current device: one flag per device and instantiation
  // (launches come from several threads, and a process may drive several GPUs)
  static std::atomic<bool> attr_set[kMaxDevices] = {};
  const int dev = ps_kernels_internal::CurrentDevice();
  if (!attr_set[dev].load(std::memory_order_acquire)) {
    cudaFuncSetAttribute(k_update_tma<FMT, OPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
    attr_set[dev].store(true, std::memory_order_release);
  }
  const int num_sms = ps_kernels_internal::NumSMs();
  int grid = static_cast<int>(tiles < static_cast<size_t>(num_sms) ? tiles : num_sms);
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  k_update_tma<FMT, OPT><<<grid, kThreads, smem, st>>>(d, o);
  return true;
}

/*! \brief true if the TMA flavour took the launch (bf16 outputs, enough full tiles, stage fits) */
template <int FMT, int OPT>
bool LaunchUpdateTma(const UpdateDev& d, const ps_opt_params& o, bool out_f32, int max_ctas, cudaStream_t st) {
  if constexpr (FMT == PS_GRAD_MC_BF16) {
    return false;  // the switch does the reduction inside the load; nothing to stage
  } else {
    return LaunchUpdateTmaImpl<FMT, OPT>(d, o, out_f32, max_ctas, st);
  }
}

template <int FMT, int OPT>
void LaunchUpdate(const UpdateDev& d, const ps_opt_params& o, bool out_f32, int grid,
                  cudaStream_t st) {
  if (LaunchUpdateTma<FMT, OPT>(d, o, out_f32, grid, st)) return;
  if (out_f32) k_update<FMT, OPT, true><<<grid, kThreads, 0, st>>>(d, o);
  else k_update<FMT, OPT, false><<<grid, kThreads, 0, st>>>(d, o);
}

}  // namespace

extern "C" int ps_launch_update(const ps_update_args* args, const ps_opt_params* opt, int max_ctas,
                                ps_stream_t stream_) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_);
  if (args->n == 0) return 0;
  if (args->num_grads < 1 || args->num_grads > PS_MAX_FANIN) return cudaErrorInvalidValue;
  if (args->num_outs < 0 || args->num_outs > PS_MAX_FANOUT) return cudaErrorInvalidValue;
  UpdateDev d;
  d.n = args->n;
  d.num_grads = args->num_grads;
  d.num_outs = args->num_outs;
  for (int i = 0; i < PS_MAX_FANIN; ++i) d.grads[i] = i < args->num_grads ? args->grads[i] : nullptr;
  for (int i = 0; i < PS_MAX_FANOUT; ++i) d.outs[i] = i < args->num_outs ? args->outs[i] : nullptr;
  d.master = args->master;
  d.m = args->m;
  d.v = args->v;
  d.mc_out = args->out_f32 ? nullptr : args->mc_out;
  d.body_outs = d.mc_out ? args->body_outs : args->num_outs;
  if (d.body_outs < 0 || d.body_outs > args->num_outs) return cudaErrorInvalidValue;
  // both flavours move 16-byte vectors (ld/st.v4, cp.async.bulk) through every one of these pointers
  uintptr_t addr_bits = reinterpret_cast<uintptr_t>(d.master) | reinterpret_cast<uintptr_t>(d.m) |
                        reinterpret_cast<uintptr_t>(d.mc_out);
  if (opt->optimizer == PS_OPT_ADAMW) addr_bits |= reinterpret_cast<uintptr_t>(d.v);
  for (int w = 0; w < d.num_grads; ++w) addr_bits |= reinterpret_cast<uintptr_t>(d.grads[w]);
  for (int k = 0; k < d.num_outs; ++k) addr_bits |= reinterpret_cast<uintptr_t>(d.outs[k]);
  if (addr_bits & 15) return cudaErrorMisalignedAddress;
  // 2 resident CTAs/SM x 148 keeps ~100 KB of loads in flight per SM
  const int grid = GridFor(args->n / 8 + 1, max_ctas, 4);
  const bool f32 = args->out_f32 != 0;
  const bool adam = opt->optimizer == PS_OPT_ADAMW;
  ps_opt_params o = *opt;
  if (adam) {  // the kernel multiplies by the reciprocals
    o.bias_corr1 = 1.f / opt->bias_corr1;
    o.bias_corr2 = 1.f / opt->bias_corr2;
  }
  switch (args->grad_format) {
    case PS_GRAD_BF16:
      adam ? LaunchUpdate<PS_GRAD_BF16, PS_OPT_ADAMW>(d, o, f32, grid, st)
           : LaunchUpdate<PS_GRAD_BF16, PS_OPT_SGD>(d, o, f32, grid, st);
      break;
    case PS_GRAD_FP8BLOCK:
      adam ? LaunchUpdate<PS_GRAD_FP8BLOCK, PS_OPT_ADAMW>(d, o, f32, grid, st)
           : LaunchUpdate<PS_GRAD_FP8BLOCK, PS_OPT_SGD>(d, o, f32, grid, st);
      break;
    case PS_GRAD_F32:
      adam ? LaunchUpdate<PS_GRAD_F32, PS_OPT_ADAMW>(d, o, f32, grid, st)
           : LaunchUpdate<PS_GRAD_F32, PS_OPT_SGD>(d, o, f32, grid, st);
      break;
    case PS_GRAD_MC_BF16:
      if (args->num_grads != 1) return cudaErrorInvalidValue;
      adam ? LaunchUpdate<PS_GRAD_MC_BF16, PS_OPT_ADAMW>(d, o, f32, grid, st)
           : LaunchUpdate<PS_GRAD_MC_BF16, PS_OPT_SGD>(d, o, f32, grid, st);
      break;
    default:
      return cudaErrorInvalidValue;
  }
  ps_kernels_internal::CountLaunch(1);
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ps_launch_sum(float* out, const void* const* grads, int num_grads, int fmt, size_t n,
                             float scale, int accumulate, ps_stream_t stream_) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_);
  if (n == 0) return 0;
  if (num_grads < 1 || num_grads > PS_MAX_FANIN) return cudaErrorInvalidValue;
  UpdateDev d;
  d.n = n;
  d.num_grads = num_grads;
  d.num_outs = 0;
  for (int i = 0; i < PS_MAX_FANIN; ++i) d.grads[i] = i < num_grads ? grads[i] : nullptr;
  for (int i = 0; i < PS_MAX_FANOUT; ++i) d.outs[i] = nullptr;
  d.master = d.m = d.v = nullptr;
  d.mc_out = nullptr;
  d.body_outs = 0;
  const int grid = GridFor(n / 8 + 1, 0, 4);
  if (fmt == PS_GRAD_BF16) k_sum<PS_GRAD_BF16><<<grid, kThreads, 0, st>>>(out, d, scale, accumulate);
  else if (fmt == PS_GRAD_FP8BLOCK)
    k_sum<PS_GRAD_FP8BLOCK><<<grid, kThreads, 0, st>>>(out, d, scale, accumulate);
  else if (fmt == PS_GRAD_F32)
    k_sum<PS_GRAD_F32><<<grid, kThreads, 0, st>>>(out, d, scale, accumulate);
  else if (fmt == PS_GRAD_MC_BF16 && num_grads == 1)
    k_sum<PS_GRAD_MC_BF16><<<grid, kThreads, 0, st>>>(out, d, scale, accumulate);
  else return cudaErrorInvalidValue;
  ps_kernels_internal::CountLaunch(1);
  return static_cast<int>(cudaGetLastError());
}
