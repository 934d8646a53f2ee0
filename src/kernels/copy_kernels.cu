/**
 * \file copy_kernels.cu
 * \brief K_push / K_pull: the NVLink van's data movers (sm_100a).
 *
 * What the reference does with NIC DMA (RDMA WRITE, src/rdma_transport.h:323-357)
 * or a CPU memcpy pool (IPCTransport, :524-589) is here a kernel whose *stores*
 * land in peer HBM through the NVLink mapping, fused with the transform the
 * payload needs anyway:
 *   raw        : 16-byte vector copy, 4 independent LDG.128 in flight per thread
 *                (streaming: ld.global.nc.L1::no_allocate, st.global.L1::no_allocate)
 *   raw (TMA)  : PS_COPY_TMA=1 — one elected thread per CTA drives a multi-stage
 *                cp.async.bulk global->smem->global pipeline (UBLKCP), no
 *                register staging, mbarrier complete_tx tracking
 *   f32->bf16  : gradient scale (1/W) + cast fused into the push
 *   ->fp8 block: e4m3 payload + one e8m0 exponent per 32 elements (amax via
 *                quad shuffles), halving NVLink bytes vs bf16
 * All kernels are grid-stride persistent: grid = min(work, 148 SMs x resident CTAs).
 */
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdlib>

#include "kernels/ps_kernels.h"

namespace {

std::atomic<unsigned long long> g_launches{0};

constexpr int kThreads = 256;

constexpr int kMaxDevices = 16;

/*! \brief index of the current device for per-device caches, in [0, kMaxDevices) */
int CurrentDevice() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev < 0 || dev >= kMaxDevices ? 0 : dev;
}

/*! \brief SM count of the current device (148 on B200), asked once per device */
int NumSMs() {
  static std::atomic<int> cached[kMaxDevices] = {};
  const int dev = CurrentDevice();
  int n = cached[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

__device__ __forceinline__ int4 ld_stream(const int4* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(int4* p, const int4& v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}
__device__ __forceinline__ void st_stream8(uint2* p, const uint2& v) {
  asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y)
               : "memory");
}

// ---------------------------------------------------------------------------
// in-kernel completion signal (ps_signal): every CTA fences its stores at system scope and
// counts itself in; the last one publishes the value with st.release.sys. No cudaEvent, no
// host thread between the copy and the receiver that polls the flag.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
/*! \brief called by ONE thread of a CTA after all of that CTA's stores are ordered before it */
__device__ __forceinline__ void signal_arrive(const ps_signal& sig) {
  __threadfence_system();
  const unsigned total = gridDim.x * gridDim.y * gridDim.z;
  if (atomicAdd(sig.counter, 1u) == total - 1) {
    *sig.counter = 0;        // the next kernel on this stream starts from zero again
    __threadfence_system();  // acquire side of the counter: all CTAs' stores are ordered before the flag
    st_release_sys(sig.flag, sig.value);
  }
}
/*! \brief tail of a kernel whose CTAs all reach this point with all their threads */
__device__ __forceinline__ void signal_tail(const ps_signal& sig) {
  if (sig.flag == nullptr) return;
  __syncthreads();
  if (threadIdx.x == 0) signal_arrive(sig);
}

__global__ void k_signal(const ps_signal sig) {
  __threadfence_system();
  st_release_sys(sig.flag, sig.value);
}

// ---------------------------------------------------------------------------
// raw copy, LDG/STG flavour
// ---------------------------------------------------------------------------
template <int UNROLL>
__global__ void __launch_bounds__(kThreads)
k_copy_vec16(int4* __restrict__ dst, const int4* __restrict__ src, size_t n16, const ps_signal sig) {
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  size_t i = static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x;
  // UNROLL independent 16-byte loads are issued before the first store
  for (; i + (UNROLL - 1) * stride < n16; i += UNROLL * stride) {
    int4 v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) v[u] = ld_stream(src + i + u * stride);
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) st_stream(dst + i + u * stride, v[u]);
  }
  for (; i < n16; i += stride) st_stream(dst + i, ld_stream(src + i));
  signal_tail(sig);
}

// ---------------------------------------------------------------------------
// K_pull through the switch: the destination is a MULTICAST address bound to the same offset
// of every worker's buffer — each 16-byte vector leaves this GPU once (multimem.st) and the
// NVSwitch replicates it into all of them (NVLS). The source is read once, the server's
// egress is 1x the payload instead of W x. The reference's IPC pull copies into one shared
// segment per peer (src/rdma_transport.h:524-589).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void multimem_st16(void* p, const int4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
               "r"(v.z), "r"(v.w)
               : "memory");
}
template <int UNROLL>
__global__ void __launch_bounds__(kThreads)
k_copy_mc16(int4* __restrict__ mc_dst, const int4* __restrict__ src, size_t n16, const ps_signal sig) {
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  size_t i = static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x;
  for (; i + (UNROLL - 1) * stride < n16; i += UNROLL * stride) {
    int4 v[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) v[u] = ld_stream(src + i + u * stride);
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) multimem_st16(mc_dst + i + u * stride, v[u]);
  }
  for (; i < n16; i += stride) multimem_st16(mc_dst + i, ld_stream(src + i));
  signal_tail(sig);
}

__global__ void k_copy_bytes(unsigned char* __restrict__ dst, const unsigned char* __restrict__ src,
                             size_t n, const ps_signal sig) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = src[i];
  signal_tail(sig);
}

// ---------------------------------------------------------------------------
// raw copy of MANY buffers in one launch (launch coalescing): blockIdx.y picks the segment,
// the x-blocks grid-stride over it. A 4 MB message costs ~3 us of copy time but ~3 us of CPU
// per launch + event; a round of 40 pushes becomes 2 launches and ONE event.
// ---------------------------------------------------------------------------
struct MultiSegs {
  unsigned char* dst[PS_MAX_COPY_SEGS];
  const unsigned char* src[PS_MAX_COPY_SEGS];
  size_t bytes[PS_MAX_COPY_SEGS];
};

__global__ void __launch_bounds__(kThreads) k_copy_multi(const MultiSegs segs) {
  const int sgi = blockIdx.y;
  unsigned char* __restrict__ dst = segs.dst[sgi];
  const unsigned char* __restrict__ src = segs.src[sgi];
  const size_t n = segs.bytes[sgi];
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  const size_t tid = static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x;
  const bool aligned = ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15) == 0;
  size_t done = 0;
  if (aligned) {
    const size_t n16 = n / 16;
    int4* d4 = reinterpret_cast<int4*>(dst);
    const int4* s4 = reinterpret_cast<const int4*>(src);
    size_t i = tid;
    for (; i + 3 * stride < n16; i += 4 * stride) {
      int4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ld_stream(s4 + i + u * stride);
#pragma unroll
      for (int u = 0; u < 4; ++u) st_stream(d4 + i + u * stride, v[u]);
    }
    for (; i < n16; i += stride) st_stream(d4 + i, ld_stream(s4 + i));
    done = n16 * 16;
  }
  for (size_t i = done + tid; i < n; i += stride) dst[i] = src[i];  // tail / unaligned segment
}

// ---------------------------------------------------------------------------
// raw copy, TMA bulk flavour: global -> smem -> global, driven by one thread
// ---------------------------------------------------------------------------
constexpr int kTmaStages = 4;
constexpr int kTmaChunk = 32 * 1024;  // bytes per stage; 4 x 32 KB = 128 KB smem / CTA

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t}" ::"r"(smem_u32(bar)),
      "r"(phase)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes,
                                         uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem_dst)),
      "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}

__global__ void __launch_bounds__(32)
k_copy_tma(unsigned char* __restrict__ dst, const unsigned char* __restrict__ src,
           size_t n_chunks, size_t n_bytes, const ps_signal sig) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t full[kTmaStages];
  if (threadIdx.x == 0) {
    for (int s = 0; s < kTmaStages; ++s) mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  if (threadIdx.x != 0) return;
  // chunks owned by this CTA: blockIdx.x, blockIdx.x + grid, ...
  const size_t first = blockIdx.x, step = gridDim.x;
  const size_t mine = first < n_chunks ? (n_chunks - first + step - 1) / step : 0;
  auto chunk_bytes = [&](size_t k) -> uint32_t {
    const size_t off = (first + k * step) * static_cast<size_t>(kTmaChunk);
    const size_t left = n_bytes - off;
    return static_cast<uint32_t>(left < static_cast<size_t>(kTmaChunk) ? left : kTmaChunk);
  };
  // software pipeline: loads run kLook chunks ahead of stores. Stage reuse at step k
  // needs the store of chunk k-S (issued at step k-S+kLook = k-2) to have drained
  // its smem reads; one younger store (chunk k-S+1) may still be reading.
  constexpr int kLook = kTmaStages - 2;
  for (size_t k = 0; k < mine + kLook; ++k) {
    if (k < mine) {
      const int s = static_cast<int>(k % kTmaStages);
      if (k >= static_cast<size_t>(kTmaStages)) {
        asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      }
      const uint32_t b = chunk_bytes(k);
      mbar_expect_tx(&full[s], b);
      bulk_g2s(smem + static_cast<size_t>(s) * kTmaChunk,
               src + (first + k * step) * static_cast<size_t>(kTmaChunk), b, &full[s]);
    }
    if (k >= static_cast<size_t>(kLook)) {
      const size_t j = k - kLook;
      const int s = static_cast<int>(j % kTmaStages);
      mbar_wait(&full[s], static_cast<uint32_t>((j / kTmaStages) & 1));
      bulk_s2g(dst + (first + j * step) * static_cast<size_t>(kTmaChunk),
               smem + static_cast<size_t>(s) * kTmaChunk, chunk_bytes(j));
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  }
  // all stores complete (not just smem reads) before the kernel retires
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  // the bulk stores went through the async proxy: order them before the generic-proxy flag store
  asm volatile("fence.proxy.async;" ::: "memory");
  if (sig.flag != nullptr) signal_arrive(sig);
}

// ---------------------------------------------------------------------------
// scale + cast to bf16
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 t = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(t);
}

/*! 8 fp32 in (2 x LDG.128) -> 8 bf16 out (1 x STG.128) per thread-iteration */
__global__ void __launch_bounds__(kThreads)
k_f32_to_bf16(int4* __restrict__ dst, const int4* __restrict__ src, size_t n8, float scale,
              const ps_signal sig) {
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  for (size_t i = static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x; i < n8; i += stride) {
    const int4 a = ld_stream(src + 2 * i), b = ld_stream(src + 2 * i + 1);
    int4 o;
    o.x = pack_bf16x2(__int_as_float(a.x) * scale, __int_as_float(a.y) * scale);
    o.y = pack_bf16x2(__int_as_float(a.z) * scale, __int_as_float(a.w) * scale);
    o.z = pack_bf16x2(__int_as_float(b.x) * scale, __int_as_float(b.y) * scale);
    o.w = pack_bf16x2(__int_as_float(b.z) * scale, __int_as_float(b.w) * scale);
    st_stream(dst + i, o);
  }
  signal_tail(sig);
}
__global__ void k_f32_to_bf16_tail(__nv_bfloat16* dst, const float* src, size_t from, size_t n,
                                   float scale, const ps_signal sig) {
  size_t i = from + blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __float2bfloat16_rn(src[i] * scale);
  signal_tail(sig);
}

__global__ void __launch_bounds__(kThreads)
k_bf16_scale(int4* __restrict__ dst, const int4* __restrict__ src, size_t n8, float scale,
             const ps_signal sig) {
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  for (size_t i = static_cast<size_t>(blockIdx.x) * kThreads + threadIdx.x; i < n8; i += stride) {
    const int4 a = ld_stream(src + i);
    int4 o;
    float2 f;
    f = unpack_bf16x2(a.x); o.x = pack_bf16x2(f.x * scale, f.y * scale);
    f = unpack_bf16x2(a.y); o.y = pack_bf16x2(f.x * scale, f.y * scale);
    f = unpack_bf16x2(a.z); o.z = pack_bf16x2(f.x * scale, f.y * scale);
    f = unpack_bf16x2(a.w); o.w = pack_bf16x2(f.x * scale, f.y * scale);
    st_stream(dst + i, o);
  }
  signal_tail(sig);
}
__global__ void k_bf16_scale_tail(__nv_bfloat16* dst, const __nv_bfloat16* src, size_t from,
                                  size_t n, float scale, const ps_signal sig) {
  size_t i = from + blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __float2bfloat16_rn(__bfloat162float(src[i]) * scale);
  signal_tail(sig);
}

// ---------------------------------------------------------------------------
// block-scaled fp8 (e4m3 payload, one e8m0 exponent per 32 elements)
// ---------------------------------------------------------------------------
/*!
 * exponent e such that amax / 2^e <= 448 (largest finite e4m3); biased by 127. e is clamped to
 * [-126, 127]: the decoders read byte 0 as 2^-126 (the smallest normal fp32 scale), so byte 0 is
 * left to the all-zero block, where any scale decodes to zero.
 */
__device__ __forceinline__ uint32_t e8m0_for_amax(float amax) {
  if (!(amax > 0.f)) return 0u;
  const uint32_t bits = __float_as_uint(amax);
  int k = static_cast<int>((bits >> 23) & 0xff) - 127;     // amax = m * 2^k, m in [1,2)
  const uint32_t mant = bits & 0x7fffffu;
  int e = k - 8 + (mant > 0x600000u ? 1 : 0);              // 448 = 1.75 * 2^8
  e = max(-126, min(127, e));
  return static_cast<uint32_t>(e + 127);
}
__device__ __forceinline__ float exp2_from_e8m0_neg(uint32_t biased) {
  // 2^-(biased-127) built directly in the exponent field
  const int e = 127 - static_cast<int>(biased);
  const int be = max(1, min(254, e + 127));
  return __uint_as_float(static_cast<uint32_t>(be) << 23);
}
__device__ __forceinline__ float exp2_from_e8m0(uint32_t biased) {
  const int be = max(1, min(254, static_cast<int>(biased)));
  return __uint_as_float(static_cast<uint32_t>(be) << 23);
}
__device__ __forceinline__ uint32_t quant4(float a, float b, float c, float d) {
  const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
  const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
  return (lo & 0xffffu) | (hi << 16);
}

/*!
 * Thread t handles elements [8t, 8t+8); four neighbouring lanes form one 32-element
 * block and agree on amax with two xor-shuffles. `n` is the true element count;
 * reads beyond it are treated as zero, the wire buffer is padded to 32.
 */
template <bool SRC_BF16>
__global__ void __launch_bounds__(kThreads)
k_quant_fp8_block(unsigned char* __restrict__ payload, unsigned char* __restrict__ scales,
                  const void* __restrict__ src, size_t n, float scale, const ps_signal sig) {
  const size_t n8 = (n + 31) / 32 * 4;  // thread-iterations, padded to whole blocks
  const size_t stride = static_cast<size_t>(gridDim.x) * kThreads;
  // n8 is a multiple of 4 and every loop bound below a multiple of 32, so the four lanes of a
  // block stay together; the trip count is made WARP-uniform on top of that (a lane past the end
  // idles through the shuffles): the full-mask shuffles and the __syncthreads of the signal tail
  // must be reached by whole warps
  for (size_t base = static_cast<size_t>(blockIdx.x) * kThreads + (threadIdx.x & ~31u); base < n8;
       base += stride) {
    const size_t i = base + (threadIdx.x & 31u);
    const bool live = i < n8;
    float x[8];
    const size_t e0 = i * 8;
    if (live && e0 + 8 <= n) {
      if (SRC_BF16) {
        const int4 a = ld_stream(reinterpret_cast<const int4*>(src) + i);
        float2 f;
        f = unpack_bf16x2(a.x); x[0] = f.x; x[1] = f.y;
        f = unpack_bf16x2(a.y); x[2] = f.x; x[3] = f.y;
        f = unpack_bf16x2(a.z); x[4] = f.x; x[5] = f.y;
        f = unpack_bf16x2(a.w); x[6] = f.x; x[7] = f.y;
      } else {
        const int4 a = ld_stream(reinterpret_cast<const int4*>(src) + 2 * i);
        const int4 b = ld_stream(reinterpret_cast<const int4*>(src) + 2 * i + 1);
        x[0] = __int_as_float(a.x); x[1] = __int_as_float(a.y);
        x[2] = __int_as_float(a.z); x[3] = __int_as_float(a.w);
        x[4] = __int_as_float(b.x); x[5] = __int_as_float(b.y);
        x[6] = __int_as_float(b.z); x[7] = __int_as_float(b.w);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const size_t e = e0 + j;
        float v = 0.f;
        if (live && e < n) {
          v = SRC_BF16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src)[e])
                       : reinterpret_cast<const float*>(src)[e];
        }
        x[j] = v;
      }
    }
    float amax = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      x[j] *= scale;
      amax = fmaxf(amax, fabsf(x[j]));
    }
    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 1));
    amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, 2));
    const uint32_t eb = e8m0_for_amax(amax);
    const float inv = exp2_from_e8m0_neg(eb);
    uint2 q;
    q.x = quant4(x[0] * inv, x[1] * inv, x[2] * inv, x[3] * inv);
    q.y = quant4(x[4] * inv, x[5] * inv, x[6] * inv, x[7] * inv);
    if (live) {
      st_stream8(reinterpret_cast<uint2*>(payload) + i, q);
      if ((threadIdx.x & 3) == 0) scales[i >> 2] = static_cast<unsigned char>(eb);
    }
  }
  signal_tail(sig);
}

// ---------------------------------------------------------------------------
// decode (wire -> fp32), used by tests / unpack
// ---------------------------------------------------------------------------
__global__ void k_decode_bf16(float* dst, const __nv_bfloat16* src, size_t n) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = __bfloat162float(src[i]);
}
__global__ void k_decode_fp8_block(float* dst, const unsigned char* payload,
                                   const unsigned char* scales, size_t n) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) {
    const __half_raw h = __nv_cvt_fp8_to_halfraw(payload[i], __NV_E4M3);
    dst[i] = __half2float(__half(h)) * exp2_from_e8m0(scales[i >> 5]);
  }
}

// ---------------------------------------------------------------------------
// stress-test helpers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
__global__ void k_fill_u32(uint32_t* dst, size_t n, uint32_t seed) {
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = mix32(static_cast<uint32_t>(i) ^ seed);
}
__global__ void k_checksum_u32(const uint32_t* src, size_t n, unsigned long long* out) {
  unsigned long long acc = 0;
  const size_t stride = static_cast<size_t>(gridDim.x) * blockDim.x;
  for (size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride)
    acc += src[i];
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, acc);
}

int GridFor(size_t work_items, int max_ctas, int resident_per_sm) {
  size_t want = (work_items + kThreads - 1) / kThreads;
  size_t cap = max_ctas > 0 ? static_cast<size_t>(max_ctas)
                            : static_cast<size_t>(NumSMs()) * resident_per_sm;
  if (want > cap) want = cap;
  return want < 1 ? 1 : static_cast<int>(want);
}

bool UseTma() {
  static int v = [] {
    const char* e = getenv("PS_COPY_TMA");
    return e ? atoi(e) : 0;
  }();
  return v != 0;
}

}  // namespace

extern "C" unsigned long long ps_kernel_launch_count(void) { return g_launches.load(); }

namespace ps_kernels_internal {
void CountLaunch(int n) { g_launches += static_cast<unsigned long long>(n); }
int NumSMs() { return ::NumSMs(); }
int CurrentDevice() { return ::CurrentDevice(); }
}

extern "C" int ps_launch_signal(const ps_signal* sig, ps_stream_t stream_) {
  if (!sig || !sig->flag) return 0;
  k_signal<<<1, 1, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(*sig);
  ++g_launches;
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ps_launch_copy(void* dst, const void* src, size_t n, int codec, float scale,
                              int max_ctas, ps_stream_t stream_) {
  return ps_launch_copy_signal(dst, src, n, codec, scale, max_ctas, nullptr, stream_);
}

extern "C" int ps_launch_copy_signal(void* dst, const void* src, size_t n, int codec, float scale,
                                     int max_ctas, const ps_signal* sig_, ps_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const ps_signal none = {nullptr, nullptr, 0};
  const ps_signal sig = (sig_ && sig_->flag) ? *sig_ : none;
  if (n == 0) return ps_launch_signal(&sig, stream_);
  // a transfer made of a body and a tail kernel signals from the one launched last
  // (stream order: the body has completed before the tail starts)
  auto sig_if = [&](bool last) -> const ps_signal& { return last ? sig : none; };
  const uintptr_t d = reinterpret_cast<uintptr_t>(dst), s = reinterpret_cast<uintptr_t>(src);
  switch (codec) {
    case PS_CODEC_RAW: {
      if (((d | s) & 15) != 0) {
        k_copy_bytes<<<GridFor(n, max_ctas, 8), kThreads, 0, stream>>>(
            static_cast<unsigned char*>(dst), static_cast<const unsigned char*>(src), n, sig);
        ++g_launches;
        break;
      }
      if (UseTma() && n >= static_cast<size_t>(kTmaChunk)) {
        static std::atomic<bool> attr_set[kMaxDevices] = {};  // the attribute is per device
        const int smem_bytes = kTmaStages * kTmaChunk;
        const int dev = CurrentDevice();
        if (!attr_set[dev].load(std::memory_order_acquire)) {
          cudaFuncSetAttribute(k_copy_tma, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
          attr_set[dev].store(true, std::memory_order_release);
        }
        const size_t body = n & ~size_t(15);
        const size_t chunks = (body + kTmaChunk - 1) / kTmaChunk;
        int grid = static_cast<int>(chunks < static_cast<size_t>(NumSMs()) ? chunks : NumSMs());
        if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
        k_copy_tma<<<grid, 32, smem_bytes, stream>>>(static_cast<unsigned char*>(dst),
                                                      static_cast<const unsigned char*>(src),
                                                      chunks, body, sig_if(n == body));
        ++g_launches;
        if (n > body) {
          k_copy_bytes<<<1, 32, 0, stream>>>(static_cast<unsigned char*>(dst) + body,
                                             static_cast<const unsigned char*>(src) + body,
                                             n - body, sig);
          ++g_launches;
        }
        break;
      }
      const size_t n16 = n / 16;
      if (n16) {
        k_copy_vec16<4><<<GridFor((n16 + 3) / 4, max_ctas, 8), kThreads, 0, stream>>>(
            static_cast<int4*>(dst), static_cast<const int4*>(src), n16, sig_if((n & 15) == 0));
        ++g_launches;
      }
      if (n & 15) {
        k_copy_bytes<<<1, 32, 0, stream>>>(static_cast<unsigned char*>(dst) + n16 * 16,
                                           static_cast<const unsigned char*>(src) + n16 * 16,
                                           n & 15, sig);
        ++g_launches;
      }
      break;
    }
    case PS_CODEC_F32_TO_BF16: {
      const size_t ne = n / 4, n8 = ((d & 15) || (s & 15)) ? 0 : ne / 8;
      const bool tail = ne > n8 * 8;
      if (n8) {
        k_f32_to_bf16<<<GridFor(n8, max_ctas, 8), kThreads, 0, stream>>>(
            static_cast<int4*>(dst), static_cast<const int4*>(src), n8, scale, sig_if(!tail));
        ++g_launches;
      }
      if (tail) {
        const size_t rest = ne - n8 * 8;
        k_f32_to_bf16_tail<<<static_cast<int>((rest + 255) / 256), 256, 0, stream>>>(
            static_cast<__nv_bfloat16*>(dst), static_cast<const float*>(src), n8 * 8, ne, scale, sig);
        ++g_launches;
      }
      if (!n8 && !tail) return ps_launch_signal(&sig, stream_);
      break;
    }
    case PS_CODEC_BF16_SCALE: {
      const size_t ne = n / 2, n8 = ((d & 15) || (s & 15)) ? 0 : ne / 8;
      const bool tail = ne > n8 * 8;
      if (n8) {
        k_bf16_scale<<<GridFor(n8, max_ctas, 8), kThreads, 0, stream>>>(
            static_cast<int4*>(dst), static_cast<const int4*>(src), n8, scale, sig_if(!tail));
        ++g_launches;
      }
      if (tail) {
        const size_t rest = ne - n8 * 8;
        k_bf16_scale_tail<<<static_cast<int>((rest + 255) / 256), 256, 0, stream>>>(
            static_cast<__nv_bfloat16*>(dst), static_cast<const __nv_bfloat16*>(src), n8 * 8, ne,
            scale, sig);
        ++g_launches;
      }
      if (!n8 && !tail) return ps_launch_signal(&sig, stream_);
      break;
    }
    case PS_CODEC_F32_TO_FP8BLOCK:
    case PS_CODEC_BF16_TO_FP8BLOCK: {
      const bool bf = codec == PS_CODEC_BF16_TO_FP8BLOCK;
      const size_t ne = n / (bf ? 2 : 4);
      const size_t npad = (ne + 31) / 32 * 32;
      unsigned char* payload = static_cast<unsigned char*>(dst);
      unsigned char* scales = payload + npad;
      if ((s & 15) || (d & 7)) return static_cast<int>(cudaErrorMisalignedAddress);
      if (npad == 0) return ps_launch_signal(&sig, stream_);
      const int grid = GridFor(npad / 8, max_ctas, 8);
      if (bf) {
        k_quant_fp8_block<true><<<grid, kThreads, 0, stream>>>(payload, scales, src, ne, scale, sig);
      } else {
        k_quant_fp8_block<false><<<grid, kThreads, 0, stream>>>(payload, scales, src, ne, scale, sig);
      }
      ++g_launches;
      break;
    }
    default:
      return static_cast<int>(cudaErrorInvalidValue);
  }
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ps_launch_copy_multicast(void* mc_dst, const void* src, size_t n, int max_ctas,
                                        const ps_signal* sig_, ps_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  const ps_signal none = {nullptr, nullptr, 0};
  const ps_signal sig = (sig_ && sig_->flag) ? *sig_ : none;
  const uintptr_t d = reinterpret_cast<uintptr_t>(mc_dst), s = reinterpret_cast<uintptr_t>(src);
  // multimem operates on naturally aligned 4 / 8 / 16-byte words: whole vectors only
  if (((d | s) & 15) != 0 || (n & 15) != 0) return static_cast<int>(cudaErrorMisalignedAddress);
  if (n == 0) return ps_launch_signal(&sig, stream_);
  const size_t n16 = n / 16;
  k_copy_mc16<4><<<GridFor((n16 + 3) / 4, max_ctas, 8), kThreads, 0, stream>>>(
      static_cast<int4*>(mc_dst), static_cast<const int4*>(src), n16, sig);
  ++g_launches;
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ps_launch_copy_multi(const ps_copy_seg* segs, int nseg, int max_ctas,
                                    ps_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  int at = 0;
  while (at < nseg) {
    MultiSegs m;
    int cnt = 0;
    size_t longest = 0;
    for (; at < nseg && cnt < PS_MAX_COPY_SEGS; ++at) {
      if (segs[at].bytes == 0) continue;
      m.dst[cnt] = static_cast<unsigned char*>(segs[at].dst);
      m.src[cnt] = static_cast<const unsigned char*>(segs[at].src);
      m.bytes[cnt] = segs[at].bytes;
      longest = longest > segs[at].bytes ? longest : segs[at].bytes;
      ++cnt;
    }
    if (cnt == 0) break;
    for (int i = cnt; i < PS_MAX_COPY_SEGS; ++i) {
      m.dst[i] = nullptr;
      m.src[i] = nullptr;
      m.bytes[i] = 0;
    }
    // enough x-blocks that the longest segment gets 4 x 16 B per thread per pass, but not more
    // than 8 resident CTAs per SM over all segments
    size_t want = (longest / 64 + kThreads - 1) / kThreads;
    size_t cap = static_cast<size_t>(max_ctas > 0 ? max_ctas : NumSMs() * 8) / static_cast<size_t>(cnt);
    if (cap < 1) cap = 1;
    if (want > cap) want = cap;
    if (want < 1) want = 1;
    dim3 grid(static_cast<unsigned>(want), static_cast<unsigned>(cnt));
    k_copy_multi<<<grid, kThreads, 0, stream>>>(m);
    ++g_launches;
  }
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ps_launch_decode(void* dst_f32, const void* wire, size_t n, int fmt,
                                ps_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  if (n == 0) return 0;
  const int grid = GridFor(n, 0, 8);
  if (fmt == PS_GRAD_BF16) {
    k_decode_bf16<<<grid, kThreads, 0, stream>>>(static_cast<float*>(dst_f32),
                                                 static_cast<const __nv_bfloat16*>(wire), n);
  } else if (fmt == PS_GRAD_FP8BLOCK) {
    const size_t npad = (n + 31) / 32 * 32;
    const unsigned char* p = static_cast<const unsigned char*>(wire);
    k_decode_fp8_block<<<grid, kThreads, 0, stream>>>(static_cast<float*>(dst_f32), p, p + npad, n);
  } else {
    return ps_launch_copy(dst_f32, wire, n * 4, PS_CODEC_RAW, 1.f, 0, stream_);
  }
  ++g_launches;
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ps_launch_fill_u32(void* dst, size_t n, uint32_t seed, ps_stream_t stream_) {
  if (n == 0) return 0;
  k_fill_u32<<<GridFor(n, 0, 8), kThreads, 0, reinterpret_cast<cudaStream_t>(stream_)>>>(
      static_cast<uint32_t*>(dst), n, seed);
  ++g_launches;
  return static_cast<int>(cudaGetLastError());
}

extern "C" int ps_launch_checksum_u32(const void* src, size_t n, unsigned long long* out_dev,
                                      ps_stream_t stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  cudaMemsetAsync(out_dev, 0, sizeof(unsigned long long), stream);
  if (n) {
    k_checksum_u32<<<GridFor(n, 0, 4), kThreads, 0, stream>>>(static_cast<const uint32_t*>(src), n,
                                                              out_dev);
    ++g_launches;
  }
  return static_cast<int>(cudaGetLastError());
}
