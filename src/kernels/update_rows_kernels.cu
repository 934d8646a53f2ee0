/**
 * \file update_rows_kernels.cu
 * \brief K_update for row-sparse shards (embedding tables), sm_100a.
 *
 * A step of an embedding table touches a few of its rows. Each worker pushes only those rows
 * (ids + values, see ps_update_rows_args); this launch updates the union of them and writes
 * the new rows into the destinations, so its cost is bounded by the touched rows, not the table.
 * Two kernels on the caller's stream, no host synchronisation:
 *   k_rows_mark    one thread per pushed id: slot_of[w][id] = position in slot w (the first
 *                  occurrence wins, later ones and ids >= rows are counted as bad), and the
 *                  first slot to touch a row appends it to the union list.
 *   k_rows_update  a grid sized to the GPU, one warp per listed row (count read from device
 *                  memory): gather-sum over w = 0..W-1, optimizer step, store to every output;
 *                  then the warp clears that row's scratch, and the last CTA clears the count,
 *                  so the scratch is clean for the next round without an O(rows) memset.
 * The union's order varies from launch to launch; each row's arithmetic does not (the sum runs
 * in slot order and one warp owns the row), so results are bit-identical across launches.
 * Roofline per touched row: W_r rows of gradient + 24 B/element of state traffic + 2 (or 4) B
 * per element and destination.
 */
#include <cuda_runtime.h>

#include <cstdint>

#include "kernels/ps_kernels.h"
#include "kernels/update_math.cuh"

namespace ps_kernels_internal {
void CountLaunch(int n);
int NumSMs();
}

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

struct RowsDev {
  size_t rows;
  int dim;
  int num_grads;
  const uint32_t* ids[PS_MAX_FANIN];
  const unsigned char* vals[PS_MAX_FANIN];  // first value byte of slot w
  uint32_t num_rows[PS_MAX_FANIN];
  uint32_t first_entry[PS_MAX_FANIN + 1];   // prefix sums of num_rows
  float* master;
  float* m;
  float* v;
  int num_outs;
  void* outs[PS_MAX_FANOUT];
  ps_rows_scratch_hdr* hdr;
  uint32_t* touched;
  uint32_t* list;
  uint32_t* slot_of;  // [W][rows]: ~position (0 = absent), so the zero-filled scratch is empty
};

__global__ void __launch_bounds__(kThreads) k_rows_mark(const RowsDev a) {
  const uint32_t total = a.first_entry[a.num_grads];
  for (uint32_t t = blockIdx.x * kThreads + threadIdx.x; t < total; t += gridDim.x * kThreads) {
    int w = 0;
    while (t >= a.first_entry[w + 1]) ++w;
    const uint32_t i = t - a.first_entry[w];
    const uint32_t id = a.ids[w][i];
    if (id >= a.rows) {
      atomicAdd(&a.hdr->bad, 1ull);
      continue;
    }
    // atomicMax of ~i keeps the smallest position: a duplicate resolves the same way every launch
    if (atomicMax(&a.slot_of[static_cast<size_t>(w) * a.rows + id], ~i) != 0u) atomicAdd(&a.hdr->bad, 1ull);
    if (atomicExch(&a.touched[id], 1u) == 0u) a.list[atomicAdd(&a.hdr->count, 1u)] = id;
  }
}

/*! \brief sum over the slots that hold this row of 8 elements starting at column c */
template <int FMT>
__device__ __forceinline__ void gather_row(const RowsDev& a, const int* pos, size_t c, float* g) {
#pragma unroll
  for (int j = 0; j < 8; ++j) g[j] = 0.f;
  // unrolled so that pos[] stays in registers
#pragma unroll
  for (int w = 0; w < PS_MAX_FANIN; ++w) {
    if (w >= a.num_grads || pos[w] < 0) continue;
    const size_t e = static_cast<size_t>(pos[w]) * a.dim + c;  // element index in slot w's value block
    const unsigned char* base = a.vals[w];
    if (FMT == PS_GRAD_BF16) {
      const int4 q = ldg16(base + e * 2);
      float2 f;
      f = bf2(q.x); g[0] += f.x; g[1] += f.y;
      f = bf2(q.y); g[2] += f.x; g[3] += f.y;
      f = bf2(q.z); g[4] += f.x; g[5] += f.y;
      f = bf2(q.w); g[6] += f.x; g[7] += f.y;
    } else if (FMT == PS_GRAD_FP8BLOCK) {
      const uint2 q = ldg8(base + e);
      const float s = e8m0(base[static_cast<size_t>(a.num_rows[w]) * a.dim + (e >> 5)]);
      float t[8];
      fp8x4_to_f32(q.x, s, t);
      fp8x4_to_f32(q.y, s, t + 4);
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] += t[j];
    } else {
      const int4 q0 = ldg16(base + e * 4), q1 = ldg16(base + e * 4 + 16);
      g[0] += __int_as_float(q0.x); g[1] += __int_as_float(q0.y);
      g[2] += __int_as_float(q0.z); g[3] += __int_as_float(q0.w);
      g[4] += __int_as_float(q1.x); g[5] += __int_as_float(q1.y);
      g[6] += __int_as_float(q1.z); g[7] += __int_as_float(q1.w);
    }
  }
}

template <int FMT, int OPT, bool OUT_F32>
__global__ void __launch_bounds__(kThreads) k_rows_update(const RowsDev a, const ps_opt_params o) {
  const int lane = threadIdx.x & 31;
  const uint32_t count = *reinterpret_cast<volatile uint32_t*>(&a.hdr->count);
  const uint32_t warps = gridDim.x * kWarps;
  for (uint32_t r = blockIdx.x * kWarps + (threadIdx.x >> 5); r < count; r += warps) {
    const uint32_t id = a.list[r];
    // lane w looks up the row's position in slot w; every lane gets all W of them
    int my = -1;
    if (lane < a.num_grads) {
      const uint32_t s = a.slot_of[static_cast<size_t>(lane) * a.rows + id];
      my = s ? static_cast<int>(~s) : -1;
    }
    int pos[PS_MAX_FANIN];
#pragma unroll
    for (int w = 0; w < PS_MAX_FANIN; ++w) pos[w] = __shfl_sync(0xffffffffu, my, w);
    const size_t row0 = static_cast<size_t>(id) * a.dim;
#pragma unroll 1
    for (size_t c = static_cast<size_t>(lane) * 8; c < static_cast<size_t>(a.dim); c += 32 * 8) {
      const size_t e = row0 + c;
      float4 p0 = ldf4(a.master + e), p1 = ldf4(a.master + e + 4);
      float4 m0 = ldf4(a.m + e), m1 = ldf4(a.m + e + 4);
      float4 v0 = make_float4(0, 0, 0, 0), v1 = v0;
      if (OPT == PS_OPT_ADAMW) {
        v0 = ldf4(a.v + e);
        v1 = ldf4(a.v + e + 4);
      }
      float g[8];
      gather_row<FMT>(a, pos, c, g);
#pragma unroll
      for (int j = 0; j < 8; ++j) g[j] *= o.grad_scale;
      step<OPT>(p0.x, m0.x, v0.x, g[0], o); step<OPT>(p0.y, m0.y, v0.y, g[1], o);
      step<OPT>(p0.z, m0.z, v0.z, g[2], o); step<OPT>(p0.w, m0.w, v0.w, g[3], o);
      step<OPT>(p1.x, m1.x, v1.x, g[4], o); step<OPT>(p1.y, m1.y, v1.y, g[5], o);
      step<OPT>(p1.z, m1.z, v1.z, g[6], o); step<OPT>(p1.w, m1.w, v1.w, g[7], o);
      stf4(a.master + e, p0); stf4(a.master + e + 4, p1);
      stf4(a.m + e, m0); stf4(a.m + e + 4, m1);
      if (OPT == PS_OPT_ADAMW) {
        stf4(a.v + e, v0);
        stf4(a.v + e + 4, v1);
      }
      if (OUT_F32) {
#pragma unroll 1
        for (int k = 0; k < a.num_outs; ++k) {
          stf4(static_cast<float*>(a.outs[k]) + e, p0);
          stf4(static_cast<float*>(a.outs[k]) + e + 4, p1);
        }
      } else {
        int4 out;
        out.x = pk(p0.x, p0.y); out.y = pk(p0.z, p0.w);
        out.z = pk(p1.x, p1.y); out.w = pk(p1.z, p1.w);
#pragma unroll 1
        for (int k = 0; k < a.num_outs; ++k) st16(static_cast<char*>(a.outs[k]) + e * 2, out);
      }
    }
    // every lane has read slot_of above (the shuffles): clear this row's scratch for the next round
    if (lane < a.num_grads) a.slot_of[static_cast<size_t>(lane) * a.rows + id] = 0u;
    if (lane == 0) a.touched[id] = 0u;
  }
  // each CTA read `count` before it arrives here: the last one to arrive may clear it
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&a.hdr->done, 1u) == gridDim.x - 1) {
      a.hdr->count = 0u;
      a.hdr->done = 0u;
    }
  }
}

template <int FMT, int OPT>
void LaunchRows(const RowsDev& d, const ps_opt_params& o, bool out_f32, int grid, cudaStream_t st) {
  if (out_f32) k_rows_update<FMT, OPT, true><<<grid, kThreads, 0, st>>>(d, o);
  else k_rows_update<FMT, OPT, false><<<grid, kThreads, 0, st>>>(d, o);
}

}  // namespace

extern "C" int ps_launch_update_rows(const ps_update_rows_args* args, const ps_opt_params* opt,
                                     int max_ctas, ps_stream_t stream_) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_);
  if (args->num_grads < 1 || args->num_grads > PS_MAX_FANIN) return cudaErrorInvalidValue;
  if (args->num_outs < 0 || args->num_outs > PS_MAX_FANOUT) return cudaErrorInvalidValue;
  if (args->dim <= 0 || args->dim % 8 != 0) return cudaErrorInvalidValue;
  if (args->grad_format == PS_GRAD_FP8BLOCK && args->dim % 32 != 0) return cudaErrorInvalidValue;
  if (args->grad_format != PS_GRAD_F32 && args->grad_format != PS_GRAD_BF16 &&
      args->grad_format != PS_GRAD_FP8BLOCK)
    return cudaErrorInvalidValue;
  if (args->rows > 0xffffffffull) return cudaErrorInvalidValue;  // ids are u32
  RowsDev d;
  d.rows = args->rows;
  d.dim = args->dim;
  d.num_grads = args->num_grads;
  d.first_entry[0] = 0;
  uintptr_t addr_bits = reinterpret_cast<uintptr_t>(args->master) | reinterpret_cast<uintptr_t>(args->m) |
                        reinterpret_cast<uintptr_t>(args->scratch);
  if (opt->optimizer == PS_OPT_ADAMW) addr_bits |= reinterpret_cast<uintptr_t>(args->v);
  uint64_t total = 0;
  for (int w = 0; w < PS_MAX_FANIN; ++w) {
    const bool used = w < args->num_grads;
    const uint32_t r = used ? args->num_rows[w] : 0u;
    const unsigned char* slot = used ? static_cast<const unsigned char*>(args->grads[w]) : nullptr;
    if (used) addr_bits |= reinterpret_cast<uintptr_t>(slot);
    d.ids[w] = reinterpret_cast<const uint32_t*>(slot);
    d.vals[w] = slot ? slot + (static_cast<size_t>(r) + 3) / 4 * 16 : nullptr;
    d.num_rows[w] = r;
    total += r;
    if (total > 0xffffffffull) return cudaErrorInvalidValue;
    d.first_entry[w + 1] = static_cast<uint32_t>(total);
  }
  d.master = args->master;
  d.m = args->m;
  d.v = args->v;
  d.num_outs = args->num_outs;
  for (int k = 0; k < PS_MAX_FANOUT; ++k) {
    d.outs[k] = k < args->num_outs ? args->outs[k] : nullptr;
    if (k < args->num_outs) addr_bits |= reinterpret_cast<uintptr_t>(d.outs[k]);
  }
  // rows move as 16-byte vectors through every one of these pointers
  if (addr_bits & 15) return cudaErrorMisalignedAddress;
  if (total == 0) return 0;  // nobody touched a row: nothing to mark, step or store
  d.hdr = static_cast<ps_rows_scratch_hdr*>(args->scratch);
  d.touched = reinterpret_cast<uint32_t*>(d.hdr + 1);
  d.list = d.touched + args->rows;
  d.slot_of = d.list + args->rows;

  const int num_sms = ps_kernels_internal::NumSMs();
  int mark_grid = static_cast<int>((total + kThreads - 1) / kThreads);
  if (mark_grid > num_sms * 8) mark_grid = num_sms * 8;
  k_rows_mark<<<mark_grid, kThreads, 0, st>>>(d);
  // the union is at most min(total, rows) rows: no more warps than that are useful
  const uint64_t max_rows = total < args->rows ? total : args->rows;
  uint64_t want = (max_rows + kWarps - 1) / kWarps;
  const uint64_t cap = max_ctas > 0 ? static_cast<uint64_t>(max_ctas) : static_cast<uint64_t>(num_sms) * 4;
  if (want > cap) want = cap;
  const int grid = want < 1 ? 1 : static_cast<int>(want);
  const bool f32 = args->out_f32 != 0;
  const bool adam = opt->optimizer == PS_OPT_ADAMW;
  ps_opt_params o = *opt;
  if (adam) {  // the kernel multiplies by the reciprocals
    o.bias_corr1 = 1.f / opt->bias_corr1;
    o.bias_corr2 = 1.f / opt->bias_corr2;
  }
  switch (args->grad_format) {
    case PS_GRAD_BF16:
      adam ? LaunchRows<PS_GRAD_BF16, PS_OPT_ADAMW>(d, o, f32, grid, st)
           : LaunchRows<PS_GRAD_BF16, PS_OPT_SGD>(d, o, f32, grid, st);
      break;
    case PS_GRAD_FP8BLOCK:
      adam ? LaunchRows<PS_GRAD_FP8BLOCK, PS_OPT_ADAMW>(d, o, f32, grid, st)
           : LaunchRows<PS_GRAD_FP8BLOCK, PS_OPT_SGD>(d, o, f32, grid, st);
      break;
    default:
      adam ? LaunchRows<PS_GRAD_F32, PS_OPT_ADAMW>(d, o, f32, grid, st)
           : LaunchRows<PS_GRAD_F32, PS_OPT_SGD>(d, o, f32, grid, st);
      break;
  }
  ps_kernels_internal::CountLaunch(2);
  return static_cast<int>(cudaGetLastError());
}
