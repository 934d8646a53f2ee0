/**
 * \file host_kernels.cc
 * \brief CPU twins of the data-plane kernels (see host_kernels.h).
 *
 * Same wire formats and the same rounding decisions as src/kernels/copy_kernels.cu /
 * update_kernels.cu, written as plain loops split over a few threads:
 *   bf16        round-to-nearest-even of the fp32 value (NaN stays NaN)
 *   fp8-block   32 elements share one e8m0 exponent chosen so that amax maps into
 *               [224, 448] of e4m3; values are rounded to nearest-even and saturate at 448
 * The optimizer step uses IEEE sqrt / division where the GPU kernel uses MUFU
 * approximations, so the two agree to a few ulp, not bit for bit.
 */
#include "kernels/host_kernels.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

namespace {

inline uint32_t F2U(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
}
inline float U2F(uint32_t u) {
  float f;
  memcpy(&f, &u, 4);
  return f;
}

inline uint16_t F32ToBf16(float f) {
  uint32_t u = F2U(f);
  if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);  // quiet NaN
  u += 0x7fffu + ((u >> 16) & 1u);
  return static_cast<uint16_t>(u >> 16);
}
inline float Bf16ToF32(uint16_t h) { return U2F(static_cast<uint32_t>(h) << 16); }

/*! \brief e4m3 (bias 7, no infinities, 0x7f = NaN) -> fp32, by table */
const float* E4m3Table() {
  static float table[256];
  static bool ready = [] {
    for (int b = 0; b < 256; ++b) {
      const int sign = b >> 7, exp = (b >> 3) & 0xf, man = b & 7;
      float v;
      if (exp == 0) {
        v = std::ldexp(static_cast<float>(man), -9);  // subnormal: man/8 * 2^-6
      } else if (exp == 15 && man == 7) {
        v = std::nanf("");
      } else {
        v = std::ldexp(1.f + man / 8.f, exp - 7);
      }
      table[b] = sign ? -v : v;
    }
    return true;
  }();
  (void)ready;
  return table;
}

/*! \brief fp32 -> e4m3, round to nearest even, saturating at +-448 (cvt.rn.satfinite) */
inline uint8_t F32ToE4m3(float f) {
  uint32_t u = F2U(f);
  const uint8_t sign = static_cast<uint8_t>((u >> 24) & 0x80);
  u &= 0x7fffffffu;
  if (u > 0x7f800000u) return static_cast<uint8_t>(sign | 0x7f);  // NaN
  const float a = U2F(u);
  if (a < 0.015625f) {
    // below 2^-6 the grid is uniform (step 2^-9): subnormals, and 8 * 2^-9 is the first normal
    return static_cast<uint8_t>(sign | static_cast<uint8_t>(std::lrintf(a * 512.f)));
  }
  // keep 3 mantissa bits: add half of the dropped 20 bits (ties to even), truncate
  u += 0x7ffffu + ((u >> 20) & 1u);
  u &= 0xfff00000u;
  if (u > 0x43e00000u) return static_cast<uint8_t>(sign | 0x7e);  // > 448 (or inf): saturate
  const uint32_t exp = (u >> 23) - 120u;  // biased by 7: 2^-6 -> 1
  return static_cast<uint8_t>(sign | (exp << 3) | ((u >> 20) & 7u));
}

inline uint32_t E8m0ForAmax(float amax) {
  if (!(amax > 0.f)) return 0u;
  const uint32_t bits = F2U(amax);
  const int k = static_cast<int>((bits >> 23) & 0xff) - 127;
  const uint32_t mant = bits & 0x7fffffu;
  int e = k - 8 + (mant > 0x600000u ? 1 : 0);  // 448 = 1.75 * 2^8
  e = std::max(-126, std::min(127, e));         // byte 0 only for the all-zero block (see copy_kernels.cu)
  return static_cast<uint32_t>(e + 127);
}
inline float Exp2FromE8m0(uint32_t biased) {
  const int be = std::max(1, std::min(254, static_cast<int>(biased)));
  return U2F(static_cast<uint32_t>(be) << 23);
}
inline float Exp2FromE8m0Neg(uint32_t biased) {
  const int e = 127 - static_cast<int>(biased);
  const int be = std::max(1, std::min(254, e + 127));
  return U2F(static_cast<uint32_t>(be) << 23);
}

/*! \brief run fn(begin, end) over [0, n) in `grain`-aligned pieces on a few threads */
template <typename Fn>
void ParallelFor(size_t n, size_t grain, Fn fn) {
  const size_t kMinPerThread = 1u << 18;
  size_t threads = std::min<size_t>(8, std::max<unsigned>(1, std::thread::hardware_concurrency()));
  threads = std::min(threads, std::max<size_t>(1, n / kMinPerThread));
  if (threads <= 1) {
    fn(static_cast<size_t>(0), n);
    return;
  }
  size_t chunk = (n + threads - 1) / threads;
  chunk = (chunk + grain - 1) / grain * grain;
  std::vector<std::thread> pool;
  for (size_t a = chunk; a < n; a += chunk) {
    const size_t b = std::min(n, a + chunk);
    pool.emplace_back([=] { fn(a, b); });
  }
  fn(static_cast<size_t>(0), std::min(n, chunk));
  for (auto& t : pool) t.join();
}

template <bool SRC_BF16>
void QuantFp8Block(unsigned char* payload, unsigned char* scales, const void* src, size_t n,
                   float scale) {
  const size_t blocks = (n + 31) / 32;
  ParallelFor(blocks, 1, [=](size_t b0, size_t b1) {
    for (size_t b = b0; b < b1; ++b) {
      float x[32];
      float amax = 0.f;
      for (int j = 0; j < 32; ++j) {
        const size_t e = b * 32 + j;
        float v = 0.f;
        if (e < n) {
          v = SRC_BF16 ? Bf16ToF32(static_cast<const uint16_t*>(src)[e])
                       : static_cast<const float*>(src)[e];
        }
        x[j] = v * scale;
        amax = std::max(amax, std::fabs(x[j]));
      }
      const uint32_t eb = E8m0ForAmax(amax);
      const float inv = Exp2FromE8m0Neg(eb);
      for (int j = 0; j < 32; ++j) payload[b * 32 + j] = F32ToE4m3(x[j] * inv);
      scales[b] = static_cast<unsigned char>(eb);
    }
  });
}

/*! \brief value of element e of a gradient slot in format fmt */
inline float LoadGrad(const void* slot, int fmt, size_t e, size_t npad, const float* e4m3) {
  const unsigned char* base = static_cast<const unsigned char*>(slot);
  switch (fmt) {
    case PS_GRAD_BF16:
      return Bf16ToF32(reinterpret_cast<const uint16_t*>(base)[e]);
    case PS_GRAD_FP8BLOCK:
      return e4m3[base[e]] * Exp2FromE8m0(base[npad + (e >> 5)]);
    default:
      return reinterpret_cast<const float*>(base)[e];
  }
}

}  // namespace

extern "C" int ps_host_copy(void* dst, const void* src, size_t n, int codec, float scale) {
  if (n == 0) return 0;
  switch (codec) {
    case PS_CODEC_RAW: {
      if (dst == src) return 0;
      const char* s8 = static_cast<const char*>(src);
      char* d8 = static_cast<char*>(dst);
      const bool overlap = d8 < s8 + n && s8 < d8 + n;
      if (n < (2u << 20) || overlap) {
        memmove(dst, src, n);
      } else {
        // one core moves ~10 GB/s; large messages (the shm van's push / pull payloads) are split
        ParallelFor(n, 4096, [=](size_t a, size_t b) { memcpy(d8 + a, s8 + a, b - a); });
      }
      return 0;
    }
    case PS_CODEC_F32_TO_BF16: {
      const float* s = static_cast<const float*>(src);
      uint16_t* d = static_cast<uint16_t*>(dst);
      ParallelFor(n / 4, 1, [=](size_t a, size_t b) {
        for (size_t i = a; i < b; ++i) d[i] = F32ToBf16(s[i] * scale);
      });
      return 0;
    }
    case PS_CODEC_BF16_SCALE: {
      const uint16_t* s = static_cast<const uint16_t*>(src);
      uint16_t* d = static_cast<uint16_t*>(dst);
      ParallelFor(n / 2, 1, [=](size_t a, size_t b) {
        for (size_t i = a; i < b; ++i) d[i] = F32ToBf16(Bf16ToF32(s[i]) * scale);
      });
      return 0;
    }
    case PS_CODEC_F32_TO_FP8BLOCK:
    case PS_CODEC_BF16_TO_FP8BLOCK: {
      const bool bf = codec == PS_CODEC_BF16_TO_FP8BLOCK;
      const size_t ne = n / (bf ? 2 : 4);
      const size_t npad = (ne + 31) / 32 * 32;
      unsigned char* payload = static_cast<unsigned char*>(dst);
      if (bf) QuantFp8Block<true>(payload, payload + npad, src, ne, scale);
      else QuantFp8Block<false>(payload, payload + npad, src, ne, scale);
      return 0;
    }
    default:
      return 1;
  }
}

extern "C" int ps_host_decode(float* dst, const void* wire, size_t n, int fmt) {
  if (n == 0) return 0;
  if (fmt != PS_GRAD_BF16 && fmt != PS_GRAD_FP8BLOCK && fmt != PS_GRAD_F32) return 1;
  const size_t npad = (n + 31) / 32 * 32;
  const float* e4m3 = E4m3Table();
  ParallelFor(n, 32, [=](size_t a, size_t b) {
    for (size_t i = a; i < b; ++i) dst[i] = LoadGrad(wire, fmt, i, npad, e4m3);
  });
  return 0;
}

extern "C" int ps_host_sum(float* out, const void* const* grads, int num_grads, int fmt, size_t n,
                           float scale, int accumulate) {
  if (n == 0) return 0;
  if (num_grads < 1 || num_grads > PS_MAX_FANIN) return 1;
  if (fmt != PS_GRAD_BF16 && fmt != PS_GRAD_FP8BLOCK && fmt != PS_GRAD_F32) return 1;
  const size_t npad = (n + 31) / 32 * 32;
  const float* e4m3 = E4m3Table();
  std::vector<const void*> g(grads, grads + num_grads);
  ParallelFor(n, 32, [=, &g](size_t a, size_t b) {
    for (size_t i = a; i < b; ++i) {
      float s = 0.f;
      for (const void* slot : g) s += LoadGrad(slot, fmt, i, npad, e4m3);
      out[i] = (accumulate ? out[i] : 0.f) + s * scale;
    }
  });
  return 0;
}

namespace {
/*! \brief g[0..cnt) = sum over the W slots of elements [i0, i0+cnt), format fixed at compile time */
template <int FMT>
inline void GatherBlock(const ps_update_args& a, size_t i0, int cnt, size_t npad, const float* e4m3,
                        float* g) {
  for (int j = 0; j < cnt; ++j) g[j] = 0.f;
  for (int w = 0; w < a.num_grads; ++w) {
    const unsigned char* base = static_cast<const unsigned char*>(a.grads[w]);
    if (FMT == PS_GRAD_BF16) {
      const uint16_t* s = reinterpret_cast<const uint16_t*>(base) + i0;
      for (int j = 0; j < cnt; ++j) g[j] += Bf16ToF32(s[j]);
    } else if (FMT == PS_GRAD_FP8BLOCK) {
      const unsigned char* q = base + i0;
      const unsigned char* sc = base + npad;
      for (int j = 0; j < cnt; ++j) g[j] += e4m3[q[j]] * Exp2FromE8m0(sc[(i0 + j) >> 5]);
    } else {
      const float* s = reinterpret_cast<const float*>(base) + i0;
      for (int j = 0; j < cnt; ++j) g[j] += s[j];
    }
  }
}

template <int FMT>
void UpdateRange(const ps_update_args& args, const ps_opt_params& opt, size_t b0, size_t b1) {
  constexpr int kBlock = 256;
  const size_t npad = (args.n + 31) / 32 * 32;
  const float* e4m3 = E4m3Table();
  const bool adam = opt.optimizer == PS_OPT_ADAMW;
  const float inv_bc1 = adam ? 1.f / opt.bias_corr1 : 1.f, inv_bc2 = adam ? 1.f / opt.bias_corr2 : 1.f;
  float g[kBlock], pnew[kBlock];
  for (size_t i0 = b0; i0 < b1; i0 += kBlock) {
    const int cnt = static_cast<int>(std::min<size_t>(kBlock, b1 - i0));
    GatherBlock<FMT>(args, i0, cnt, npad, e4m3, g);
    float* p = args.master + i0;
    float* m = args.m + i0;
    if (adam) {
      float* v = args.v + i0;
      for (int j = 0; j < cnt; ++j) {
        const float gj = g[j] * opt.grad_scale;
        const float mj = opt.beta1 * m[j] + (1.f - opt.beta1) * gj;
        const float vj = opt.beta2 * v[j] + (1.f - opt.beta2) * gj * gj;
        const float denom = std::sqrt(vj * inv_bc2) + opt.eps;
        pnew[j] = p[j] - opt.lr * ((mj * inv_bc1) / denom + opt.weight_decay * p[j]);
        m[j] = mj;
        v[j] = vj;
      }
    } else {
      for (int j = 0; j < cnt; ++j) {
        const float gj = g[j] * opt.grad_scale + opt.weight_decay * p[j];
        const float mj = opt.beta1 * m[j] + gj;
        pnew[j] = p[j] - opt.lr * mj;
        m[j] = mj;
      }
    }
    for (int j = 0; j < cnt; ++j) p[j] = pnew[j];
    for (int k = 0; k < args.num_outs; ++k) {
      if (args.out_f32) {
        float* out = static_cast<float*>(args.outs[k]) + i0;
        for (int j = 0; j < cnt; ++j) out[j] = pnew[j];
      } else {
        uint16_t* out = static_cast<uint16_t*>(args.outs[k]) + i0;
        for (int j = 0; j < cnt; ++j) out[j] = F32ToBf16(pnew[j]);
      }
    }
  }
}
}  // namespace

extern "C" int ps_host_update(const ps_update_args* a, const ps_opt_params* o) {
  if (a->n == 0) return 0;
  if (a->num_grads < 1 || a->num_grads > PS_MAX_FANIN) return 1;
  if (a->num_outs < 0 || a->num_outs > PS_MAX_FANOUT) return 1;
  const int fmt = a->grad_format;
  if (fmt != PS_GRAD_BF16 && fmt != PS_GRAD_FP8BLOCK && fmt != PS_GRAD_F32) return 1;
  const ps_update_args args = *a;
  const ps_opt_params opt = *o;
  ParallelFor(args.n, 256, [=](size_t b0, size_t b1) {
    if (fmt == PS_GRAD_BF16) UpdateRange<PS_GRAD_BF16>(args, opt, b0, b1);
    else if (fmt == PS_GRAD_FP8BLOCK) UpdateRange<PS_GRAD_FP8BLOCK>(args, opt, b0, b1);
    else UpdateRange<PS_GRAD_F32>(args, opt, b0, b1);
  });
  return 0;
}

extern "C" size_t ps_rows_scratch_bytes(size_t rows, int max_grads) {
  return sizeof(ps_rows_scratch_hdr) + rows * 4 * (2 + static_cast<size_t>(max_grads));
}

namespace {
template <int FMT>
void UpdateRows(const ps_update_rows_args& a, const ps_opt_params& opt, const uint32_t* pos,
                const uint32_t* list, size_t r0, size_t r1) {
  const size_t D = static_cast<size_t>(a.dim);
  const float* e4m3 = E4m3Table();
  const bool adam = opt.optimizer == PS_OPT_ADAMW;
  const float inv_bc1 = adam ? 1.f / opt.bias_corr1 : 1.f, inv_bc2 = adam ? 1.f / opt.bias_corr2 : 1.f;
  std::vector<float> g(D);
  for (size_t r = r0; r < r1; ++r) {
    const size_t id = list[r];
    std::fill(g.begin(), g.end(), 0.f);
    for (int w = 0; w < a.num_grads; ++w) {  // fixed slot order, as on the GPU
      const uint32_t s = pos[static_cast<size_t>(w) * a.rows + id];
      if (s == 0) continue;
      const size_t i = ~s;
      const unsigned char* vals = static_cast<const unsigned char*>(a.grads[w]) +
                                  (static_cast<size_t>(a.num_rows[w]) + 3) / 4 * 16;
      if (FMT == PS_GRAD_BF16) {
        const uint16_t* q = reinterpret_cast<const uint16_t*>(vals) + i * D;
        for (size_t j = 0; j < D; ++j) g[j] += Bf16ToF32(q[j]);
      } else if (FMT == PS_GRAD_FP8BLOCK) {
        const unsigned char* q = vals + i * D;
        const unsigned char* sc = vals + static_cast<size_t>(a.num_rows[w]) * D + i * D / 32;
        for (size_t j = 0; j < D; ++j) g[j] += e4m3[q[j]] * Exp2FromE8m0(sc[j >> 5]);
      } else {
        const float* q = reinterpret_cast<const float*>(vals) + i * D;
        for (size_t j = 0; j < D; ++j) g[j] += q[j];
      }
    }
    float* p = a.master + id * D;
    float* m = a.m + id * D;
    float* v = adam ? a.v + id * D : nullptr;
    for (size_t j = 0; j < D; ++j) {
      const float gj = g[j] * opt.grad_scale;
      float pn;
      if (adam) {
        const float mj = opt.beta1 * m[j] + (1.f - opt.beta1) * gj;
        const float vj = opt.beta2 * v[j] + (1.f - opt.beta2) * gj * gj;
        const float denom = std::sqrt(vj * inv_bc2) + opt.eps;
        pn = p[j] - opt.lr * ((mj * inv_bc1) / denom + opt.weight_decay * p[j]);
        m[j] = mj;
        v[j] = vj;
      } else {
        const float gw = gj + opt.weight_decay * p[j];
        const float mj = opt.beta1 * m[j] + gw;
        pn = p[j] - opt.lr * mj;
        m[j] = mj;
      }
      p[j] = pn;
    }
    for (int k = 0; k < a.num_outs; ++k) {
      if (a.out_f32) {
        memcpy(static_cast<float*>(a.outs[k]) + id * D, p, D * 4);
      } else {
        uint16_t* out = static_cast<uint16_t*>(a.outs[k]) + id * D;
        for (size_t j = 0; j < D; ++j) out[j] = F32ToBf16(p[j]);
      }
    }
  }
}
}  // namespace

extern "C" int ps_host_update_rows(const ps_update_rows_args* args, const ps_opt_params* o) {
  const ps_update_rows_args a = *args;
  if (a.num_grads < 1 || a.num_grads > PS_MAX_FANIN) return 1;
  if (a.num_outs < 0 || a.num_outs > PS_MAX_FANOUT) return 1;
  if (a.dim <= 0 || a.dim % 8 != 0 || a.rows > 0xffffffffull) return 1;
  const int fmt = a.grad_format;
  if (fmt != PS_GRAD_BF16 && fmt != PS_GRAD_FP8BLOCK && fmt != PS_GRAD_F32) return 1;
  if (fmt == PS_GRAD_FP8BLOCK && a.dim % 32 != 0) return 1;
  size_t total = 0;
  for (int w = 0; w < a.num_grads; ++w) total += a.num_rows[w];
  if (total == 0) return 0;
  // the same scratch and the same marking rules as k_rows_mark (update_rows_kernels.cu)
  ps_rows_scratch_hdr* hdr = static_cast<ps_rows_scratch_hdr*>(a.scratch);
  uint32_t* touched = reinterpret_cast<uint32_t*>(hdr + 1);
  uint32_t* list = touched + a.rows;
  uint32_t* pos = list + a.rows;
  uint32_t count = 0;
  for (int w = 0; w < a.num_grads; ++w) {
    const uint32_t* ids = static_cast<const uint32_t*>(a.grads[w]);
    for (uint32_t i = 0; i < a.num_rows[w]; ++i) {
      const uint32_t id = ids[i];
      if (id >= a.rows) {
        ++hdr->bad;
        continue;
      }
      uint32_t& s = pos[static_cast<size_t>(w) * a.rows + id];
      if (s != 0) {  // a repeated id: its first occurrence stays
        ++hdr->bad;
        continue;
      }
      s = ~i;
      if (!touched[id]) {
        touched[id] = 1;
        list[count++] = id;
      }
    }
  }
  const ps_opt_params opt = *o;
  ParallelFor(static_cast<size_t>(count) * a.dim, a.dim, [&](size_t e0, size_t e1) {
    const size_t r0 = e0 / a.dim, r1 = e1 / a.dim;
    if (fmt == PS_GRAD_BF16) UpdateRows<PS_GRAD_BF16>(a, opt, pos, list, r0, r1);
    else if (fmt == PS_GRAD_FP8BLOCK) UpdateRows<PS_GRAD_FP8BLOCK>(a, opt, pos, list, r0, r1);
    else UpdateRows<PS_GRAD_F32>(a, opt, pos, list, r0, r1);
  });
  for (uint32_t r = 0; r < count; ++r) {
    const uint32_t id = list[r];
    touched[id] = 0;
    for (int w = 0; w < a.num_grads; ++w) pos[static_cast<size_t>(w) * a.rows + id] = 0;
  }
  return 0;
}
