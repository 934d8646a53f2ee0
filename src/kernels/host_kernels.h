/**
 * \file host_kernels.h
 * \brief CPU twins of the sm_100a data-plane kernels (ps_kernels.h), same wire formats.
 *
 * The reference's servers are CPU processes (`store[key] += val`, include/ps/kv_app.h:441-447);
 * a deployment that keeps CPU servers, a host-only van (tcp / shm) that is asked for a wire
 * codec, and every test that has to run without a GPU use these. They are also the
 * independent implementation the GPU kernels are compared against.
 * All functions are synchronous and return 0 on success.
 */
#ifndef PS_KERNELS_HOST_KERNELS_H_
#define PS_KERNELS_HOST_KERNELS_H_
#include "kernels/ps_kernels.h"

#ifdef __cplusplus
extern "C" {
#endif

/*! \brief dst <- codec(src); n_src_bytes counts bytes of the source (PS_CODEC_*) */
int ps_host_copy(void* dst, const void* src, size_t n_src_bytes, int codec, float scale);
/*! \brief wire (PS_GRAD_*) -> fp32 */
int ps_host_decode(float* dst_f32, const void* wire, size_t n_elems, int grad_format);
/*! \brief out[i] (+)= scale * sum_w decode(grads[w])[i] */
int ps_host_sum(float* out_f32, const void* const* grads, int num_grads, int grad_format, size_t n,
                float scale, int accumulate);
/*! \brief fused dequant + W-way sum + AdamW / SGD + bf16 (or fp32) fan-out; mc_out is ignored */
int ps_host_update(const ps_update_args* args, const ps_opt_params* opt);
/*! \brief row-sparse twin of ps_launch_update_rows: same slot layout, scratch and bad-id counting */
int ps_host_update_rows(const ps_update_rows_args* args, const ps_opt_params* opt);

#ifdef __cplusplus
}
#endif
#endif  // PS_KERNELS_HOST_KERNELS_H_
