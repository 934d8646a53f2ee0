/**
 * \file ps_kernels.h
 * \brief Host-side launch API of the sm_100a data-plane kernels.
 *
 * These kernels are the "NIC" of the NVLink van and the compute of the
 * GPU-resident server (SURVEY §2.4 D1-D3: the reference does this work with NIC
 * DMA, CPU memcpy and a scalar `store[key] += val` loop):
 *   ps_launch_copy      K_push / K_pull: move (and optionally scale, cast to bf16,
 *                       or block-quantise to fp8-e4m3) a value buffer into a
 *                       destination that may be *peer* HBM mapped over NVLink.
 *   ps_launch_update    K_update: for one parameter shard, dequantise + sum the W
 *                       worker gradient slots, apply SGD-momentum or AdamW on the
 *                       fp32 master / moments, and emit bf16 parameters to up to
 *                       8 destinations at once (local shard copy + every worker's
 *                       parameter buffer, i.e. update fused with the pull reply).
 *   ps_launch_update_rows  the same for a row-sparse shard (embedding table): only the rows
 *                       some worker pushed are summed, stepped and fanned out.
 *   ps_launch_sum       plain W-way dequantising reduction (KVServer default handle).
 * All take a cudaStream_t and never synchronise. No cuBLAS/NCCL anywhere.
 */
#ifndef PS_KERNELS_PS_KERNELS_H_
#define PS_KERNELS_PS_KERNELS_H_
#include <cstddef>
#include <cstdint>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* ps_stream_t;

/*! \brief wire formats; numerically identical to ps::WireCodec */
enum {
  PS_CODEC_RAW = 0,
  PS_CODEC_F32_TO_BF16 = 1,
  PS_CODEC_BF16_SCALE = 2,
  PS_CODEC_F32_TO_FP8BLOCK = 3,
  PS_CODEC_BF16_TO_FP8BLOCK = 4,
};

/*! \brief gradient slot formats K_update / ps_launch_sum can read */
enum {
  PS_GRAD_F32 = 0,
  PS_GRAD_BF16 = 1,
  /* [n_pad e4m3 bytes][n_pad/32 e8m0 bytes], n_pad = roundup(n,32). Scale byte b means 2^(b-127);
   * encoders write b in [1, 254] (exponent in [-126, 127]) and b = 0 only for an all-zero block. */
  PS_GRAD_FP8BLOCK = 2,
  /* NVLS in-switch aggregation: grads[0] is a MULTICAST address bound to the same offset of
   * every worker's (symmetric) bf16 gradient buffer; num_grads must be 1. The kernel reads it
   * with multimem.ld_reduce.add (fp32 accumulation inside the NVSwitch), so the W-way sum
   * costs one 2 B/element stream on the server's link instead of W slot reads. The buffers
   * must be padded to an even element count (the ragged tail loads bf16 pairs). */
  PS_GRAD_MC_BF16 = 3,
};

enum { PS_OPT_SGD = 0, PS_OPT_ADAMW = 1 };

#define PS_MAX_FANIN 8
#define PS_MAX_FANOUT 9

/*!
 * \brief dst <- codec(src). n_src_bytes counts bytes of the *source*.
 * \param max_ctas cap on the grid (0 = default: enough to saturate NVLink / HBM)
 * \return 0 on success, else a cudaError_t
 */
int ps_launch_copy(void* dst, const void* src, size_t n_src_bytes, int codec, float scale,
                   int max_ctas, ps_stream_t stream);

/*!
 * \brief in-kernel completion: when every CTA of the (last) kernel of a launch has stored its
 *        bytes, the last one to finish stores `value` to `*flag` with st.release.sys — the
 *        receiver of the payload (a van thread polling a shared-memory ring, or a peer GPU)
 *        needs no host thread of the sender to learn that the data has landed. This is the
 *        "immediate" of the reference's RDMA WRITE_WITH_IMM (src/rdma_transport.h:211-231).
 *        `counter` is a zero-initialised device word owned by the stream (reset by the kernel).
 */
typedef struct {
  unsigned* counter;
  unsigned long long* flag;   // device-visible address (device memory or mapped host memory)
  unsigned long long value;
} ps_signal;

/*! \brief ps_launch_copy + completion signal (sig may be null) */
int ps_launch_copy_signal(void* dst, const void* src, size_t n_src_bytes, int codec, float scale,
                          int max_ctas, const ps_signal* sig, ps_stream_t stream);
/*!
 * \brief pull fan-out through the switch: `mc_dst` is a multicast address (see
 *        Van::AllocSymmetric) — every 16-byte vector is stored once with multimem.st and lands in
 *        all bound buffers. Addresses and `n_bytes` must be multiples of 16.
 */
int ps_launch_copy_multicast(void* mc_dst, const void* src, size_t n_bytes, int max_ctas,
                             const ps_signal* sig, ps_stream_t stream);
/*! \brief only the signal: ordered after everything enqueued on `stream` before it */
int ps_launch_signal(const ps_signal* sig, ps_stream_t stream);

/*!
 * \brief the copy engine (engine_kernels.cu): descriptors are POSTED into a ring in mapped host
 *        memory and executed by an on-demand persistent kernel — no driver call per copy. One
 *        engine per device and process (ps_engine_create hands out the shared instance).
 *        Completions are published in posting order: `value` is stored to `*flag`
 *        (st.release.sys; flag may be null) once the bytes are visible system-wide.
 */
typedef struct ps_engine ps_engine;
ps_engine* ps_engine_create(int device, int num_ctas, int idle_us);
void ps_engine_destroy(ps_engine* e);
int ps_engine_post(ps_engine* e, void* dst, const void* src, size_t bytes, unsigned long long* flag,
                   unsigned long long value, unsigned long long* ticket);
/*! \brief completions are published in posting order: has / wait until the post that returned `ticket` completed
 *  (an engine is shared by everything on its device; a user waits for ITS last ticket, not for everybody) */
int ps_engine_done(ps_engine* e, unsigned long long ticket);
void ps_engine_wait(ps_engine* e, unsigned long long ticket);
/*! \brief has everything posted so far been completed? / wait until it has */
int ps_engine_idle(ps_engine* e);
void ps_engine_drain(ps_engine* e);
void ps_engine_stats(ps_engine* e, unsigned long long* launches, unsigned long long* items);

/*! \brief byte copies of up to PS_MAX_COPY_SEGS unrelated buffers per kernel launch */
#define PS_MAX_COPY_SEGS 32
typedef struct {
  void* dst;
  const void* src;
  size_t bytes;
} ps_copy_seg;
int ps_launch_copy_multi(const ps_copy_seg* segs, int nseg, int max_ctas, ps_stream_t stream);

/*! \brief inverse transforms, for tests and for unpacking a pulled wire buffer */
int ps_launch_decode(void* dst_f32, const void* wire, size_t n_elems, int grad_format,
                     ps_stream_t stream);

typedef struct {
  int optimizer;        // PS_OPT_*
  float lr;
  float beta1;          // SGD: momentum
  float beta2;
  float eps;
  float weight_decay;   // decoupled (AdamW) / L2 for SGD
  float bias_corr1;     // 1 - beta1^t (host computed), 1 for SGD
  float bias_corr2;     // 1 - beta2^t
  float grad_scale;     // applied to the summed gradient (e.g. 1/W)
} ps_opt_params;

typedef struct {
  size_t n;                            // elements in the shard
  int num_grads;                       // W
  int grad_format;                     // PS_GRAD_*
  const void* grads[PS_MAX_FANIN];     // W slots (local HBM, written by the workers)
  float* master;                       // fp32 parameters (in/out)
  float* m;                            // first moment / momentum (in/out)
  float* v;                            // second moment (AdamW only)
  int num_outs;                        // bf16 destinations
  void* outs[PS_MAX_FANOUT];           // local copy and/or peer-mapped worker buffers
  int out_f32;                         // outs[] receive fp32 instead of bf16
  /* NVLS: a multicast address (cuMulticast / symmetric memory) bound to the SAME offset of
   * every worker's parameter buffer. When set, the 16-byte body stores go out as ONE
   * multimem.st per vector (the switch replicates it to all workers) and only
   * outs[0..body_outs) are written unicast in the body; the ragged tail (< 8 elements)
   * still uses all of outs[]. */
  void* mc_out;
  int body_outs;
} ps_update_args;

/*!
 * \brief fused dequant + W-way sum + optimizer + bf16 fan-out for one shard
 * \return cudaErrorMisalignedAddress, before anything is launched, unless master, m, v (AdamW),
 *         every grads[w], every outs[k] and mc_out are 16-byte aligned
 */
int ps_launch_update(const ps_update_args* args, const ps_opt_params* opt, int max_ctas,
                     ps_stream_t stream);

/*!
 * \brief one round of a ROW-SPARSE shard of rows x dim fp32 elements (an embedding table).
 *        Slot w holds num_rows[w] = R_w unique local row ids and their gradient rows:
 *            [u32 ids, R_w entries, zero-padded to a multiple of 4][values]
 *            values: PS_GRAD_F32  R_w*dim f32 | PS_GRAD_BF16  R_w*dim bf16 |
 *                    PS_GRAD_FP8BLOCK  [R_w*dim e4m3][R_w*dim/32 e8m0]   (dim % 32 == 0)
 *        The contributions to each row of the union are summed in slot order (w = 0..W-1), the
 *        optimizer step runs on those rows only ("lazy": untouched rows keep master, m and v bit
 *        for bit and get no weight decay), and the new rows are stored at their row offsets into
 *        every outs[k]; nothing else of a destination is written. R_w = 0 is legal.
 *        An id >= rows, or an id repeated within one slot (its first occurrence is used), is
 *        skipped and counted in the scratch header's `bad`.
 */
typedef struct {
  size_t rows;                         // rows in the shard
  int dim;                             // D: elements per row, a multiple of 8
  int num_grads;                       // W, 1..PS_MAX_FANIN
  int grad_format;                     // PS_GRAD_F32 / PS_GRAD_BF16 / PS_GRAD_FP8BLOCK
  const void* grads[PS_MAX_FANIN];     // W slots in the layout above
  uint32_t num_rows[PS_MAX_FANIN];     // R_w
  float* master;                       // rows x dim fp32 (in/out)
  float* m;
  float* v;                            // AdamW only
  int num_outs;                        // destinations, each rows x dim
  void* outs[PS_MAX_FANOUT];
  int out_f32;                         // outs[] receive fp32 instead of bf16
  /* ps_rows_scratch_bytes(rows, >= W) bytes, zero-filled once when allocated: every launch
   * leaves it zeroed again except for the header's `bad`, so it is kept between rounds */
  void* scratch;
} ps_update_rows_args;

/*! \brief head of the row-sparse scratch; then u32 touched[rows], list[rows], slot_of[W][rows] */
typedef struct {
  uint32_t count;            // rows in the union of the current launch
  uint32_t done;             // CTAs finished (the last one resets count and done)
  unsigned long long bad;    // ids skipped since the scratch was allocated (never reset)
} ps_rows_scratch_hdr;

size_t ps_rows_scratch_bytes(size_t rows, int max_grads);

/*!
 * \brief row-sparse fused update: marks the union on the device, then one grid sized to the GPU
 *        walks it (gather-sum, optimizer, scatter). No host synchronisation.
 * \return cudaErrorInvalidValue for bad counts, formats or dim; cudaErrorMisalignedAddress, before
 *         anything is launched, unless master, m, v (AdamW), every grads[w] and every outs[k] are
 *         16-byte aligned
 */
int ps_launch_update_rows(const ps_update_rows_args* args, const ps_opt_params* opt, int max_ctas,
                          ps_stream_t stream);

/*! \brief out_f32[i] (+)= sum_w decode(grads[w])[i] * scale */
int ps_launch_sum(float* out_f32, const void* const* grads, int num_grads, int grad_format,
                  size_t n, float scale, int accumulate, ps_stream_t stream);

/*! \brief fill with a deterministic pattern / checksum helpers used by stress tests */
int ps_launch_fill_u32(void* dst, size_t n_words, uint32_t seed, ps_stream_t stream);
int ps_launch_checksum_u32(const void* src, size_t n_words, unsigned long long* out_dev,
                           ps_stream_t stream);

/*! \brief number of kernels launched by this library in this process (bench accounting) */
unsigned long long ps_kernel_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif  // PS_KERNELS_PS_KERNELS_H_
