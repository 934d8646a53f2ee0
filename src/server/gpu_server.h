/**
 * \file gpu_server.h
 * \brief GpuServer: a GPU-resident synchronous parameter server built on KVServer.
 *
 * The reference stops at "call the user's ReqHandle" (include/ps/kv_app.h:378-385)
 * and ships only `store[key] += val` (:430-452); aggregation, optimizer and the
 * BytePS-style sync rounds live outside it. This engine is that missing half,
 * designed for B200:
 *   - every key is a parameter shard whose fp32 master + optimizer moments stay
 *     resident in this server's HBM (ZeRO-like sharding by key range);
 *   - a push lands (one-sidedly, over NVLink) in a per-(key, worker) slot in wire
 *     form (bf16 or block-scaled fp8); it is acked on arrival;
 *   - when all W workers have pushed a key — and, in fused mode, asked to pull
 *     it — ONE kernel (src/kernels/update_kernels.cu) dequantises and sums the W
 *     slots, runs AdamW / SGD on the fp32 state and stores bf16 parameters
 *     directly into every worker's parameter buffer through the peer mapping:
 *     push handler + optimizer + pull reply in a single memory-bound pass;
 *   - pulls that cannot be fused (late, or initial fetch) are cast from the fp32 master
 *     straight into the worker's buffer by the copy kernel; the server keeps no bf16
 *     copy of its shards (12 B of state per parameter).
 * The handler only enqueues work on the van's data stream and never blocks, so
 * it can run inline on the van thread (PS_DIRECT_DISPATCH=1).
 *
 * The same engine runs on CPU servers — the reference's deployment model — when the
 * process uses a host van (tcp / shm / multivan) or PS_SERVER_DEVICE=cpu: shards in host
 * memory, the CPU twins of the kernels (src/kernels/host_kernels.cc), pull replies written
 * into the worker's shared-memory buffer by the shm van or sent two-sided over TCP.
 */
#ifndef PS_SERVER_GPU_SERVER_H_
#define PS_SERVER_GPU_SERVER_H_
#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "kernels/ps_kernels.h"
#include "ps/kv_app.h"

namespace ps {

/*! \brief KVMeta::option bits of an initial-value push (per-shard optimizer settings) */
enum GpuServerInitOption : int {
  kInitNoWeightDecay = 1,  // norms, biases, embeddings: exclude this shard from weight decay
  /* a row-sparse shard (embedding table): option = flags | (D << 8), D = row width in elements
   * (a multiple of 8, D < 2^23); gradients then arrive as kCmdGradRows pushes */
  kInitRowSparse = 2,
};

/*! \brief `cmd` values understood by GpuServer */
enum GpuServerCmd : int {
  kCmdGrad = 0,        // push: gradient contribution for the current round
  kCmdInitBf16 = 101,  // push: initial parameter values, bf16 (first writer wins)
  kCmdInitF32 = 102,   // push: initial parameter values, fp32
  kCmdSetLr = 103,     // push: one fp32 value = new learning rate of this server (any key it owns)
  /* push, codec kCodecRaw, option = (R << 2) | PS_GRAD_F32 / PS_GRAD_BF16 / PS_GRAD_FP8BLOCK:
   * R rows of a row-sparse shard, laid out as ps_update_rows_args describes. R may be 0. */
  kCmdGradRows = 104,
};

struct GpuServerConfig {
  int num_workers = 1;
  /*! \brief format of kCodecRaw pushes (PS_GRAD_BF16 or PS_GRAD_F32) */
  int raw_grad_format = PS_GRAD_BF16;
  ps_opt_params opt;
  /*! \brief wait for all W pulls of a round and fan the new parameters out from the update kernel */
  bool fuse_pull = true;
  /*!
   * \brief asynchronous SGD (docs/overview.md of the reference: "asynchronous: the server
   *        updates as soon as a gradient arrives"): every push is applied on arrival as its own
   *        optimizer step, pulls are answered at once with the current parameters; there are no
   *        rounds and no barrier between workers. `opt.grad_scale` is applied per push.
   */
  bool async_updates = false;
  /*! \brief cap on CTAs per kernel, 0 = fill the GPU */
  int max_ctas = 0;
  GpuServerConfig() {
    opt.optimizer = PS_OPT_ADAMW;
    opt.lr = 1e-3f;
    opt.beta1 = 0.9f;
    opt.beta2 = 0.95f;
    opt.eps = 1e-8f;
    opt.weight_decay = 0.f;
    opt.bias_corr1 = 1.f;
    opt.bias_corr2 = 1.f;
    opt.grad_scale = 1.f;
  }
};

class GpuServer {
 public:
  GpuServer(int app_id, const GpuServerConfig& cfg, int instance_idx = 0);
  ~GpuServer();

  void SetLearningRate(float lr);
  float learning_rate();
  /*!
   * \brief NVLS pull fan-out. Every worker keeps its parameters in a buffer that is
   *        symmetric across the job (same layout at the same offset) and bound to one
   *        multicast object. `mc_base` is this process's mapping of the multicast address,
   *        `peer_bases[w]` its unicast mapping of worker w's buffer. Pull requests that
   *        name their destination as MemRef{kSymmetricRegion, offset} are then answered by
   *        ONE multimem.st stream from the update kernel instead of W unicast streams.
   */
  void SetSymmetricParams(void* mc_base, const std::vector<void*>& peer_bases, size_t bytes);
  /*!
   * \brief NVLS aggregation. Workers stage bf16 gradients in a second symmetric buffer and
   *        push only a descriptor {kSymmetricRegion, offset}; `mc_base` is this process's
   *        multicast mapping of that buffer. The update kernel then reads the W-way SUM with
   *        multimem.ld_reduce (the switch adds in fp32): no landing slots, one 2 B/element
   *        stream into the server instead of W. Server-only ranks keep their copy zeroed.
   */
  void SetSymmetricGrads(void* mc_base, size_t bytes);
  /*! \brief update kernels whose gradients were reduced inside the switch */
  uint64_t num_switch_reductions() const { return mc_reduce_.load(); }
  /*! \brief update kernels whose fan-out went through the multicast address */
  uint64_t num_multicast_fanouts() const { return mcast_.load(); }
  /*! \brief optimizer steps applied, summed over keys */
  uint64_t num_updates() const { return updates_.load(); }
  /*! \brief update kernels whose destinations included worker buffers (fused pull replies) */
  uint64_t num_fused_fanouts() const { return fused_.load(); }
  size_t num_keys();
  /*! \brief bytes of HBM held by parameter + optimizer state (and the scratch of row-sparse shards) */
  size_t state_bytes();
  /*! \brief row ids skipped by row-sparse updates (>= rows, or repeated in one push), summed over
   *         shards. Synchronous device read: for tests and diagnostics */
  uint64_t num_bad_rows();

  /*! \brief dump / restore every shard this server owns (fp32 master, m, v, step) */
  bool SaveCheckpoint(const std::string& path);
  bool LoadCheckpoint(const std::string& path);

  /*! \brief copy of a shard's fp32 master to host (tests, evaluation) */
  bool ReadMaster(Key key, std::vector<float>* out);

  KVServer<char>* kv() { return server_.get(); }
  /*! \brief true: shards in HBM, sm_100a kernels; false: shards in host memory, CPU twins */
  bool on_device() const;

  class Backend;  // memory + math provider (gpu_server.cc)

 private:
  struct Shard {
    size_t n = 0;
    float* master = nullptr;
    float* m = nullptr;
    float* v = nullptr;
    bool initialized = false;
    bool no_weight_decay = false;
    int step = 0;
    int grad_format = PS_GRAD_BF16;
    int dim = 0;                         // row-sparse shard: row width; 0 = dense
    void* scratch = nullptr;             // row-sparse shard: ps_rows_scratch_bytes(n / dim, W)
    std::vector<uint32_t> num_rows;      // row-sparse shard: rows pushed per worker rank this round
    std::vector<const void*> slots;      // per worker rank: landing slot of this round
    std::vector<SArray<char>> slot_refs; // host shards: keeps a two-sided payload alive until the round runs
    std::vector<void*> staged;           // device shards: per rank, where a gradient that arrived in HOST memory
    std::vector<size_t> staged_cap;      //   (worker on another host) is uploaded to; kept and reused
    std::vector<char> pushed;            // per worker rank: pushed in the open round
    int num_pushed = 0;
    std::vector<KVMeta> waiting_pulls;   // pulls of workers that already pushed this round
  };

  void Handle(const KVMeta& req, const KVPairs<char>& data, KVServer<char>* server);
  void HandleInit(Shard* s, const KVMeta& req, const KVPairs<char>& data);
  void HandleGrad(Shard* s, const KVMeta& req, const KVPairs<char>& data);
  void HandlePull(Shard* s, const KVMeta& req, const KVPairs<char>& data);
  void MaybeRunRound(Key key, Shard* s);
  void ApplyOnArrival(Shard* s, int rank);
  void ServePullFromLocal(Key key, Shard* s, const KVMeta& req);
  void MakeRowSparse(Shard* s, int dim);
  void RunUpdate(Shard* s, const ps_update_args& a, const ps_opt_params& o, int first_rank);
  Shard* GetShard(Key key, size_t n);
  void* WorkerDest(const KVMeta& pull);
  static size_t ElemsOf(const KVMeta& req);
  static int FormatOf(const KVMeta& req, int raw_format);

  GpuServerConfig cfg_;
  int instance_idx_;
  int dev_ = 0;
  void* stream_ = nullptr;
  std::unique_ptr<Backend> be_;
  std::unique_ptr<KVServer<char>> server_;
  Postoffice* po_ = nullptr;
  std::mutex mu_;
  std::unordered_map<Key, Shard> shards_;
  std::atomic<uint64_t> updates_{0};
  std::atomic<uint64_t> fused_{0};
  std::atomic<uint64_t> mcast_{0};
  std::atomic<uint64_t> mc_reduce_{0};
  void* mc_grad_base_ = nullptr;
  size_t symm_grad_bytes_ = 0;
  void* mc_base_ = nullptr;
  std::vector<void*> peer_bases_;
  size_t symm_bytes_ = 0;
};

}  // namespace ps
#endif  // PS_SERVER_GPU_SERVER_H_
