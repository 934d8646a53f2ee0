/**
 * \file gpu_server.cc
 * \brief GpuServer implementation (see gpu_server.h).
 */
#include "server/gpu_server.h"

#ifdef PS_USE_CUDA
#include <cuda_runtime.h>
#endif

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "core/nvtx.h"
#include "kernels/host_kernels.h"
#include "van/mem_domain.h"

namespace ps {

/*!
 * \brief where the shards live and who does the math. The round logic above it (sync
 *        rounds, fused pull fan-out, late pulls, checkpoints) is the same for both:
 *        CudaBackend — HBM + the sm_100a kernels on the van's stream (asynchronous);
 *        HostBackend — host memory + the CPU twins (synchronous): the engine for CPU
 *        servers (the reference's deployment model) and for GPU-less tests.
 */
class GpuServer::Backend {
 public:
  virtual ~Backend() {}
  virtual bool on_device() const = 0;
  virtual void Bind() {}
  /*! \brief zero-filled memory for fp32 state */
  virtual void* Alloc(size_t bytes) = 0;
  virtual void Free(void* p) = 0;
  virtual void Decode(float* dst, const void* wire, size_t n, int fmt) = 0;
  virtual void Update(const ps_update_args& a, const ps_opt_params& o, int max_ctas) = 0;
  virtual void UpdateRows(const ps_update_rows_args& a, const ps_opt_params& o, int max_ctas) = 0;
  virtual void Copy(void* dst, const void* src, size_t n_src_bytes, int codec, float scale,
                    int max_ctas) = 0;
  /*! \brief synchronous transfers between backend memory and host memory */
  virtual void Upload(void* dst, const void* host, size_t bytes) = 0;
  virtual void Download(void* host, const void* src, size_t bytes) = 0;
  /*! \brief all queued work has completed */
  virtual void Sync() = 0;
};

namespace {

class HostBackend : public GpuServer::Backend {
 public:
  bool on_device() const override { return false; }
  void* Alloc(size_t bytes) override {
    void* p = calloc(1, bytes ? bytes : 1);
    CHECK(p) << "out of host memory for " << bytes << " B of server state";
    return p;
  }
  void Free(void* p) override { free(p); }
  void Decode(float* dst, const void* wire, size_t n, int fmt) override {
    CHECK_EQ(ps_host_decode(dst, wire, n, fmt), 0);
  }
  void Update(const ps_update_args& a, const ps_opt_params& o, int /*max_ctas*/) override {
    CHECK_EQ(ps_host_update(&a, &o), 0) << "unsupported gradient format " << a.grad_format;
  }
  void UpdateRows(const ps_update_rows_args& a, const ps_opt_params& o, int /*max_ctas*/) override {
    CHECK_EQ(ps_host_update_rows(&a, &o), 0) << "bad row-sparse update (format " << a.grad_format << ")";
  }
  void Copy(void* dst, const void* src, size_t n, int codec, float scale, int /*max_ctas*/) override {
    CHECK_EQ(ps_host_copy(dst, src, n, codec, scale), 0);
  }
  void Upload(void* dst, const void* host, size_t bytes) override { memcpy(dst, host, bytes); }
  void Download(void* host, const void* src, size_t bytes) override { memcpy(host, src, bytes); }
  void Sync() override {}
};

#ifdef PS_USE_CUDA
#define GS_CUDA(expr)                                                             \
  do {                                                                            \
    cudaError_t e_ = (expr);                                                      \
    CHECK(e_ == cudaSuccess) << "CUDA: " #expr " -> " << cudaGetErrorString(e_);  \
  } while (0)

class CudaBackend : public GpuServer::Backend {
 public:
  CudaBackend(int dev, void* stream) : dev_(dev), stream_(static_cast<cudaStream_t>(stream)) {
    GS_CUDA(cudaSetDevice(dev_));
    if (!stream_) {
      GS_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
      own_stream_ = true;
    }
  }
  ~CudaBackend() override {
    cudaSetDevice(dev_);
    cudaStreamSynchronize(stream_);
    if (own_stream_) cudaStreamDestroy(stream_);
  }
  bool on_device() const override { return true; }
  void Bind() override { GS_CUDA(cudaSetDevice(dev_)); }
  void* Alloc(size_t bytes) override {
    void* p = nullptr;
    GS_CUDA(cudaMalloc(&p, bytes ? bytes : 1));
    GS_CUDA(cudaMemsetAsync(p, 0, bytes, stream_));
    return p;
  }
  void Free(void* p) override { cudaFree(p); }
  void Decode(float* dst, const void* wire, size_t n, int fmt) override {
    CHECK_EQ(ps_launch_decode(dst, wire, n, fmt, ps_stream()), 0);
  }
  void Update(const ps_update_args& a, const ps_opt_params& o, int max_ctas) override {
    CHECK_EQ(ps_launch_update(&a, &o, max_ctas, ps_stream()), 0);
  }
  void UpdateRows(const ps_update_rows_args& a, const ps_opt_params& o, int max_ctas) override {
    CHECK_EQ(ps_launch_update_rows(&a, &o, max_ctas, ps_stream()), 0);
  }
  void Copy(void* dst, const void* src, size_t n, int codec, float scale, int max_ctas) override {
    CHECK_EQ(ps_launch_copy(dst, src, n, codec, scale, max_ctas, ps_stream()), 0);
  }
  void Upload(void* dst, const void* host, size_t bytes) override {
    GS_CUDA(cudaMemcpyAsync(dst, host, bytes, cudaMemcpyHostToDevice, stream_));
    GS_CUDA(cudaStreamSynchronize(stream_));
  }
  void Download(void* host, const void* src, size_t bytes) override {
    GS_CUDA(cudaMemcpyAsync(host, src, bytes, cudaMemcpyDeviceToHost, stream_));
    GS_CUDA(cudaStreamSynchronize(stream_));
  }
  void Sync() override { GS_CUDA(cudaStreamSynchronize(stream_)); }

 private:
  ps_stream_t ps_stream() const { return reinterpret_cast<ps_stream_t>(stream_); }
  int dev_;
  cudaStream_t stream_;
  bool own_stream_ = false;
};
#endif  // PS_USE_CUDA

}  // namespace

namespace {
SArray<Key> OneKey(Key k) {
  SArray<Key> a(1);
  a[0] = k;
  return a;
}
SArray<int> OneLen(size_t bytes) {
  SArray<int> a(1);
  a[0] = static_cast<int>(std::min<size_t>(bytes, 0x7fffffff));
  return a;
}
}  // namespace

GpuServer::GpuServer(int app_id, const GpuServerConfig& cfg, int instance_idx)
    : cfg_(cfg), instance_idx_(instance_idx) {
  CHECK_GE(cfg_.num_workers, 1);
  CHECK_LE(cfg_.num_workers, PS_MAX_FANIN);
  po_ = Postoffice::GetServer(instance_idx);
  dev_ = po_->van()->my_node().dev_id;
  stream_ = po_->van()->DataStream();
  const std::string van_type = po_->van()->GetType();
  // a GPU van (nvl, nccl) means GPU-resident shards; host vans (tcp, shm, multivan) get the
  // CPU engine unless PS_SERVER_DEVICE=cuda asks for the GPU anyway
  bool want_device = dev_ >= 0 || van_type == "nvl" || van_type == "nccl";
  const std::string forced = GetEnvStr("PS_SERVER_DEVICE", "");
  if (forced == "cuda") want_device = true;
  if (forced == "cpu") want_device = false;
#ifdef PS_USE_CUDA
  if (want_device) {
    if (dev_ < 0) GS_CUDA(cudaGetDevice(&dev_));
    be_.reset(new CudaBackend(dev_, stream_));
  }
#else
  CHECK(!want_device) << "this build has no CUDA support (PS_USE_CUDA)";
#endif
  if (!be_) be_.reset(new HostBackend());
  server_.reset(new KVServer<char>(app_id, false, instance_idx));
  using namespace std::placeholders;
  server_->set_request_handle(std::bind(&GpuServer::Handle, this, _1, _2, _3));
  // Handle() never waits for the network (it enqueues kernels and sends replies): run it on the
  // receive thread while the queue is idle — one thread hop less per request
  // (not with launch coalescing: there the customer thread handles whole batches under one cork)
  server_->set_inline_dispatch(GetEnv("PS_SERVER_INLINE", 1) != 0 && GetEnv("PS_COALESCE_LAUNCHES", 0) == 0);
}

GpuServer::~GpuServer() {
  server_.reset();
  try {
    be_->Bind();
    be_->Sync();
  } catch (const std::exception& e) {  // e.g. the CUDA context is already gone at exit
    LOG(WARNING) << "server engine teardown: " << e.what();
  }
  for (auto& kv : shards_) {
    be_->Free(kv.second.master);
    be_->Free(kv.second.m);
    be_->Free(kv.second.v);
    if (kv.second.scratch) be_->Free(kv.second.scratch);
    for (void* p : kv.second.staged) {
      if (p) be_->Free(p);
    }
  }
}

bool GpuServer::on_device() const { return be_->on_device(); }

void GpuServer::SetLearningRate(float lr) {
  std::lock_guard<std::mutex> lk(mu_);
  cfg_.opt.lr = lr;
}

float GpuServer::learning_rate() {
  std::lock_guard<std::mutex> lk(mu_);
  return cfg_.opt.lr;
}

void GpuServer::SetSymmetricParams(void* mc_base, const std::vector<void*>& peer_bases,
                                   size_t bytes) {
  std::lock_guard<std::mutex> lk(mu_);
  CHECK_EQ(peer_bases.size(), static_cast<size_t>(cfg_.num_workers));
  mc_base_ = mc_base;
  peer_bases_ = peer_bases;
  symm_bytes_ = bytes;
}

void GpuServer::SetSymmetricGrads(void* mc_base, size_t bytes) {
  std::lock_guard<std::mutex> lk(mu_);
  mc_grad_base_ = mc_base;
  symm_grad_bytes_ = bytes;
}

size_t GpuServer::num_keys() {
  std::lock_guard<std::mutex> lk(mu_);
  return shards_.size();
}

size_t GpuServer::state_bytes() {
  std::lock_guard<std::mutex> lk(mu_);
  size_t b = 0;
  for (auto& kv : shards_) {
    b += kv.second.n * 12;
    if (kv.second.dim) b += ps_rows_scratch_bytes(kv.second.n / kv.second.dim, cfg_.num_workers);
  }
  return b;
}

uint64_t GpuServer::num_bad_rows() {
  std::lock_guard<std::mutex> lk(mu_);
  be_->Bind();
  uint64_t bad = 0;
  for (auto& kv : shards_) {
    if (!kv.second.scratch) continue;
    ps_rows_scratch_hdr h;
    be_->Download(&h, kv.second.scratch, sizeof(h));
    bad += h.bad;
  }
  return bad;
}

void GpuServer::MakeRowSparse(Shard* s, int dim) {
  CHECK_GT(dim, 0) << "a row-sparse shard needs its row width in option bits 8..30";
  CHECK_EQ(dim % 8, 0) << "row-sparse shard: the row width " << dim
                       << " is not a multiple of 8 (rows move as 16-byte vectors)";
  CHECK_EQ(s->n % static_cast<size_t>(dim), (size_t)0)
      << "row-sparse shard: " << s->n << " elements are not a whole number of rows of " << dim;
  CHECK_LE(s->n / dim, (size_t)0xffffffffu) << "row-sparse shard: row ids are 32-bit";
  s->dim = dim;
  s->scratch = be_->Alloc(ps_rows_scratch_bytes(s->n / dim, cfg_.num_workers));  // zero-filled
  s->num_rows.assign(cfg_.num_workers, 0);
}

void GpuServer::RunUpdate(Shard* s, const ps_update_args& a, const ps_opt_params& o, int first_rank) {
  if (!s->dim) {
    be_->Update(a, o, cfg_.max_ctas);
    return;
  }
  ps_update_rows_args r;
  memset(&r, 0, sizeof(r));
  r.rows = s->n / s->dim;
  r.dim = s->dim;
  r.num_grads = a.num_grads;
  r.grad_format = a.grad_format;
  for (int w = 0; w < a.num_grads; ++w) {
    r.grads[w] = a.grads[w];
    r.num_rows[w] = s->num_rows[first_rank + w];
  }
  r.master = a.master;
  r.m = a.m;
  r.v = a.v;
  r.num_outs = a.num_outs;  // unicast only: row shards never use the multicast fan-out
  for (int k = 0; k < a.num_outs; ++k) r.outs[k] = a.outs[k];
  r.scratch = s->scratch;
  be_->UpdateRows(r, o, cfg_.max_ctas);
}

size_t GpuServer::ElemsOf(const KVMeta& req) {
  const size_t bytes = static_cast<size_t>(req.val_len);
  if (req.cmd == kCmdInitF32) return bytes / 4;
  if (req.cmd == kCmdInitBf16) return bytes / 2;
  switch (req.codec) {
    case kCodecF32ToBf16:
    case kCodecF32ToFp8Block:
      return bytes / 4;
    default:
      return bytes / 2;  // bf16 sources (raw bf16, scaled bf16, bf16 -> fp8)
  }
}

int GpuServer::FormatOf(const KVMeta& req, int raw_format) {
  switch (req.codec) {
    case kCodecF32ToBf16:
    case kCodecBf16Scale:
      return PS_GRAD_BF16;
    case kCodecF32ToFp8Block:
    case kCodecBf16ToFp8Block:
      return PS_GRAD_FP8BLOCK;
    default:
      return raw_format;
  }
}

GpuServer::Shard* GpuServer::GetShard(Key key, size_t n) {
  auto it = shards_.find(key);
  if (it != shards_.end()) {
    if (n) CHECK_EQ(it->second.n, n) << "key " << key << " changed size";
    return &it->second;
  }
  CHECK_GT(n, (size_t)0) << "pull of unknown key " << key;
  Shard& s = shards_[key];
  s.n = n;
  s.master = static_cast<float*>(be_->Alloc(n * 4));
  s.m = static_cast<float*>(be_->Alloc(n * 4));
  s.v = static_cast<float*>(be_->Alloc(n * 4));
  s.slots.assign(cfg_.num_workers, nullptr);
  s.slot_refs.assign(cfg_.num_workers, SArray<char>());
  s.pushed.assign(cfg_.num_workers, 0);
  return &s;
}

void GpuServer::Handle(const KVMeta& req, const KVPairs<char>& data, KVServer<char>* /*server*/) {
  be_->Bind();
  std::lock_guard<std::mutex> lk(mu_);
  const Key key = data.keys.size() ? data.keys[0] : req.key;
  if (req.push && req.cmd == kCmdSetLr) {
    // remote control for learning-rate schedules: servers may live in other processes
    CHECK_EQ(data.vals.size(), sizeof(float)) << "CMD_SET_LR carries exactly one fp32 value";
    float lr = 0.f;
    if (data.vals.on_gpu()) be_->Download(&lr, data.vals.data(), sizeof(float));
    else memcpy(&lr, data.vals.data(), sizeof(float));
    cfg_.opt.lr = lr;
    server_->Response(req);
    return;
  }
  if (req.push && req.cmd == kCmdGradRows) {
    // the payload size varies with the rows pushed: the shard must exist (its init push came first)
    auto it = shards_.find(key);
    CHECK(it != shards_.end()) << "row-sparse gradient (kCmdGradRows) for key " << key
                               << ", which was never initialised";
    CHECK(!req.pull) << "kCmdGradRows is pushed, then pulled";
    Shard* s = &it->second;
    HandleGrad(s, req, data);
    MaybeRunRound(key, s);
    return;
  }
  if (req.push) {
    Shard* s = GetShard(key, ElemsOf(req));
    if (req.cmd == kCmdInitBf16 || req.cmd == kCmdInitF32) {
      CHECK(!req.pull) << "initial values are pushed, not push-pulled";
      HandleInit(s, req, data);
    } else {
      HandleGrad(s, req, data);
      if (req.pull) {
        // fused push-pull: the same message is also this worker's pull of the round's result;
        // it is answered once, by the pull reply (HandleGrad sent no ack)
        KVMeta pull = req;
        pull.push = false;
        pull.pull = false;
        pull.addr = req.pull_addr;
        pull.val_len = req.pull_len;
        pull.mem = req.pull_mem;
        HandlePull(s, pull, data);
      }
      MaybeRunRound(key, s);
    }
  } else {
    Shard* s = GetShard(key, 0);
    HandlePull(s, req, data);
    MaybeRunRound(key, s);
  }
}

void GpuServer::HandleInit(Shard* s, const KVMeta& req, const KVPairs<char>& data) {
  if (!s->initialized) {
    const bool f32 = req.cmd == kCmdInitF32;
    const void* src = data.vals.data();
    void* staged = nullptr;
    if (be_->on_device() && !data.vals.on_gpu()) {  // values came over a host path
      staged = be_->Alloc(data.vals.size());
      be_->Upload(staged, src, data.vals.size());
      src = staged;
    }
    be_->Decode(s->master, src, s->n, f32 ? PS_GRAD_F32 : PS_GRAD_BF16);
    if (staged) {
      be_->Sync();
      be_->Free(staged);
    }
    s->initialized = true;
    s->no_weight_decay = (req.option & kInitNoWeightDecay) != 0;
    if (req.option & kInitRowSparse) MakeRowSparse(s, (req.option >> 8) & 0x7fffff);
  }
  server_->Response(req);
}

void GpuServer::HandleGrad(Shard* s, const KVMeta& req, const KVPairs<char>& data) {
  const int rank = Postoffice::IDtoRank(req.sender);
  CHECK_LT(rank, cfg_.num_workers);
  CHECK(!s->pushed[rank]) << "worker " << rank << " pushed key " << req.key
                          << " twice in one round";
  int fmt = PS_GRAD_BF16;
  const void* slot;
  if (req.cmd == kCmdGradRows) {
    CHECK(s->dim > 0) << "key " << req.key << " is a dense shard: it takes kCmdGrad pushes, not kCmdGradRows";
    CHECK_EQ(req.codec, (int)kCodecRaw) << "kCmdGradRows payloads are encoded by the worker (codec raw)";
    CHECK_NE(req.mem.region, kSymmetricRegion) << "row-sparse gradients are not reduced in the switch";
    const int row_format = req.option & 3;
    const size_t R = static_cast<uint32_t>(req.option) >> 2;
    CHECK(row_format == PS_GRAD_F32 || row_format == PS_GRAD_BF16 || row_format == PS_GRAD_FP8BLOCK)
        << "kCmdGradRows: unknown row format " << row_format;
    CHECK(row_format != PS_GRAD_FP8BLOCK || s->dim % 32 == 0)
        << "kCmdGradRows: fp8 rows need a row width that is a multiple of 32, the shard has " << s->dim;
    const size_t e = R * s->dim;
    const size_t need = (R + 3) / 4 * 16 +
                        (row_format == PS_GRAD_F32 ? 4 * e : row_format == PS_GRAD_BF16 ? 2 * e : e + e / 32);
    CHECK_GE(data.vals.size(), need) << "kCmdGradRows: " << R << " rows need " << need << " bytes";
    s->num_rows[rank] = static_cast<uint32_t>(R);
    fmt = row_format;
  } else {
    CHECK_EQ(s->dim, 0) << "key " << req.key
                        << " is a row-sparse shard: it takes kCmdGradRows pushes only";
  }
  if (req.mem.region == kSymmetricRegion) {
    // staged in the worker's symmetric gradient buffer: read later through the multicast address
    CHECK(mc_grad_base_ != nullptr) << "symmetric push but SetSymmetricGrads was never called";
    CHECK_EQ(FormatOf(req, PS_GRAD_BF16), (int)PS_GRAD_BF16) << "in-switch reduction adds bf16 values";
    CHECK_LE(req.mem.offset + s->n * 2, symm_grad_bytes_);
    CHECK_EQ(req.mem.offset % 16, (uint64_t)0);
    fmt = PS_GRAD_MC_BF16;
    slot = static_cast<const char*>(mc_grad_base_) + req.mem.offset;
  } else {
    slot = data.vals.data();
    if (be_->on_device() && !data.vals.on_gpu()) {
      // the gradient arrived in host memory: its worker sits on another host (the one-sided van sent a
      // frame, staged through the host over there) or the transport is host-only. Upload it into a
      // per-rank device buffer on the update stream; the round's kernel runs behind it.
      const size_t bytes = data.vals.size();
      if (s->staged.size() < static_cast<size_t>(cfg_.num_workers)) {
        s->staged.resize(static_cast<size_t>(cfg_.num_workers), nullptr);
        s->staged_cap.resize(static_cast<size_t>(cfg_.num_workers), 0);
      }
      if (s->staged_cap[rank] < bytes) {
        if (s->staged[rank]) {
          be_->Sync();  // (an earlier round may still read it)
          be_->Free(s->staged[rank]);
        }
        s->staged[rank] = be_->Alloc(bytes + 16);
        s->staged_cap[rank] = bytes;
      }
      be_->Upload(s->staged[rank], data.vals.data(), bytes);
      slot = s->staged[rank];
    } else if (!be_->on_device()) {
      CHECK(!data.vals.on_gpu()) << "this server keeps its shards in host memory";
      s->slot_refs[rank] = data.vals;  // a two-sided payload lives in a pooled receive buffer
    }
    if (req.cmd != kCmdGradRows) fmt = FormatOf(req, cfg_.raw_grad_format);
  }
  if (s->num_pushed == 0) s->grad_format = fmt;
  CHECK_EQ(s->grad_format, fmt) << "workers disagree on the gradient wire format";
  if (fmt == PS_GRAD_MC_BF16 && s->num_pushed > 0) {
    for (int w = 0; w < cfg_.num_workers; ++w) {
      if (s->pushed[w]) CHECK(s->slots[w] == slot) << "workers disagree on the symmetric offset";
    }
  }
  s->slots[rank] = slot;
  s->pushed[rank] = 1;
  ++s->num_pushed;
  if (cfg_.async_updates) {
    CHECK_NE(fmt, (int)PS_GRAD_MC_BF16) << "in-switch reduction is a synchronous-round feature";
    s->grad_format = fmt;
    ApplyOnArrival(s, rank);
    if (req.pull) return;  // answered by the pull half
    if (be_->on_device()) {
      // ack only after the update has consumed the slot (descriptor gated on this stream)
      SendOpts after_update;
      after_update.codec = kCodecPlaced;
      KVPairs<char> none;
      server_->Response(req, none, after_update);
      return;
    }
  }
  if (req.pull) return;  // fused push-pull: the pull reply is the only answer
  // the payload already sits in its slot: the push is complete for the worker
  server_->Response(req);
}

void GpuServer::HandlePull(Shard* s, const KVMeta& req, const KVPairs<char>& /*data*/) {
  const int rank = Postoffice::IDtoRank(req.sender);
  CHECK_LT(rank, cfg_.num_workers);
  if (!cfg_.async_updates && s->pushed[rank]) {
    s->waiting_pulls.push_back(req);  // wants the parameters *after* this round's update
  } else {
    ServePullFromLocal(req.key, s, req);
  }
}

void* GpuServer::WorkerDest(const KVMeta& pull) {
  if (!pull.mem.valid()) return nullptr;
  const int rank = Postoffice::IDtoRank(pull.sender);
  if (pull.mem.region == kSymmetricRegion) {
    if (peer_bases_.empty() || pull.mem.offset + pull.mem.bytes > symm_bytes_) return nullptr;
    return static_cast<char*>(peer_bases_[rank]) + pull.mem.offset;
  }
  const int instance_id = po_->GroupWorkerRankToInstanceID(rank, instance_idx_);
  return po_->van()->ResolvePeerMem(instance_id, pull.mem);
}

void GpuServer::ApplyOnArrival(Shard* s, int rank) {
  ps_update_args a;
  memset(&a, 0, sizeof(a));
  a.n = s->n;
  a.num_grads = 1;
  a.grad_format = s->grad_format;
  a.grads[0] = s->slots[rank];
  a.master = s->master;
  a.m = s->m;
  a.v = s->v;
  ps_opt_params o = cfg_.opt;
  if (s->no_weight_decay) o.weight_decay = 0.f;
  ++s->step;
  if (o.optimizer == PS_OPT_ADAMW) {
    o.bias_corr1 = 1.f - std::pow(o.beta1, static_cast<float>(s->step));
    o.bias_corr2 = 1.f - std::pow(o.beta2, static_cast<float>(s->step));
  }
  RunUpdate(s, a, o, rank);
  ++updates_;
  // the slot may be overwritten by this worker's next push as soon as it is acked: on the
  // device the ack is sent behind the update on the same stream, on the host Update is synchronous
  s->pushed[rank] = 0;
  s->slot_refs[rank] = SArray<char>();
  s->num_pushed = 0;
}

void GpuServer::MaybeRunRound(Key key, Shard* s) {
  if (cfg_.async_updates) return;
  const int W = cfg_.num_workers;
  if (s->num_pushed < W) return;
  if (cfg_.fuse_pull && static_cast<int>(s->waiting_pulls.size()) < W) return;
  NvtxRange nvtx("ps.server_round");

  ps_update_args a;
  memset(&a, 0, sizeof(a));
  a.n = s->n;
  a.num_grads = W;
  a.grad_format = s->grad_format;
  for (int w = 0; w < W; ++w) a.grads[w] = s->slots[w];
  if (s->grad_format == PS_GRAD_MC_BF16) {
    a.num_grads = 1;  // one stream: the switch returns the sum over all bound GPUs
    ++mc_reduce_;
  }
  a.master = s->master;
  a.m = s->m;
  a.v = s->v;
  a.num_outs = 0;  // no server-side bf16 copy: late pulls are cast from the fp32 master on demand
  std::vector<char> placed(s->waiting_pulls.size(), 0);
  // (a row shard writes its touched rows into every placed destination with unicast stores)
  bool all_symmetric = mc_base_ != nullptr && static_cast<int>(s->waiting_pulls.size()) == W && !s->dim;
  for (size_t i = 0; i < s->waiting_pulls.size(); ++i) {
    const KVMeta& pull = s->waiting_pulls[i];
    void* dst = WorkerDest(pull);
    if (dst && a.num_outs < PS_MAX_FANOUT && pull.mem.bytes >= s->n * 2 &&
        (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
      a.outs[a.num_outs++] = dst;
      placed[i] = 1;
    }
    all_symmetric = all_symmetric && placed[i] && pull.mem.region == kSymmetricRegion &&
                    pull.mem.offset == s->waiting_pulls[0].mem.offset;
  }
  a.body_outs = a.num_outs;
  if (all_symmetric) {
    // every worker wants this shard at the same symmetric offset: one multicast store
    // stream replaces the W unicast streams (outs[1..] only serve the ragged tail)
    a.mc_out = static_cast<char*>(mc_base_) + s->waiting_pulls[0].mem.offset;
    a.body_outs = 0;
    ++mcast_;
  }
  ps_opt_params o = cfg_.opt;
  if (s->no_weight_decay) o.weight_decay = 0.f;
  ++s->step;
  if (o.optimizer == PS_OPT_ADAMW) {
    o.bias_corr1 = 1.f - std::pow(o.beta1, static_cast<float>(s->step));
    o.bias_corr2 = 1.f - std::pow(o.beta2, static_cast<float>(s->step));
  }
  RunUpdate(s, a, o, 0);
  ++updates_;
  if (a.num_outs > 0) ++fused_;

  SendOpts placed_opts;
  placed_opts.codec = kCodecPlaced;
  for (size_t i = 0; i < s->waiting_pulls.size(); ++i) {
    const KVMeta& pull = s->waiting_pulls[i];
    if (placed[i]) {
      KVPairs<char> res;
      res.keys = OneKey(key);
      // the values are already in the worker's buffer; `vals` only conveys their size
      res.vals = SArray<char>(reinterpret_cast<char*>(s->master), s->n * 2, GPU, dev_, GPU, dev_);
      res.lens = OneLen(s->n * 2);
      server_->Response(pull, res, placed_opts);
    } else {
      ServePullFromLocal(key, s, pull);
    }
  }
  s->waiting_pulls.clear();
  std::fill(s->pushed.begin(), s->pushed.end(), 0);
  for (auto& ref : s->slot_refs) ref = SArray<char>();
  s->num_pushed = 0;
}

void GpuServer::ServePullFromLocal(Key key, Shard* s, const KVMeta& req) {
  KVPairs<char> res;
  res.keys = OneKey(key);
  res.lens = OneLen(s->n * 2);
  const DeviceType where = be_->on_device() ? GPU : CPU;
  const int where_id = be_->on_device() ? dev_ : 0;
  if (void* dst = WorkerDest(req)) {
    // cast fp32 master -> bf16 straight into the worker's buffer (peer HBM / shared memory);
    // on the device this runs on the update stream, so it is ordered after any update
    CHECK_GE(req.mem.bytes, s->n * 2) << "pull destination smaller than the shard";
    be_->Copy(dst, s->master, s->n * 4, PS_CODEC_F32_TO_BF16, 1.f, cfg_.max_ctas);
    res.vals = SArray<char>(reinterpret_cast<char*>(s->master), s->n * 2, where, where_id, where, where_id);
    SendOpts placed;
    placed.codec = kCodecPlaced;
    server_->Response(req, res, placed);
    return;
  }
  CHECK(!req.mem.valid()) << "pull destination region unknown to this server";
  if (!be_->on_device()) {  // host shards, two-sided requester: cast into the reply buffer
    SArray<char> host(s->n * 2);
    be_->Copy(host.data(), s->master, s->n * 4, PS_CODEC_F32_TO_BF16, 1.f, cfg_.max_ctas);
    res.vals = host;
    server_->Response(req, res);
    return;
  }
  // device shards, two-sided requester: cast into a scratch buffer ...
  void* scratch = be_->Alloc(s->n * 2 + 16);
  be_->Copy(scratch, s->master, s->n * 4, PS_CODEC_F32_TO_BF16, 1.f, cfg_.max_ctas);
  if (po_->van()->GetType() == "nccl") {
    // ... which the nccl van sends from device memory (it orders the send behind this stream)
    Backend* be = be_.get();
    SArray<char> dvals;
    dvals.reset(static_cast<char*>(scratch), s->n * 2,
                [be](char* p) {
                  be->Bind();
                  be->Free(p);
                },
                GPU, dev_, GPU, dev_);
    res.vals = dvals;
    server_->Response(req, res);
    return;
  }
  // ... or, for a host-only transport (TCP), stage it through host memory
  SArray<char> host(s->n * 2);
  be_->Download(host.data(), scratch, s->n * 2);
  be_->Free(scratch);
  res.vals = host;
  server_->Response(req, res);
}

bool GpuServer::ReadMaster(Key key, std::vector<float>* out) {
  std::lock_guard<std::mutex> lk(mu_);
  auto it = shards_.find(key);
  if (it == shards_.end()) return false;
  be_->Bind();
  out->resize(it->second.n);
  be_->Download(out->data(), it->second.master, it->second.n * 4);
  return true;
}

namespace {
struct CkptHeader {
  char magic[8];
  uint64_t num_keys;
};
struct CkptEntry {
  uint64_t key;
  uint64_t n;
  int32_t step;
  int32_t initialized;
};
}  // namespace

bool GpuServer::SaveCheckpoint(const std::string& path) {
  std::lock_guard<std::mutex> lk(mu_);
  be_->Bind();
  be_->Sync();
  FILE* f = fopen(path.c_str(), "wb");
  if (!f) return false;
  CkptHeader h;
  memcpy(h.magic, "PSB2CKPT", 8);
  h.num_keys = shards_.size();
  bool ok = fwrite(&h, sizeof(h), 1, f) == 1;
  std::vector<float> buf;
  for (auto& kv : shards_) {
    const Shard& s = kv.second;
    // bit 0 initialized, bit 1 no weight decay, bit 2 row-sparse with the row width in bits 8..30
    CkptEntry e{kv.first, s.n, s.step,
                (s.initialized ? 1 : 0) | (s.no_weight_decay ? 2 : 0) | (s.dim ? 4 | (s.dim << 8) : 0)};
    ok = ok && fwrite(&e, sizeof(e), 1, f) == 1;
    buf.resize(s.n);
    for (float* src : {s.master, s.m, s.v}) {
      be_->Download(buf.data(), src, s.n * 4);
      ok = ok && fwrite(buf.data(), 4, s.n, f) == s.n;
    }
  }
  fclose(f);
  return ok;
}

bool GpuServer::LoadCheckpoint(const std::string& path) {
  std::lock_guard<std::mutex> lk(mu_);
  be_->Bind();
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) return false;
  CkptHeader h;
  bool ok = fread(&h, sizeof(h), 1, f) == 1 && memcmp(h.magic, "PSB2CKPT", 8) == 0;
  std::vector<float> buf;
  for (uint64_t i = 0; ok && i < h.num_keys; ++i) {
    CkptEntry e;
    ok = fread(&e, sizeof(e), 1, f) == 1;
    if (!ok) break;
    Shard* s = GetShard(e.key, e.n);
    s->step = e.step;
    s->initialized = (e.initialized & 1) != 0;
    s->no_weight_decay = (e.initialized & 2) != 0;
    const int dim = (e.initialized & 4) ? (e.initialized >> 8) & 0x7fffff : 0;
    if (dim != s->dim) {
      CHECK_EQ(s->dim, 0) << "checkpoint: key " << e.key << " has rows of " << dim << ", this server " << s->dim;
      MakeRowSparse(s, dim);  // (its scratch is not saved: a fresh one is empty)
    }
    buf.resize(e.n);
    for (float* dst : {s->master, s->m, s->v}) {
      ok = ok && fread(buf.data(), 4, e.n, f) == e.n;
      if (ok) be_->Upload(dst, buf.data(), e.n * 4);
    }
  }
  be_->Sync();
  fclose(f);
  return ok;
}

}  // namespace ps
