/**
 * \file bindings.cc
 * \brief Python / PyTorch binding of the native parameter-server runtime.
 *
 * The reference has no Python API (BytePS, its consumer, owns the torch plugin);
 * this is new scope (SURVEY §0). The binding is deliberately thin: tensors are
 * wrapped as zero-copy SArrays (placement taken from tensor.device, lifetime
 * pinned by capturing the tensor in the SArray deleter), and every call maps 1:1
 * onto the C++ API — KVWorker::ZPush/ZPull/Wait, KVServer handlers, GpuServer,
 * Postoffice barriers. CUDA work is never synchronised here: a push takes an
 * event recorded on the caller's current stream and hands it to the van's copy
 * kernel (SendOpts::wait_event).
 */
#include <torch/extension.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>

#include <cuda_runtime.h>

#include <atomic>
#include <mutex>
#include <unordered_map>

#include "kernels/model_kernels.h"
#include "kernels/host_kernels.h"
#include "kernels/ps_kernels.h"
#include "ps/ps.h"
#include "ps/simple_app.h"
#include "server/gpu_server.h"
#include "van/mem_domain.h"

namespace py = pybind11;
using namespace ps;

namespace {

bool CudaUsable() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return n > 0;
}

/*! \brief zero-copy byte view of a contiguous tensor; the tensor lives as long as the view */
SArray<char> ViewOf(const torch::Tensor& t) {
  TORCH_CHECK(t.is_contiguous(), "pslite: tensors must be contiguous");
  SArray<char> a;
  torch::Tensor keep = t;
  const bool gpu = t.is_cuda();
  const int dev = gpu ? t.get_device() : 0;
  a.reset(static_cast<char*>(t.data_ptr()), static_cast<size_t>(t.nbytes()),
          [keep](char*) mutable { keep.reset(); }, gpu ? GPU : CPU, dev, gpu ? GPU : CPU, dev);
  return a;
}

SArray<Key> OneKey(uint64_t k) {
  SArray<Key> a(1);
  a[0] = static_cast<Key>(k);
  return a;
}
SArray<int> OneLen(size_t n) {
  SArray<int> a(1);
  a[0] = static_cast<int>(std::min<size_t>(n, 0x7fffffff));
  return a;
}

/*! \brief cudaEvent recorded on the calling thread's current stream of `dev` */
cudaEvent_t RecordOnCurrentStream(int dev) {
  cudaEvent_t ev;
  TORCH_CHECK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) == cudaSuccess);
  cudaStream_t cur = at::cuda::getCurrentCUDAStream(dev).stream();
  TORCH_CHECK(cudaEventRecord(ev, cur) == cudaSuccess);
  return ev;
}

class PyKVWorker {
 public:
  PyKVWorker(int app_id, int customer_id, int instance_idx)
      : kv_(new KVWorker<char>(app_id, customer_id, instance_idx)), instance_(instance_idx) {
    // every completion callback of this class only releases references: safe on the receive thread
    kv_->set_inline_dispatch(GetEnv("PS_WORKER_INLINE", 1) != 0);
  }

  /*! \brief encode "the idx-th key owned by server `server`" like the benchmarks do */
  uint64_t server_key(int server, uint64_t idx) {
    const auto& ranges = Postoffice::GetWorker()->GetServerKeyRanges();
    TORCH_CHECK(server >= 0 && server < static_cast<int>(ranges.size()), "bad server rank");
    return ranges[server].begin() + idx;
  }

  int push(uint64_t key, const torch::Tensor& t, int cmd, int codec, float scale,
           bool order_after_current_stream, int64_t symm_offset, uint64_t symm_base, int option,
           uint64_t slot_bytes) {
    SArray<char> vals = ViewOf(t);
    SendOpts opts;
    opts.codec = codec;
    opts.scale = scale;
    opts.option = option;
    opts.slot_bytes = slot_bytes;
    if (symm_offset >= 0) {
      // stage the encoded gradient in this worker's symmetric buffer; the server reads the
      // sum of all workers' copies through the multicast address (multimem.ld_reduce)
      TORCH_CHECK(symm_base != 0, "symmetric push needs the local base address of the buffer");
      opts.dest_mem.region = kSymmetricRegion;
      opts.dest_mem.offset = static_cast<uint64_t>(symm_offset);
      opts.dest_mem.bytes = WireBytes(codec, vals.size());
      opts.stage = reinterpret_cast<void*>(symm_base + static_cast<uint64_t>(symm_offset));
    }
    cudaEvent_t ev = nullptr;
    if (t.is_cuda() && order_after_current_stream) {
      ev = RecordOnCurrentStream(t.get_device());
      opts.wait_event = ev;
    }
    py::gil_scoped_release nogil;
    // the event must outlive the copy that waits on it: destroy it on completion
    auto cb = ev ? KVWorker<char>::Callback([ev]() { cudaEventDestroy(ev); })
                 : KVWorker<char>::Callback();
    return kv_->ZPush(OneKey(key), vals, OneLen(vals.size()), cmd, cb, opts);
  }

  int pull(uint64_t key, torch::Tensor t, int cmd, int64_t symm_offset) {
    // the destination view must stay alive until the response lands: own it here
    auto* dst = new SArray<char>(ViewOf(t));
    auto* len = new SArray<int>(OneLen(dst->size()));
    SendOpts opts;
    if (symm_offset >= 0) {  // destination = offset inside the job-wide symmetric buffer
      opts.dest_mem.region = kSymmetricRegion;
      opts.dest_mem.offset = static_cast<uint64_t>(symm_offset);
      opts.dest_mem.bytes = dst->size();
    }
    py::gil_scoped_release nogil;
    return kv_->ZPull(OneKey(key), dst, len, cmd, [dst, len]() {
      delete dst;
      delete len;
    }, opts);
  }

  /*! \brief fused push + pull of one key: push `t`, receive the server's values in `out` */
  int push_pull(uint64_t key, const torch::Tensor& t, torch::Tensor out, int cmd, int codec, float scale,
                bool order_after_current_stream, int64_t pull_symm_offset) {
    SArray<char> vals = ViewOf(t);
    auto* dst = new SArray<char>(ViewOf(out));
    auto* len = new SArray<int>(OneLen(dst->size()));
    SendOpts opts;
    opts.codec = codec;
    opts.scale = scale;
    if (pull_symm_offset >= 0) {
      opts.pull_dest_mem.region = kSymmetricRegion;
      opts.pull_dest_mem.offset = static_cast<uint64_t>(pull_symm_offset);
      opts.pull_dest_mem.bytes = dst->size();
    }
    cudaEvent_t ev = nullptr;
    if (t.is_cuda() && order_after_current_stream) {
      ev = RecordOnCurrentStream(t.get_device());
      opts.wait_event = ev;
    }
    py::gil_scoped_release nogil;
    return kv_->ZPushPull(OneKey(key), vals, dst, len, cmd, [dst, len, ev]() {
      delete dst;
      delete len;
      if (ev) cudaEventDestroy(ev);
    }, opts);
  }

  void wait(int ts) {
    py::gil_scoped_release nogil;
    kv_->Wait(ts);
  }

  /*! \brief one push + one pull per (key, tensor) with a single Python call; returns all timestamps */
  std::vector<int> push_pull_batch(const std::vector<uint64_t>& keys,
                                   const std::vector<torch::Tensor>& tensors, int cmd, int codec,
                                   float scale, bool order_after_current_stream, bool do_push,
                                   bool do_pull, bool fused) {
    TORCH_CHECK(keys.size() == tensors.size(), "keys / tensors length mismatch");
    std::vector<SArray<char>> views;
    views.reserve(keys.size());
    for (const auto& t : tensors) views.push_back(ViewOf(t));
    cudaEvent_t ev = nullptr;
    if (do_push && order_after_current_stream && !tensors.empty() && tensors[0].is_cuda()) {
      ev = RecordOnCurrentStream(tensors[0].get_device());
    }
    py::gil_scoped_release nogil;
    // with PS_COALESCE_LAUNCHES all pushes of this call share kernel launches and one event
    Van::CorkScope cork(Postoffice::GetWorker(instance_)->van());
    std::vector<int> ts;
    ts.reserve(keys.size() * 2);
    auto remaining = std::make_shared<std::atomic<int>>(do_push ? static_cast<int>(keys.size()) : 0);
    for (size_t i = 0; i < keys.size(); ++i) {
      if (fused && do_push && do_pull) {
        // one ZPushPull per key: the request carries the push, its single reply the pulled values
        SendOpts opts;
        opts.codec = codec;
        opts.scale = scale;
        opts.wait_event = ev;
        auto* dst = new SArray<char>(views[i]);
        auto* len = new SArray<int>(OneLen(dst->size()));
        ts.push_back(kv_->ZPushPull(OneKey(keys[i]), views[i], dst, len, cmd, [dst, len, ev, remaining]() {
          delete dst;
          delete len;
          if (ev && remaining->fetch_sub(1) == 1) cudaEventDestroy(ev);
        }, opts));
        continue;
      }
      if (do_push) {
        SendOpts opts;
        opts.codec = codec;
        opts.scale = scale;
        opts.wait_event = ev;
        auto cb = ev ? KVWorker<char>::Callback([ev, remaining]() {
          if (remaining->fetch_sub(1) == 1) cudaEventDestroy(ev);
        }) : KVWorker<char>::Callback();
        ts.push_back(kv_->ZPush(OneKey(keys[i]), views[i], OneLen(views[i].size()), cmd, cb, opts));
      }
      if (do_pull) {
        auto* dst = new SArray<char>(views[i]);
        auto* len = new SArray<int>(OneLen(dst->size()));
        ts.push_back(kv_->ZPull(OneKey(keys[i]), dst, len, cmd, [dst, len]() {
          delete dst;
          delete len;
        }));
      }
    }
    return ts;
  }

  void wait_all(const std::vector<int>& ts) {
    py::gil_scoped_release nogil;
    for (int t : ts) kv_->Wait(t);
  }

  /*!
   * \brief a whole staged round in one call: for every key copy this step's input from (pinned) host
   *        memory into its device tensor, push it, pull the result back into the same tensor and copy
   *        that to host memory. Software-pipelined over the keys on two streams: the H2D copy of key
   *        k+1, the push + pull of key k and the D2H copy of key k-1 overlap (PCIe is full duplex);
   *        a push waits for the event of its own H2D copy only. Returns when `host_out` is complete.
   *        On a GPU-less build of the job (shm van) the "device" tensors are host tensors and the
   *        copies are plain memcpys: same control flow.
   */
  void staged_push_pull(const std::vector<uint64_t>& keys, std::vector<torch::Tensor> dev,
                        const std::vector<torch::Tensor>& host_in, std::vector<torch::Tensor> host_out, int cmd,
                        int codec, float scale) {
    const size_t n = keys.size();
    TORCH_CHECK(dev.size() == n && host_in.size() == n && host_out.size() == n, "list lengths differ");
    if (n == 0) return;
    const bool cuda = dev[0].is_cuda();
    for (size_t i = 0; i < n; ++i) {
      TORCH_CHECK(dev[i].is_cuda() == cuda && !host_in[i].is_cuda() && !host_out[i].is_cuda(),
                  "dev tensors on one device kind, host_in / host_out in host memory");
      TORCH_CHECK(dev[i].nbytes() == host_in[i].nbytes() && dev[i].nbytes() == host_out[i].nbytes(),
                  "size mismatch at position ", i);
    }
    py::gil_scoped_release nogil;
    at::NoGradGuard no_grad;
    std::vector<int> pushes(n), pulls(n);
    c10::optional<c10::cuda::CUDAStream> h2d, d2h;
    if (cuda) {
      const auto idx = static_cast<c10::DeviceIndex>(dev[0].get_device());
      h2d = c10::cuda::getStreamFromPool(false, idx);
      d2h = c10::cuda::getStreamFromPool(false, idx);
      // the device tensors may have been written on the caller's stream
      cudaEvent_t ready = RecordOnCurrentStream(idx);
      cudaStreamWaitEvent(h2d->stream(), ready, 0);
      cudaEventDestroy(ready);
    }
    {
      c10::optional<c10::cuda::CUDAStreamGuard> guard;
      if (cuda) guard.emplace(*h2d);
      for (size_t i = 0; i < n; ++i) {
        dev[i].copy_(host_in[i], /*non_blocking=*/true);
        SArray<char> view = ViewOf(dev[i]);
        SendOpts opts;
        opts.codec = codec;
        opts.scale = scale;
        cudaEvent_t ev = cuda ? RecordOnCurrentStream(dev[i].get_device()) : nullptr;
        opts.wait_event = ev;
        auto cb = ev ? KVWorker<char>::Callback([ev]() { cudaEventDestroy(ev); }) : KVWorker<char>::Callback();
        pushes[i] = kv_->ZPush(OneKey(keys[i]), view, OneLen(view.size()), cmd, cb, opts);
        auto* dst = new SArray<char>(view);
        auto* len = new SArray<int>(OneLen(dst->size()));
        pulls[i] = kv_->ZPull(OneKey(keys[i]), dst, len, cmd, [dst, len]() {
          delete dst;
          delete len;
        });
      }
    }
    {
      c10::optional<c10::cuda::CUDAStreamGuard> guard;
      if (cuda) guard.emplace(*d2h);
      for (size_t i = 0; i < n; ++i) {
        kv_->Wait(pulls[i]);  // the server's copy into dev[i] has completed
        host_out[i].copy_(dev[i], /*non_blocking=*/true);
      }
    }
    for (size_t i = 0; i < n; ++i) kv_->Wait(pushes[i]);
    if (cuda) d2h->synchronize();
  }

 private:
  std::unique_ptr<KVWorker<char>> kv_;
  int instance_ = 0;
};

/*! \brief a KVServer whose handler is a Python callable (tests, small CPU models) */
class PyKVServer {
 public:
  explicit PyKVServer(int app_id) : kv_(new KVServer<char>(app_id)) {}
  ~PyKVServer() {
    py::gil_scoped_release nogil;
    kv_.reset();
  }

  /*! \brief handler(meta: dict, key: int, vals: uint8 tensor view) -> None; must call response() */
  void set_request_handle(py::function fn) {
    handler_ = fn;
    kv_->set_request_handle([this](const KVMeta& m, const KVPairs<char>& d, KVServer<char>*) {
      py::gil_scoped_acquire gil;
      const int id = next_id_++;
      pending_[id] = m;
      py::dict meta;
      meta["id"] = id;
      meta["push"] = m.push;
      meta["cmd"] = m.cmd;
      meta["sender"] = m.sender;
      meta["sender_rank"] = Postoffice::IDtoRank(m.sender);
      meta["timestamp"] = m.timestamp;
      meta["key"] = static_cast<uint64_t>(d.keys.size() ? d.keys[0] : m.key);
      meta["val_len"] = m.val_len;
      meta["codec"] = m.codec;
      meta["scale"] = m.scale;
      py::object vals = py::none();
      if (d.vals.size()) {
        SArray<char> keep = d.vals;
        auto opts = torch::TensorOptions().dtype(torch::kUInt8);
        if (keep.on_gpu()) opts = opts.device(torch::kCUDA, keep.src_device_id_);
        vals = py::cast(torch::from_blob(keep.data(), {static_cast<int64_t>(keep.size())},
                                         [keep](void*) mutable { keep.clear(); }, opts));
      }
      handler_(meta, meta["key"], vals);
    });
  }

  void response(int id, py::object vals) {
    KVMeta m;
    {
      auto it = pending_.find(id);
      TORCH_CHECK(it != pending_.end(), "unknown / already answered request id");
      m = it->second;
      pending_.erase(it);
    }
    KVPairs<char> res;
    if (!vals.is_none()) {
      torch::Tensor t = vals.cast<torch::Tensor>();
      res.keys = OneKey(m.key);
      res.vals = ViewOf(t);
      res.lens = OneLen(res.vals.size());
    }
    py::gil_scoped_release nogil;
    kv_->Response(m, res);
  }

 private:
  std::unique_ptr<KVServer<char>> kv_;
  py::function handler_;
  std::unordered_map<int, KVMeta> pending_;  // guarded by the GIL
  int next_id_ = 0;
};

/*!
 * \brief SimpleApp from Python: small control messages (an int head and a byte-string body) between
 *        any two nodes, with handlers written in Python. `role` picks the postoffice of a joint process
 *        ("worker" / "server"); ids and groups are the reference's (kScheduler 1, kServerGroup 2,
 *        kWorkerGroup 4, or a node id). As in the reference, a server (and the scheduler) finds the
 *        customer of an incoming request by its APP id: create server-side apps with customer_id == app_id.
 */
class PySimpleApp {
 public:
  PySimpleApp(int app_id, int customer_id, const std::string& role) {
    Postoffice* po = role == "server" ? Postoffice::GetServer() : (role == "worker" ? Postoffice::GetWorker()
                                                                                      : Postoffice::Get());
    app_.reset(new SimpleApp(app_id, customer_id, po));
  }
  ~PySimpleApp() {
    py::gil_scoped_release nogil;
    app_.reset();
  }
  int request(int head, const std::string& body, int recv_id) {
    py::gil_scoped_release nogil;
    return app_->Request(head, body, recv_id);
  }
  void wait(int timestamp) {
    py::gil_scoped_release nogil;
    app_->Wait(timestamp);
  }
  /*! \brief handler(head, body: bytes, sender, timestamp) -> None | bytes | str (the body of the reply) */
  void set_request_handle(py::function fn) {
    on_request_ = fn;
    app_->set_request_handle([this](const SimpleData& req, SimpleApp* app) {
      std::string reply;
      {
        py::gil_scoped_acquire gil;
        py::object r = on_request_(req.head, py::bytes(req.body), req.sender, req.timestamp);
        if (!r.is_none()) reply = r.cast<std::string>();
      }
      app->Response(req, reply);
    });
  }
  /*! \brief handler(head, body: bytes, sender, timestamp) for every response that arrives */
  void set_response_handle(py::function fn) {
    on_response_ = fn;
    app_->set_response_handle([this](const SimpleData& res, SimpleApp*) {
      py::gil_scoped_acquire gil;
      on_response_(res.head, py::bytes(res.body), res.sender, res.timestamp);
    });
  }

 private:
  std::unique_ptr<SimpleApp> app_;
  py::function on_request_, on_response_;
};

/*!
 * \brief native twin of test_benchmark's server: the first push of a key becomes its
 *        store (the landing slot itself), pulls are answered from the store.
 */
class PyBenchServer {
 public:
  explicit PyBenchServer(int app_id) : kv_(new KVServer<char>(app_id)) {
    kv_->set_request_handle([this](const KVMeta& m, const KVPairs<char>& d, KVServer<char>* s) {
      const uint64_t key = d.keys.size() ? d.keys[0] : m.key;
      if (m.push) {
        {
          std::lock_guard<std::mutex> lk(mu_);
          auto it = store_.find(key);
          if (it == store_.end()) {
            KVPairs<char>& slot = store_[key];
            slot.keys.CopyFrom(d.keys);
            slot.lens.CopyFrom(d.lens);
            slot.vals = d.vals;
          } else if (it->second.vals.data() != d.vals.data()) {
            // a one-sided push lands in the same slot every time (nothing to do); a push that travelled
            // in a frame (TCP van, peer on another host) arrives in a fresh buffer: the newest one is the value
            it->second.vals = d.vals;
          }
        }
        ++pushes_;
        if (m.pull) {  // fused push-pull: reply with the stored values instead of an ack
          KVPairs<char> res;
          {
            std::lock_guard<std::mutex> lk(mu_);
            res = store_[key];
          }
          ++pulls_;
          s->Response(m, res);
        } else {
          s->Response(m);
        }
      } else {
        KVPairs<char> res;
        {
          std::lock_guard<std::mutex> lk(mu_);
          auto it = store_.find(key);
          CHECK(it != store_.end()) << "pull of a key that was never pushed: " << key;
          res = it->second;
        }
        ++pulls_;
        s->Response(m, res);
      }
    });
    // the handler never waits for the network; with launch coalescing the customer thread batches instead
    kv_->set_inline_dispatch(GetEnv("PS_SERVER_INLINE", 1) != 0 && GetEnv("PS_COALESCE_LAUNCHES", 0) == 0);
  }
  ~PyBenchServer() {
    py::gil_scoped_release nogil;
    kv_.reset();
  }
  uint64_t pushes() const { return pushes_.load(); }
  uint64_t pulls() const { return pulls_.load(); }

 private:
  std::unique_ptr<KVServer<char>> kv_;
  std::mutex mu_;
  std::unordered_map<uint64_t, KVPairs<char>> store_;
  std::atomic<uint64_t> pushes_{0}, pulls_{0};
};

class PyGpuServer {
 public:
  PyGpuServer(int app_id, int num_workers, const std::string& optimizer, float lr, float beta1,
              float beta2, float eps, float weight_decay, float grad_scale, bool fuse_pull,
              const std::string& raw_grad, int max_ctas, bool async_updates) {
    GpuServerConfig c;
    c.num_workers = num_workers;
    c.opt.optimizer = optimizer == "sgd" ? PS_OPT_SGD : PS_OPT_ADAMW;
    c.opt.lr = lr;
    c.opt.beta1 = beta1;
    c.opt.beta2 = beta2;
    c.opt.eps = eps;
    c.opt.weight_decay = weight_decay;
    c.opt.grad_scale = grad_scale;
    c.fuse_pull = fuse_pull;
    c.async_updates = async_updates;
    c.raw_grad_format = raw_grad == "f32" ? PS_GRAD_F32 : PS_GRAD_BF16;
    c.max_ctas = max_ctas;
    impl_.reset(new GpuServer(app_id, c));
  }
  ~PyGpuServer() {
    py::gil_scoped_release nogil;
    impl_.reset();
  }
  void set_lr(float lr) { impl_->SetLearningRate(lr); }
  float lr() { return impl_->learning_rate(); }
  void set_symmetric(uint64_t mc_ptr, const std::vector<uint64_t>& peer_ptrs, uint64_t bytes) {
    std::vector<void*> peers;
    for (uint64_t p : peer_ptrs) peers.push_back(reinterpret_cast<void*>(p));
    impl_->SetSymmetricParams(reinterpret_cast<void*>(mc_ptr), peers, bytes);
  }
  void set_symmetric_grads(uint64_t mc_ptr, uint64_t bytes) {
    impl_->SetSymmetricGrads(reinterpret_cast<void*>(mc_ptr), bytes);
  }
  uint64_t num_switch_reductions() { return impl_->num_switch_reductions(); }
  uint64_t num_multicast_fanouts() { return impl_->num_multicast_fanouts(); }
  uint64_t num_updates() { return impl_->num_updates(); }
  bool on_device() { return impl_->on_device(); }
  uint64_t num_fused_fanouts() { return impl_->num_fused_fanouts(); }
  size_t num_keys() { return impl_->num_keys(); }
  size_t state_bytes() { return impl_->state_bytes(); }
  uint64_t num_bad_rows() {
    py::gil_scoped_release nogil;
    return impl_->num_bad_rows();
  }
  bool save(const std::string& path) {
    py::gil_scoped_release nogil;
    return impl_->SaveCheckpoint(path);
  }
  bool load(const std::string& path) {
    py::gil_scoped_release nogil;
    return impl_->LoadCheckpoint(path);
  }
  torch::Tensor read_master(uint64_t key) {
    std::vector<float> host;
    TORCH_CHECK(impl_->ReadMaster(static_cast<Key>(key), &host), "unknown key");
    return torch::from_blob(host.data(), {static_cast<int64_t>(host.size())}, torch::kFloat32).clone();
  }

 private:
  std::unique_ptr<GpuServer> impl_;
};

ps_stream_t CurrentStream(const torch::Tensor& t) {
  return reinterpret_cast<ps_stream_t>(at::cuda::getCurrentCUDAStream(t.get_device()).stream());
}

void CheckRc(int rc, const char* what) {
  TORCH_CHECK(rc == 0, what, " failed: ", cudaGetErrorString(static_cast<cudaError_t>(rc)));
}

/*! \brief bytes of a row-sparse gradient slot (ps_update_rows_args): ids padded to 16 B, then the values */
int64_t RowsSlotBytes(int64_t num_rows, int64_t dim, int grad_format) {
  const int64_t ids = (num_rows + 3) / 4 * 16, e = num_rows * dim;
  switch (grad_format) {
    case PS_GRAD_F32: return ids + 4 * e;
    case PS_GRAD_BF16: return ids + 2 * e;
    default: return ids + e + e / 32;  // fp8 block: dim % 32 == 0
  }
}

}  // namespace

PYBIND11_MODULE(_C, m) {
  m.doc() = "pslite_b200 native runtime";
  m.def("set_env", [](const std::string& k, const std::string& v) { Environment::Get()->set(k, v); });
  m.def("cuda_usable", &CudaUsable);
  m.def("start_ps", [](int customer_id, const std::string& role, int rank, bool do_barrier) {
    py::gil_scoped_release nogil;
    StartPS(customer_id, GetRole(role), rank, do_barrier);
  }, py::arg("customer_id") = 0, py::arg("role"), py::arg("rank") = -1, py::arg("do_barrier") = true);
  m.def("finalize", [](int customer_id, const std::string& role, bool do_barrier) {
    py::gil_scoped_release nogil;
    Finalize(customer_id, GetRole(role), do_barrier);
  }, py::arg("customer_id") = 0, py::arg("role"), py::arg("do_barrier") = true);
  m.def("reset", []() { Postoffice::Reset(); });
  m.def("num_workers", []() { return NumWorkers(); });
  m.def("num_servers", []() { return NumServers(); });
  m.def("worker_rank", []() { return Postoffice::GetWorker()->my_rank(); });
  m.def("server_rank", []() { return Postoffice::GetServer()->my_rank(); });
  m.def("barrier", [](int customer_id, int group, const std::string& as_role) {
    py::gil_scoped_release nogil;
    Postoffice* po = as_role == "server" ? Postoffice::GetServer()
                     : as_role == "scheduler" ? Postoffice::GetScheduler() : Postoffice::GetWorker();
    po->Barrier(customer_id, group);
  }, py::arg("customer_id") = 0, py::arg("group") = kWorkerGroup + kServerGroup,
     py::arg("as_role") = "worker");
  m.attr("SCHEDULER_GROUP") = static_cast<int>(kScheduler);
  m.attr("SERVER_GROUP") = static_cast<int>(kServerGroup);
  m.attr("WORKER_GROUP") = static_cast<int>(kWorkerGroup);
  m.attr("CODEC_RAW") = static_cast<int>(kCodecRaw);
  m.attr("CODEC_F32_TO_BF16") = static_cast<int>(kCodecF32ToBf16);
  m.attr("CODEC_BF16_SCALE") = static_cast<int>(kCodecBf16Scale);
  m.attr("CODEC_F32_TO_FP8BLOCK") = static_cast<int>(kCodecF32ToFp8Block);
  m.attr("CODEC_BF16_TO_FP8BLOCK") = static_cast<int>(kCodecBf16ToFp8Block);
  m.attr("CMD_GRAD") = static_cast<int>(kCmdGrad);
  m.attr("CMD_INIT_BF16") = static_cast<int>(kCmdInitBf16);
  m.attr("CMD_INIT_F32") = static_cast<int>(kCmdInitF32);
  m.attr("GRAD_F32") = static_cast<int>(PS_GRAD_F32);
  m.attr("GRAD_BF16") = static_cast<int>(PS_GRAD_BF16);
  m.attr("CMD_SET_LR") = static_cast<int>(kCmdSetLr);
  m.attr("INIT_NO_WEIGHT_DECAY") = static_cast<int>(kInitNoWeightDecay);
  m.attr("INIT_ROW_SPARSE") = static_cast<int>(kInitRowSparse);
  m.attr("CMD_GRAD_ROWS") = static_cast<int>(kCmdGradRows);
  m.attr("GRAD_FP8BLOCK") = static_cast<int>(PS_GRAD_FP8BLOCK);
  m.attr("GRAD_MC_BF16") = static_cast<int>(PS_GRAD_MC_BF16);

  m.def("dead_nodes", [](int timeout_s, const std::string& as_role) {
    // liveness as the scheduler sees it (PS_HEARTBEAT_INTERVAL must be set): ids of nodes that
    // have not reported for `timeout_s` seconds
    Postoffice* po = as_role == "scheduler" ? Postoffice::GetScheduler()
                     : as_role == "server"  ? Postoffice::GetServer() : Postoffice::GetWorker();
    TORCH_CHECK(po != nullptr, "no such role in this process");
    return po->GetDeadNodes(timeout_s);
  }, py::arg("timeout_s") = 60, py::arg("as_role") = "worker");
  m.def("wire_bytes", [](int codec, uint64_t src_bytes) { return WireBytes(codec, src_bytes); });
  m.def("kernel_launch_count", []() { return ps_kernel_launch_count(); });
  m.def("van_stats", [](const std::string& as_role) {
    Postoffice* po = as_role == "server" ? Postoffice::GetServer() : Postoffice::GetWorker();
    std::vector<std::pair<std::string, uint64_t>> kv;
    if (po && po->van()) po->van()->TransportStats(&kv);
    py::dict d;
    for (auto& e : kv) d[py::str(e.first)] = e.second;
    return d;
  }, py::arg("as_role") = "worker");
  m.def("van_bytes", []() {
    Van* v = Postoffice::Get()->van();
    return std::make_pair(v->send_bytes(), v->recv_bytes());
  });

  /*! \brief exportable memory of the worker van as a uint8 tensor (HBM on nvl, shm on shm) */
  m.def("alloc_exportable", [](int64_t nbytes, const std::string& as_role) {
    Postoffice* po = as_role == "server" ? Postoffice::GetServer() : Postoffice::GetWorker();
    Van* van = po->van();
    void* p = van->AllocExportable(static_cast<size_t>(nbytes));
    TORCH_CHECK(p, "allocation failed");
    auto opts = torch::TensorOptions().dtype(torch::kUInt8);
    const int dev = van->my_node().dev_id;
    if (van->GetType() == "nvl") opts = opts.device(torch::kCUDA, dev);
    return torch::from_blob(p, {nbytes}, [van](void* q) { van->FreeExportable(q); }, opts);
  }, py::arg("nbytes"), py::arg("as_role") = "worker");

  /*!
   * \brief collective over all worker / server processes: symmetric memory without torch's private
   *        API. Returns (local uint8 tensor, multicast address or 0, [address of every member's block
   *        as mapped here], my index, member count, [block of worker rank r], [block of server rank r]).
   */
  m.def("alloc_symmetric", [](const std::string& tag, int64_t nbytes, const std::string& as_role) {
    Postoffice* po = as_role == "server" ? Postoffice::GetServer() : Postoffice::GetWorker();
    TORCH_CHECK(po != nullptr && po->van() != nullptr, "the PS runtime is not started");
    Van* van = po->van();
    SymmetricBuffer sb;
    bool ok;
    {
      py::gil_scoped_release nogil;
      ok = van->AllocSymmetric(tag, static_cast<size_t>(nbytes), &sb);
    }
    TORCH_CHECK(ok, "AllocSymmetric('", tag, "') failed on the ", van->GetType(), " van");
    auto opts = torch::TensorOptions().dtype(torch::kUInt8);
    if (van->GetType() == "nvl") opts = opts.device(torch::kCUDA, van->my_node().dev_id);
    torch::Tensor local = torch::from_blob(sb.local, {static_cast<int64_t>(sb.bytes)}, [](void*) {}, opts);
    std::vector<uint64_t> peers;
    for (void* p : sb.peers) peers.push_back(reinterpret_cast<uint64_t>(p));
    // block of worker rank r / server rank r as mapped here (0 if that node is not a member)
    std::vector<uint64_t> worker_blocks, server_blocks;
    for (int r = 0; r < NumWorkers(); ++r) {
      const int m = sb.MemberOfNode(Postoffice::WorkerRankToID(r));
      worker_blocks.push_back(m >= 0 ? peers[static_cast<size_t>(m)] : 0);
    }
    for (int r = 0; r < NumServers(); ++r) {
      const int m = sb.MemberOfNode(Postoffice::ServerRankToID(r));
      server_blocks.push_back(m >= 0 ? peers[static_cast<size_t>(m)] : 0);
    }
    return py::make_tuple(local, reinterpret_cast<uint64_t>(sb.mc), peers, sb.index, sb.count, worker_blocks,
                          server_blocks);
  }, py::arg("tag"), py::arg("nbytes"), py::arg("as_role") = "worker");
  /*! \brief a uint8 view of `nbytes` at a raw address of this process (a peer mapping from alloc_symmetric) */
  m.def("tensor_at", [](uint64_t addr, int64_t nbytes, int cuda_device) {
    auto opts = torch::TensorOptions().dtype(torch::kUInt8);
    if (cuda_device >= 0) {
      // a peer mapping reports its OWNER's device: name that one (any device of the process can
      // still address the bytes — the mapping is in the unified address space)
      cudaPointerAttributes attr;
      if (cudaPointerGetAttributes(&attr, reinterpret_cast<void*>(addr)) == cudaSuccess &&
          (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged)) {
        cuda_device = attr.device;
      } else {
        cudaGetLastError();
      }
      opts = opts.device(torch::kCUDA, cuda_device);
    }
    return torch::from_blob(reinterpret_cast<void*>(addr), {nbytes}, [](void*) {}, opts);
  }, py::arg("addr"), py::arg("nbytes"), py::arg("cuda_device") = -1);

  /*! \brief copy `nbytes` at a raw address of this process (host or device, e.g. a peer mapping) into a CPU tensor */
  m.def("read_bytes", [](uint64_t addr, int64_t nbytes, bool device) {
    torch::Tensor out = torch::empty({nbytes}, torch::TensorOptions().dtype(torch::kUInt8));
    if (device) {
      // through the CURRENT device: that is the one the mapping was made accessible to
      TORCH_CHECK(cudaMemcpy(out.data_ptr(), reinterpret_cast<void*>(addr), static_cast<size_t>(nbytes),
                             cudaMemcpyDeviceToHost) == cudaSuccess, "cudaMemcpy from a mapped address failed");
    } else {
      memcpy(out.data_ptr(), reinterpret_cast<void*>(addr), static_cast<size_t>(nbytes));
    }
    return out;
  }, py::arg("addr"), py::arg("nbytes"), py::arg("device") = false);

  py::class_<PyKVWorker>(m, "KVWorker")
      .def(py::init<int, int, int>(), py::arg("app_id") = 0, py::arg("customer_id") = 0,
           py::arg("instance_idx") = 0)
      .def("server_key", &PyKVWorker::server_key)
      .def("push", &PyKVWorker::push, py::arg("key"), py::arg("tensor"), py::arg("cmd") = 0,
           py::arg("codec") = 0, py::arg("scale") = 1.0f,
           py::arg("order_after_current_stream") = true, py::arg("symm_offset") = -1,
           py::arg("symm_base") = 0, py::arg("option") = 0, py::arg("slot_bytes") = 0)
      .def("pull", &PyKVWorker::pull, py::arg("key"), py::arg("tensor"), py::arg("cmd") = 0,
           py::arg("symm_offset") = -1)
      .def("push_pull", &PyKVWorker::push_pull, py::arg("key"), py::arg("tensor"), py::arg("out"),
           py::arg("cmd") = 0, py::arg("codec") = 0, py::arg("scale") = 1.0f,
           py::arg("order_after_current_stream") = true, py::arg("pull_symm_offset") = -1)
      .def("wait", &PyKVWorker::wait)
      .def("wait_all", &PyKVWorker::wait_all)
      .def("push_pull_batch", &PyKVWorker::push_pull_batch, py::arg("keys"), py::arg("tensors"),
           py::arg("cmd") = 0, py::arg("codec") = 0, py::arg("scale") = 1.0f,
           py::arg("order_after_current_stream") = true, py::arg("push") = true,
           py::arg("pull") = true, py::arg("fused") = false)
      .def("staged_push_pull", &PyKVWorker::staged_push_pull, py::arg("keys"), py::arg("dev"),
           py::arg("host_in"), py::arg("host_out"), py::arg("cmd") = 0, py::arg("codec") = 0,
           py::arg("scale") = 1.0f);

  py::class_<PyKVServer>(m, "KVServer")
      .def(py::init<int>(), py::arg("app_id") = 0)
      .def("set_request_handle", &PyKVServer::set_request_handle)
      .def("response", &PyKVServer::response, py::arg("id"), py::arg("vals") = py::none());

  py::class_<PySimpleApp>(m, "SimpleApp")
      .def(py::init<int, int, const std::string&>(), py::arg("app_id") = 0, py::arg("customer_id") = 0,
           py::arg("role") = "")
      .def("request", &PySimpleApp::request, py::arg("head"), py::arg("body") = "", py::arg("recv_id") = 2)
      .def("wait", &PySimpleApp::wait)
      .def("set_request_handle", &PySimpleApp::set_request_handle)
      .def("set_response_handle", &PySimpleApp::set_response_handle);

  py::class_<PyBenchServer>(m, "BenchServer")
      .def(py::init<int>(), py::arg("app_id") = 0)
      .def("pushes", &PyBenchServer::pushes)
      .def("pulls", &PyBenchServer::pulls);

  py::class_<PyGpuServer>(m, "GpuServer")
      .def(py::init<int, int, const std::string&, float, float, float, float, float, float, bool,
                    const std::string&, int, bool>(),
           py::arg("app_id") = 0, py::arg("num_workers") = 1, py::arg("optimizer") = "adamw",
           py::arg("lr") = 1e-3f, py::arg("beta1") = 0.9f, py::arg("beta2") = 0.95f,
           py::arg("eps") = 1e-8f, py::arg("weight_decay") = 0.0f, py::arg("grad_scale") = 1.0f,
           py::arg("fuse_pull") = true, py::arg("raw_grad") = "bf16", py::arg("max_ctas") = 0,
           py::arg("async_updates") = false)
      .def("set_lr", &PyGpuServer::set_lr)
      .def("lr", &PyGpuServer::lr)
      .def("set_symmetric", &PyGpuServer::set_symmetric, py::arg("mc_ptr"), py::arg("peer_ptrs"),
           py::arg("bytes"))
      .def("num_multicast_fanouts", &PyGpuServer::num_multicast_fanouts)
      .def("on_device", &PyGpuServer::on_device)
      .def("set_symmetric_grads", &PyGpuServer::set_symmetric_grads, py::arg("mc_ptr"), py::arg("bytes"))
      .def("num_switch_reductions", &PyGpuServer::num_switch_reductions)
      .def("num_updates", &PyGpuServer::num_updates)
      .def("num_fused_fanouts", &PyGpuServer::num_fused_fanouts)
      .def("num_keys", &PyGpuServer::num_keys)
      .def("state_bytes", &PyGpuServer::state_bytes)
      .def("num_bad_rows", &PyGpuServer::num_bad_rows)
      .def("save", &PyGpuServer::save)
      .def("load", &PyGpuServer::load)
      .def("read_master", &PyGpuServer::read_master);

  // ---- fused Llama-block kernels (see pslite_b200/ops/fused.py for the autograd wrappers) ----
  m.def("rope_split", [](const torch::Tensor& qkv, const torch::Tensor& cos, const torch::Tensor& sin,
                         int n_heads, int n_kv, int hd) {
    TORCH_CHECK(qkv.is_cuda() && qkv.is_contiguous() && qkv.scalar_type() == torch::kBFloat16);
    TORCH_CHECK(cos.scalar_type() == torch::kFloat32 && cos.is_contiguous() && sin.is_contiguous());
    const int64_t B = qkv.size(0), S = qkv.size(1);
    TORCH_CHECK(qkv.size(2) == static_cast<int64_t>(n_heads + 2 * n_kv) * hd && cos.size(0) >= S);
    auto q = torch::empty({B, S, n_heads, hd}, qkv.options());
    auto k = torch::empty({B, S, n_kv, hd}, qkv.options());
    auto v = torch::empty({B, S, n_kv, hd}, qkv.options());
    CheckRc(ps_launch_rope_split(qkv.data_ptr(), q.data_ptr(), k.data_ptr(), v.data_ptr(),
                                 cos.data_ptr<float>(), sin.data_ptr<float>(),
                                 static_cast<size_t>(B * S), static_cast<int>(S), n_heads, n_kv, hd,
                                 CurrentStream(qkv)), "rope_split");
    return std::make_tuple(q, k, v);
  });
  m.def("rope_merge_bwd", [](const torch::Tensor& dq, const torch::Tensor& dk, const torch::Tensor& dv,
                             const torch::Tensor& cos, const torch::Tensor& sin, int n_heads, int n_kv,
                             int hd) {
    TORCH_CHECK(dq.is_contiguous() && dk.is_contiguous() && dv.is_contiguous());
    const int64_t B = dq.size(0), S = dq.size(1);
    auto dqkv = torch::empty({B, S, static_cast<int64_t>(n_heads + 2 * n_kv) * hd}, dq.options());
    CheckRc(ps_launch_rope_merge_bwd(dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), dqkv.data_ptr(),
                                     cos.data_ptr<float>(), sin.data_ptr<float>(),
                                     static_cast<size_t>(B * S), static_cast<int>(S), n_heads, n_kv,
                                     hd, CurrentStream(dq)), "rope_merge_bwd");
    return dqkv;
  });
  m.def("swiglu_fwd", [](const torch::Tensor& gu) {
    TORCH_CHECK(gu.is_cuda() && gu.is_contiguous() && gu.scalar_type() == torch::kBFloat16);
    const int64_t f = gu.size(-1) / 2;
    auto sizes = gu.sizes().vec();
    sizes.back() = f;
    auto out = torch::empty(sizes, gu.options());
    CheckRc(ps_launch_swiglu_fwd(gu.data_ptr(), out.data_ptr(), static_cast<size_t>(gu.numel() / (2 * f)),
                                 static_cast<int>(f), CurrentStream(gu)), "swiglu_fwd");
    return out;
  });
  m.def("swiglu_bwd", [](const torch::Tensor& gu, const torch::Tensor& dout) {
    TORCH_CHECK(gu.is_contiguous() && dout.is_contiguous());
    const int64_t f = gu.size(-1) / 2;
    auto dgu = torch::empty_like(gu);
    CheckRc(ps_launch_swiglu_bwd(gu.data_ptr(), dout.data_ptr(), dgu.data_ptr(),
                                 static_cast<size_t>(gu.numel() / (2 * f)), static_cast<int>(f),
                                 CurrentStream(gu)), "swiglu_bwd");
    return dgu;
  });

  // the engine is not tied to a GPU (host backend on host vans): a neutral alias
  m.attr("ParamServer") = m.attr("GpuServer");

  // ---- raw kernel entry points (numerics tests, standalone use) ----
  m.def("copy_codec", [](torch::Tensor dst, const torch::Tensor& src, int codec, float scale,
                         int max_ctas) {
    if (!dst.is_cuda() && !src.is_cuda()) {  // CPU twin (src/kernels/host_kernels.cc)
      TORCH_CHECK(ps_host_copy(dst.data_ptr(), src.data_ptr(), static_cast<size_t>(src.nbytes()), codec,
                               scale) == 0, "ps_host_copy: unknown codec");
      return;
    }
    TORCH_CHECK(dst.is_cuda() && src.is_cuda(), "copy_codec needs both tensors on the same kind of device");
    CheckRc(ps_launch_copy(dst.data_ptr(), src.data_ptr(), static_cast<size_t>(src.nbytes()), codec,
                           scale, max_ctas, CurrentStream(src)), "ps_launch_copy");
  }, py::arg("dst"), py::arg("src"), py::arg("codec") = 0, py::arg("scale") = 1.0f,
     py::arg("max_ctas") = 0);
  // the same copy, finishing with the in-kernel completion signal: `flag` (a one-element int64
  // tensor in pinned host memory or on the device) receives `value` once the bytes are visible
  m.def("copy_signal", [](torch::Tensor dst, const torch::Tensor& src, int codec, float scale, int max_ctas,
                          torch::Tensor flag, int64_t value, torch::Tensor counter) {
    TORCH_CHECK(dst.is_cuda() && src.is_cuda() && counter.is_cuda(), "copy_signal is a device operation");
    TORCH_CHECK(flag.numel() == 1 && flag.element_size() == 8, "flag: one 64-bit word");
    void* fptr = flag.data_ptr();
    if (!flag.is_cuda()) {
      TORCH_CHECK(flag.is_pinned(), "a host flag must live in pinned memory");
      TORCH_CHECK(cudaHostGetDevicePointer(&fptr, flag.data_ptr(), 0) == cudaSuccess, "flag is not device-mapped");
    }
    ps_signal sig;
    sig.counter = reinterpret_cast<unsigned*>(counter.data_ptr());
    sig.flag = static_cast<unsigned long long*>(fptr);
    sig.value = static_cast<unsigned long long>(value);
    CheckRc(ps_launch_copy_signal(dst.data_ptr(), src.data_ptr(), static_cast<size_t>(src.nbytes()), codec,
                                  scale, max_ctas, &sig, CurrentStream(src)), "ps_launch_copy_signal");
  }, py::arg("dst"), py::arg("src"), py::arg("codec"), py::arg("scale"), py::arg("max_ctas"),
     py::arg("flag"), py::arg("value"), py::arg("counter"));
  // K_pull through the switch: src -> every buffer bound to the multicast address (one multimem.st stream)
  m.def("copy_multicast", [](uint64_t mc_dst, const torch::Tensor& src, int max_ctas) {
    TORCH_CHECK(src.is_cuda() && mc_dst != 0, "copy_multicast: device source and a multicast address");
    CheckRc(ps_launch_copy_multicast(reinterpret_cast<void*>(mc_dst), src.data_ptr(), static_cast<size_t>(src.nbytes()),
                                     max_ctas, nullptr, CurrentStream(src)), "ps_launch_copy_multicast");
  }, py::arg("mc_dst"), py::arg("src"), py::arg("max_ctas") = 0);
  m.def("copy_multi", [](std::vector<torch::Tensor> dsts, const std::vector<torch::Tensor>& srcs, int max_ctas) {
    TORCH_CHECK(dsts.size() == srcs.size(), "dsts / srcs length mismatch");
    if (dsts.empty()) return;
    std::vector<ps_copy_seg> segs;
    for (size_t i = 0; i < dsts.size(); ++i) {
      TORCH_CHECK(dsts[i].nbytes() >= srcs[i].nbytes(), "destination ", i, " too small");
      TORCH_CHECK(dsts[i].is_cuda() == srcs[0].is_cuda() && srcs[i].is_cuda() == srcs[0].is_cuda(),
                  "all tensors must live on the same kind of device");
      segs.push_back(ps_copy_seg{dsts[i].data_ptr(), srcs[i].data_ptr(), static_cast<size_t>(srcs[i].nbytes())});
    }
    if (!srcs[0].is_cuda()) {
      for (const ps_copy_seg& g : segs) ps_host_copy(g.dst, g.src, g.bytes, PS_CODEC_RAW, 1.f);
      return;
    }
    CheckRc(ps_launch_copy_multi(segs.data(), static_cast<int>(segs.size()), max_ctas, CurrentStream(srcs[0])),
            "ps_launch_copy_multi");
  }, py::arg("dsts"), py::arg("srcs"), py::arg("max_ctas") = 0);
  m.def("decode", [](torch::Tensor dst_f32, const torch::Tensor& wire, int64_t n, int fmt) {
    if (!wire.is_cuda()) {
      TORCH_CHECK(ps_host_decode(dst_f32.data_ptr<float>(), wire.data_ptr(), static_cast<size_t>(n), fmt) == 0,
                  "ps_host_decode: unknown format");
      return;
    }
    CheckRc(ps_launch_decode(dst_f32.data_ptr(), wire.data_ptr(), static_cast<size_t>(n), fmt,
                             CurrentStream(wire)), "ps_launch_decode");
  });
  m.def("fused_update", [](std::vector<torch::Tensor> grads, int grad_format, torch::Tensor master,
                           torch::Tensor mom, torch::Tensor var, std::vector<torch::Tensor> outs,
                           const std::string& optimizer, float lr, float beta1, float beta2,
                           float eps, float wd, int step, float grad_scale, int max_ctas,
                           uint64_t mc_ptr, uint64_t grad_mc_ptr) {
    // the kernel and its CPU twin trust every size below: an undersized tensor is an out-of-bounds write
    const int64_t n = master.numel();
    const bool adam = optimizer == "adamw";
    TORCH_CHECK(adam || optimizer == "sgd", "fused_update: optimizer must be 'adamw' or 'sgd'");
    TORCH_CHECK(!adam || step >= 1, "fused_update: the AdamW step count starts at 1");
    TORCH_CHECK(outs.size() <= PS_MAX_FANOUT, "fused_update: at most ", PS_MAX_FANOUT, " outputs");
    auto check_tensor = [&](const torch::Tensor& t, const char* what) {
      TORCH_CHECK(t.is_contiguous(), "fused_update: ", what, " must be contiguous");
      TORCH_CHECK(t.device() == master.device(), "fused_update: ", what, " is on ", t.device(),
                  ", master on ", master.device());
    };
    check_tensor(master, "master");
    check_tensor(mom, "m");
    TORCH_CHECK(mom.numel() >= n, "fused_update: m has ", mom.numel(), " elements, master ", n);
    if (adam) {
      check_tensor(var, "v");
      TORCH_CHECK(var.numel() >= n, "fused_update: v has ", var.numel(), " elements, master ", n);
    }
    if (!grad_mc_ptr) {
      TORCH_CHECK(grads.size() >= 1 && grads.size() <= PS_MAX_FANIN, "fused_update: 1 to ", PS_MAX_FANIN,
                  " gradient slots, got ", grads.size());
      const int64_t npad = (n + 31) / 32 * 32;
      int64_t slot_bytes = 0;
      switch (grad_format) {
        case PS_GRAD_BF16: slot_bytes = 2 * n; break;
        case PS_GRAD_F32: slot_bytes = 4 * n; break;
        case PS_GRAD_FP8BLOCK: slot_bytes = npad + npad / 32; break;
        default: TORCH_CHECK(false, "fused_update: unknown gradient format ", grad_format);
      }
      for (size_t i = 0; i < grads.size(); ++i) {
        check_tensor(grads[i], "a gradient slot");
        TORCH_CHECK(static_cast<int64_t>(grads[i].nbytes()) >= slot_bytes, "fused_update: gradient slot ", i,
                    " holds ", grads[i].nbytes(), " bytes, the format needs ", slot_bytes);
      }
    }
    for (size_t k = 0; k < outs.size(); ++k) {
      check_tensor(outs[k], "an output");
      TORCH_CHECK(outs[k].scalar_type() == outs[0].scalar_type() &&
                  (outs[0].scalar_type() == torch::kBFloat16 || outs[0].scalar_type() == torch::kFloat32),
                  "fused_update: the outputs must all be bfloat16 or all float32");
      TORCH_CHECK(outs[k].numel() >= n, "fused_update: output ", k, " has ", outs[k].numel(),
                  " elements, master ", n);
    }
    ps_update_args a;
    memset(&a, 0, sizeof(a));
    a.n = static_cast<size_t>(n);
    a.num_grads = static_cast<int>(grads.size());
    a.grad_format = grad_format;
    for (size_t i = 0; i < grads.size() && i < PS_MAX_FANIN; ++i) a.grads[i] = grads[i].data_ptr();
    if (grad_mc_ptr) {  // PS_GRAD_MC_BF16: the gradients are read through a multicast address
      a.num_grads = 1;
      a.grads[0] = reinterpret_cast<const void*>(grad_mc_ptr);
    }
    a.master = master.data_ptr<float>();
    a.m = mom.data_ptr<float>();
    a.v = var.data_ptr<float>();
    a.num_outs = static_cast<int>(outs.size());
    for (size_t i = 0; i < outs.size(); ++i) a.outs[i] = outs[i].data_ptr();
    a.out_f32 = !outs.empty() && outs[0].scalar_type() == torch::kFloat32;
    a.mc_out = reinterpret_cast<void*>(mc_ptr);
    a.body_outs = mc_ptr ? std::min<int>(1, a.num_outs) : a.num_outs;
    ps_opt_params o;
    o.optimizer = optimizer == "sgd" ? PS_OPT_SGD : PS_OPT_ADAMW;
    o.lr = lr; o.beta1 = beta1; o.beta2 = beta2; o.eps = eps; o.weight_decay = wd;
    o.bias_corr1 = o.optimizer == PS_OPT_ADAMW ? 1.f - std::pow(beta1, (float)step) : 1.f;
    o.bias_corr2 = o.optimizer == PS_OPT_ADAMW ? 1.f - std::pow(beta2, (float)step) : 1.f;
    o.grad_scale = grad_scale;
    if (!master.is_cuda()) {
      TORCH_CHECK(ps_host_update(&a, &o) == 0, "ps_host_update: bad arguments");
      return;
    }
    CheckRc(ps_launch_update(&a, &o, max_ctas, CurrentStream(master)), "ps_launch_update");
  }, py::arg("grads"), py::arg("grad_format"), py::arg("master"), py::arg("m"), py::arg("v"),
     py::arg("outs"), py::arg("optimizer") = "adamw", py::arg("lr") = 1e-3f,
     py::arg("beta1") = 0.9f, py::arg("beta2") = 0.95f, py::arg("eps") = 1e-8f,
     py::arg("weight_decay") = 0.0f, py::arg("step") = 1, py::arg("grad_scale") = 1.0f,
     py::arg("max_ctas") = 0, py::arg("mc_ptr") = 0, py::arg("grad_mc_ptr") = 0);
  m.def("rows_scratch_bytes", [](uint64_t rows, int max_grads) {
    return static_cast<uint64_t>(ps_rows_scratch_bytes(rows, max_grads));
  });
  m.def("rows_slot_bytes", [](int64_t num_rows, int64_t dim, int grad_format) {
    return RowsSlotBytes(num_rows, dim, grad_format);
  });
  m.def("fused_update_rows", [](std::vector<torch::Tensor> grads, std::vector<int64_t> num_rows, int grad_format,
                                int64_t dim, torch::Tensor master, torch::Tensor mom, torch::Tensor var,
                                std::vector<torch::Tensor> outs, torch::Tensor scratch,
                                const std::string& optimizer, float lr, float beta1, float beta2, float eps,
                                float wd, int step, float grad_scale, int max_ctas) {
    // the kernel and its CPU twin trust every size below: an undersized tensor is an out-of-bounds access
    const int64_t n = master.numel();
    const bool adam = optimizer == "adamw";
    TORCH_CHECK(adam || optimizer == "sgd", "fused_update_rows: optimizer must be 'adamw' or 'sgd'");
    TORCH_CHECK(!adam || step >= 1, "fused_update_rows: the AdamW step count starts at 1");
    TORCH_CHECK(grads.size() >= 1 && grads.size() <= PS_MAX_FANIN, "fused_update_rows: 1 to ", PS_MAX_FANIN,
                " gradient slots, got ", grads.size());
    TORCH_CHECK(num_rows.size() == grads.size(), "fused_update_rows: ", grads.size(), " slots but ",
                num_rows.size(), " row counts");
    TORCH_CHECK(outs.size() <= PS_MAX_FANOUT, "fused_update_rows: at most ", PS_MAX_FANOUT, " outputs");
    TORCH_CHECK(grad_format == PS_GRAD_F32 || grad_format == PS_GRAD_BF16 || grad_format == PS_GRAD_FP8BLOCK,
                "fused_update_rows: unknown gradient format ", grad_format);
    TORCH_CHECK(dim > 0 && dim % 8 == 0, "fused_update_rows: the row width must be a positive multiple of 8, got ",
                dim);
    TORCH_CHECK(grad_format != PS_GRAD_FP8BLOCK || dim % 32 == 0,
                "fused_update_rows: fp8 rows need a row width that is a multiple of 32, got ", dim);
    TORCH_CHECK(master.scalar_type() == torch::kFloat32 && n % dim == 0,
                "fused_update_rows: master must be float32 with a whole number of rows of ", dim);
    const int64_t rows = n / dim;
    auto check_tensor = [&](const torch::Tensor& t, const char* what) {
      TORCH_CHECK(t.is_contiguous(), "fused_update_rows: ", what, " must be contiguous");
      TORCH_CHECK(t.device() == master.device(), "fused_update_rows: ", what, " is on ", t.device(),
                  ", master on ", master.device());
    };
    check_tensor(master, "master");
    check_tensor(mom, "m");
    TORCH_CHECK(mom.scalar_type() == torch::kFloat32 && mom.numel() >= n, "fused_update_rows: m must be float32 with ",
                n, " elements");
    if (adam) {
      check_tensor(var, "v");
      TORCH_CHECK(var.scalar_type() == torch::kFloat32 && var.numel() >= n,
                  "fused_update_rows: v must be float32 with ", n, " elements");
    }
    for (size_t i = 0; i < grads.size(); ++i) {
      check_tensor(grads[i], "a gradient slot");
      TORCH_CHECK(num_rows[i] >= 0 && num_rows[i] <= 0xffffffffll, "fused_update_rows: bad row count ",
                  num_rows[i]);
      const int64_t need = RowsSlotBytes(num_rows[i], dim, grad_format);
      TORCH_CHECK(static_cast<int64_t>(grads[i].nbytes()) >= need, "fused_update_rows: gradient slot ", i, " holds ",
                  grads[i].nbytes(), " bytes, ", num_rows[i], " rows need ", need);
    }
    for (size_t k = 0; k < outs.size(); ++k) {
      check_tensor(outs[k], "an output");
      TORCH_CHECK(outs[k].scalar_type() == outs[0].scalar_type() &&
                  (outs[0].scalar_type() == torch::kBFloat16 || outs[0].scalar_type() == torch::kFloat32),
                  "fused_update_rows: the outputs must all be bfloat16 or all float32");
      TORCH_CHECK(outs[k].numel() >= n, "fused_update_rows: output ", k, " has ", outs[k].numel(),
                  " elements, master ", n);
    }
    check_tensor(scratch, "scratch");
    const size_t scratch_need = ps_rows_scratch_bytes(static_cast<size_t>(rows), static_cast<int>(grads.size()));
    TORCH_CHECK(scratch.nbytes() >= scratch_need, "fused_update_rows: scratch holds ", scratch.nbytes(),
                " bytes, needs ", scratch_need);
    ps_update_rows_args a;
    memset(&a, 0, sizeof(a));
    a.rows = static_cast<size_t>(rows);
    a.dim = static_cast<int>(dim);
    a.num_grads = static_cast<int>(grads.size());
    a.grad_format = grad_format;
    for (size_t i = 0; i < grads.size(); ++i) {
      a.grads[i] = grads[i].data_ptr();
      a.num_rows[i] = static_cast<uint32_t>(num_rows[i]);
    }
    a.master = master.data_ptr<float>();
    a.m = mom.data_ptr<float>();
    a.v = adam ? var.data_ptr<float>() : nullptr;
    a.num_outs = static_cast<int>(outs.size());
    for (size_t i = 0; i < outs.size(); ++i) a.outs[i] = outs[i].data_ptr();
    a.out_f32 = !outs.empty() && outs[0].scalar_type() == torch::kFloat32;
    a.scratch = scratch.data_ptr();
    ps_opt_params o;
    o.optimizer = adam ? PS_OPT_ADAMW : PS_OPT_SGD;
    o.lr = lr; o.beta1 = beta1; o.beta2 = beta2; o.eps = eps; o.weight_decay = wd;
    o.bias_corr1 = adam ? 1.f - std::pow(beta1, (float)step) : 1.f;
    o.bias_corr2 = adam ? 1.f - std::pow(beta2, (float)step) : 1.f;
    o.grad_scale = grad_scale;
    if (!master.is_cuda()) {
      TORCH_CHECK(ps_host_update_rows(&a, &o) == 0, "ps_host_update_rows: bad arguments");
      return;
    }
    CheckRc(ps_launch_update_rows(&a, &o, max_ctas, CurrentStream(master)), "ps_launch_update_rows");
  }, py::arg("grads"), py::arg("num_rows"), py::arg("grad_format"), py::arg("dim"), py::arg("master"),
     py::arg("m"), py::arg("v"), py::arg("outs"), py::arg("scratch"), py::arg("optimizer") = "adamw",
     py::arg("lr") = 1e-3f, py::arg("beta1") = 0.9f, py::arg("beta2") = 0.95f, py::arg("eps") = 1e-8f,
     py::arg("weight_decay") = 0.0f, py::arg("step") = 1, py::arg("grad_scale") = 1.0f, py::arg("max_ctas") = 0);
}
