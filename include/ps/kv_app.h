/**
 * \file kv_app.h
 * \brief The key-value application layer: KVPairs, KVWorker (push / pull client),
 *        KVServer (request handler host), KVServerDefaultHandle.
 *
 * API parity: reference include/ps/kv_app.h:40-50 (KVPairs), :65-318 (KVWorker),
 * :321-340 (KVMeta), :345-424 (KVServer), :430-452 (default handle), :566-621
 * (default slicer). Behavioural notes:
 *   - keys must be unique and sorted; a request is cut by the server key ranges
 *     into one zero-copy message per non-empty slice;
 *   - with a one-sided van (nvl / shm, i.e. any DMLC_ENABLE_RDMA value other
 *     than unset/0/zmq) pulls are zero-copy: the server writes straight into the
 *     caller's `vals` buffer, which therefore must be pre-sized;
 *   - meta.key always carries the first key of the slice so transports and
 *     registered receive buffers can key on it without touching the payload
 *     (which may live in HBM).
 */
#ifndef PS_KV_APP_H_
#define PS_KV_APP_H_
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>
#include "ps/base.h"
#include "ps/internal/spin_mutex.h"
#include "ps/simple_app.h"

namespace ps {

/*!
 * \brief a list of key-value pairs. keys are sorted and unique; the value of
 *        keys[i] is vals[i*k, (i+1)*k) for fixed k, or described by lens[i].
 */
template <typename Val>
struct KVPairs {
  SArray<Key> keys;
  SArray<Val> vals;
  SArray<int> lens;
};

/*! \brief request descriptor handed to a KVServer handler */
struct KVMeta {
  int cmd = 0;
  bool push = false;
  /*! \brief *group-level* node id of the requesting worker */
  int sender = 0;
  int timestamp = 0;
  int customer_id = 0;
  Key key = 0;
  uint64_t addr = 0;
  int64_t val_len = 0;
  int option = 0;
  /*! \brief peer-mappable location of the worker's value buffer (one-sided vans) */
  MemRef mem;
  /*! \brief WireCodec the sender applied to the values, and its scale */
  int codec = 0;
  float scale = 1.0f;
  /*!
   * \brief fused push-pull (KVWorker::ZPushPull): `push` is true AND the worker wants the values
   *        back. Answer with Response(req, result) — it is delivered as the pull reply to
   *        `pull_addr` / `pull_mem` — and do not send a separate ack.
   */
  bool pull = false;
  uint64_t pull_addr = 0;
  int64_t pull_len = 0;
  MemRef pull_mem;
};

namespace kv_detail {
/*! \brief true if DMLC_ENABLE_RDMA / DMLC_ENABLE_UCX / PS_VAN_TYPE select a one-sided van */
inline bool OneSidedVanSelected() {
  if (GetEnv("DMLC_ENABLE_UCX", 0) == 1) return true;
  std::string t = GetEnvStr("DMLC_ENABLE_RDMA", "zmq");
  if (const char* v = Environment::Get()->find("PS_VAN_TYPE")) t = v;
  return !(t.empty() || t == "0" || t == "zmq" || t == "tcp" || t == "multivan");
}
/*! \brief non-owning view of a caller-owned destination container */
template <typename T>
inline SArray<T> ViewOf(SArray<T>* a) { return *a; }
template <typename T>
inline SArray<T> ViewOf(std::vector<T>* v) { return SArray<T>(v->data(), v->size(), false); }
}  // namespace kv_detail

/*!
 * \brief push / pull client of a worker node.
 * \tparam Val a primitive value type (float, char for raw bytes, ...)
 */
template <typename Val>
class KVWorker : public SimpleApp {
 public:
  using SimpleApp::obj_;
  /*! \brief runs on the receive thread once a push is stored / a pull has landed */
  using Callback = std::function<void()>;

  /*! \brief true when pulls land directly in the caller's buffer */
  bool is_worker_zpull_;

  /*!
   * \param app_id matches the KVServer's app id
   * \param customer_id locally unique
   * \param instance_idx which worker instance of the group (DMLC_GROUP_SIZE) to use
   */
  explicit KVWorker(int app_id, int customer_id, int instance_idx = 0) : SimpleApp() {
    using namespace std::placeholders;
    postoffice_ = Postoffice::GetWorker(instance_idx);
    instance_idx_ = instance_idx;
    CHECK_GT(postoffice_->group_size(), instance_idx);
    slicer_ = std::bind(&KVWorker<Val>::DefaultSlicer, this, _1, _2, _3);
    is_worker_zpull_ = kv_detail::OneSidedVanSelected();
    obj_ = new Customer(app_id, customer_id, std::bind(&KVWorker<Val>::Process, this, _1),
                        postoffice_, false);
    obj_->Start();  // only now: Process() dereferences obj_
  }
  virtual ~KVWorker() {
    delete obj_;
    obj_ = nullptr;
  }

  /*!
   * \brief push {keys, vals} (copied) to the servers owning the keys; asynchronous.
   * \return the request timestamp for Wait()
   */
  int Push(const std::vector<Key>& keys, const std::vector<Val>& vals,
           const std::vector<int>& lens = {}, int cmd = 0, const Callback& cb = nullptr) {
    return ZPush(SArray<Key>(keys), SArray<Val>(vals), SArray<int>(lens), cmd, cb);
  }

  /*! \brief pull the values of `keys` into *vals (resized if empty); asynchronous */
  int Pull(const std::vector<Key>& keys, std::vector<Val>* vals, std::vector<int>* lens = nullptr,
           int cmd = 0, const Callback& cb = nullptr) {
    return Pull_(SArray<Key>(keys), vals, lens, cmd, cb);
  }

  /*! \brief block until the request `timestamp` has been answered by every server */
  void Wait(int timestamp) { obj_->WaitRequest(timestamp); }

  /*!
   * \brief zero-copy push: the arrays must stay untouched until completion.
   *        `vals` may live in GPU memory (tag the SArray with GPU placement).
   */
  int ZPush(const SArray<Key>& keys, const SArray<Val>& vals, const SArray<int>& lens = {},
            int cmd = 0, const Callback& cb = nullptr) {
    return ZPush(keys, vals, lens, cmd, cb, SendOpts());
  }
  /*!
   * \brief ZPush whose transport copy is fused with a transform (`opts.codec`:
   *        scale / cast to bf16 / block-scaled fp8) and gated on `opts.wait_event`.
   *        One-sided vans only; the server sees the wire form.
   */
  int ZPush(const SArray<Key>& keys, const SArray<Val>& vals, const SArray<int>& lens, int cmd,
            const Callback& cb, const SendOpts& opts) {
    const int ts = obj_->NewRequest(kServerGroup);
    AddCallback(ts, cb);
    KVPairs<Val> kvs;
    kvs.keys = keys;
    kvs.vals = vals;
    kvs.lens = lens;
    Send(ts, true, cmd, kvs, opts);
    return ts;
  }

  /*! \brief zero-copy pull into *vals (and *lens) */
  int ZPull(const SArray<Key>& keys, SArray<Val>* vals, SArray<int>* lens = nullptr, int cmd = 0,
            const Callback& cb = nullptr) {
    return Pull_(keys, vals, lens, cmd, cb);
  }
  /*! \brief ZPull whose destination the server already knows as `opts.dest_mem` */
  int ZPull(const SArray<Key>& keys, SArray<Val>* vals, SArray<int>* lens, int cmd,
            const Callback& cb, const SendOpts& opts) {
    return Pull_(keys, vals, lens, cmd, cb, opts);
  }

  /*!
   * \brief fused push + pull: push `vals`, and receive the server's values for the same keys in
   *        `*outs` with ONE request and ONE reply per server instead of two each. The server
   *        handler sees `req.push && req.pull`. When the keys span several servers `*outs` must
   *        mirror `vals` (same size, same layout); a request that goes to a single server may
   *        pull a differently sized result (e.g. push fp32 gradients, receive bf16 parameters).
   *        `opts.pull_dest_mem` names a destination the server already knows (symmetric buffer).
   */
  int ZPushPull(const SArray<Key>& keys, const SArray<Val>& vals, SArray<Val>* outs,
                SArray<int>* lens = nullptr, int cmd = 0, const Callback& cb = nullptr,
                const SendOpts& opts = SendOpts()) {
    CHECK_NOTNULL(outs);
    return Pull_(keys, outs, lens, cmd, cb, opts, &vals);
  }
  /*! \brief copying convenience form of ZPushPull */
  int PushPull(const std::vector<Key>& keys, const std::vector<Val>& vals, std::vector<Val>* outs,
               int cmd = 0, const Callback& cb = nullptr) {
    CHECK_NOTNULL(outs)->resize(vals.size());
    SArray<Val> v(vals);  // owned copy: the caller may drop `vals` right away
    return Pull_(SArray<Key>(keys), outs, static_cast<std::vector<int>*>(nullptr), cmd, cb, SendOpts(), &v);
  }

  using SlicedKVs = std::vector<std::pair<bool, KVPairs<Val>>>;
  /*! \brief cuts `send` by `ranges`; sliced[i].first==false means "nothing for server i" */
  using Slicer = std::function<void(const KVPairs<Val>& send, const std::vector<Range>& ranges,
                                    SlicedKVs* sliced)>;
  void set_slicer(const Slicer& slicer) {
    CHECK(slicer);
    slicer_ = slicer;
  }

 private:
  template <typename C, typename D>
  int Pull_(const SArray<Key>& keys, C* vals, D* lens, int cmd, const Callback& cb,
            const SendOpts& opts = SendOpts(), const SArray<Val>* push_vals = nullptr);

  void AddCallback(int timestamp, Callback cb) {
    if (!cb) return;
    std::lock_guard<SpinMutex> lk(mu_);
    callbacks_[timestamp] = std::move(cb);  // by value + move: the closure is built exactly once
  }
  void RunCallback(int timestamp);
  void Send(int timestamp, bool push, int cmd, KVPairs<Val>& kvs, const SendOpts& opts = SendOpts(),
            const SArray<Val>* pull_dest = nullptr);
  void Process(const Message& msg);
  void DefaultSlicer(const KVPairs<Val>& send, const std::vector<Range>& ranges,
                     SlicedKVs* sliced);

  std::unordered_map<int, std::vector<KVPairs<Val>>> recv_kvs_;
  std::unordered_map<int, Callback> callbacks_;
  SpinMutex mu_;  // callbacks_ / recv_kvs_: touched once per request and per response
  Slicer slicer_;
  int instance_idx_;
};

/*! \brief hosts the user's request handler on a server node */
template <typename Val>
class KVServer : public SimpleApp {
 public:
  explicit KVServer(int app_id, bool is_scheduler = false, int instance_idx = 0) : SimpleApp() {
    using namespace std::placeholders;
    postoffice_ = is_scheduler ? Postoffice::GetScheduler() : Postoffice::GetServer(instance_idx);
    CHECK(postoffice_) << is_scheduler << " " << instance_idx;
    instance_idx_ = instance_idx;
    // servers run exactly one customer per app: customer_id == app_id
    obj_ = new Customer(app_id, app_id, std::bind(&KVServer::Process, this, _1), postoffice_, false);
    obj_->Start();  // only now: Process() / Response() dereference obj_
  }
  virtual ~KVServer() {
    delete obj_;
    obj_ = nullptr;
  }

  /*! \brief user logic: aggregate pushes, answer pulls; must call Response() */
  using ReqHandle = std::function<void(const KVMeta& req_meta, const KVPairs<Val>& req_data,
                                       KVServer* server)>;
  void set_request_handle(const ReqHandle& h) {
    CHECK(h) << "invalid request handle";
    {
      std::lock_guard<std::mutex> lk(handle_mu_);
      request_handle_ = h;
      handle_ready_.store(true, std::memory_order_release);
    }
    handle_cv_.notify_all();
  }

  /*! \brief reply to `req`; `res` is empty for a push ack */
  void Response(const KVMeta& req, const KVPairs<Val>& res = KVPairs<Val>()) {
    Response(req, res, SendOpts());
  }
  /*! \brief reply whose value copy is fused with `opts.codec` and gated on `opts.wait_event` */
  void Response(const KVMeta& req, const KVPairs<Val>& res, const SendOpts& opts);

  /*! \brief deprecated: takes an instance-level worker *id* */
  void RegisterRecvBuffer(int worker_id, SArray<Key>& keys, const SArray<Val>& vals,
                          const SArray<int>& lens = {}, int cmd = 0) {
    LOG(WARNING) << "RegisterRecvBuffer is deprecated. Please use RegisterRecvBufferWithRank";
    RegisterRecvBuffer_(worker_id, keys, vals, lens, cmd);
  }
  /*!
   * \brief pushes of `keys[0]` from worker group `worker_rank` will be delivered
   *        in `vals` (no allocation, no copy; on the NVLink van `vals` is HBM)
   */
  void RegisterRecvBufferWithRank(int worker_rank, SArray<Key>& keys, const SArray<Val>& vals,
                                  const SArray<int>& lens = {}, int cmd = 0) {
    const int id = postoffice_->GroupWorkerRankToInstanceID(worker_rank, instance_idx_);
    RegisterRecvBuffer_(id, keys, vals, lens, cmd);
  }

  /*! \brief offset of this server inside its instance group */
  int instance_idx_;

 private:
  void Process(const Message& msg);
  void RegisterRecvBuffer_(int worker_id, SArray<Key>& keys, const SArray<Val>& vals,
                           const SArray<int>& lens, int cmd);
  ReqHandle request_handle_;
  // a request can arrive between the constructor (which starts receiving) and
  // set_request_handle(): Process waits for the handle instead of failing
  std::mutex handle_mu_;
  std::condition_variable handle_cv_;
  std::atomic<bool> handle_ready_{false};
};

/*! \brief example handler: store[key] += val on push, lookup on pull (scalar per key) */
template <typename Val>
struct KVServerDefaultHandle {
  void operator()(const KVMeta& req_meta, const KVPairs<Val>& req_data, KVServer<Val>* server) {
    const size_t n = req_data.keys.size();
    KVPairs<Val> res;
    if (req_meta.push) {
      CHECK_EQ(n, req_data.vals.size());
      for (size_t i = 0; i < n; ++i) store[req_data.keys[i]] += req_data.vals[i];
    }
    if (!req_meta.push || req_meta.pull) {  // a pull, or the reply half of a fused push-pull
      res.keys = req_data.keys;
      res.vals.resize(n);
      for (size_t i = 0; i < n; ++i) res.vals[i] = store[req_data.keys[i]];
    }
    server->Response(req_meta, res);
  }
  std::unordered_map<Key, Val> store;
};

// ---------------------------------------------------------------------------
// KVServer
// ---------------------------------------------------------------------------

template <typename Val>
void KVServer<Val>::RegisterRecvBuffer_(int worker_id, SArray<Key>& keys, const SArray<Val>& vals,
                                        const SArray<int>& lens, int cmd) {
  CHECK(keys.size());
  CHECK(lens.size());
  Message msg;
  msg.meta.request = true;
  msg.meta.push = true;
  msg.meta.head = cmd;
  msg.meta.sender = worker_id;
  msg.meta.key = keys[0];
  msg.AddData(keys);
  msg.AddData(vals);
  msg.AddData(lens);
  postoffice_->van()->RegisterRecvBuffer(msg);
}

template <typename Val>
void KVServer<Val>::Process(const Message& msg) {
  if (msg.meta.simple_app) {
    SimpleApp::Process(msg);
    return;
  }
  KVMeta meta;
  meta.cmd = msg.meta.head;
  meta.push = msg.meta.push;
  // handlers see the worker *group* id, whichever instance of it sent the message
  meta.sender = Postoffice::WorkerRankToID(postoffice_->InstanceIDtoGroupRank(msg.meta.sender));
  meta.timestamp = msg.meta.timestamp;
  meta.customer_id = msg.meta.customer_id;
  meta.key = msg.meta.key;
  meta.addr = msg.meta.addr;
  meta.val_len = msg.meta.val_len;
  meta.option = msg.meta.option;
  meta.mem = msg.meta.mem;
  meta.codec = msg.meta.codec;
  meta.scale = msg.meta.scale;
  meta.pull = msg.meta.pull;
  meta.pull_addr = msg.meta.pull_addr;
  meta.pull_len = msg.meta.pull_len;
  meta.pull_mem = msg.meta.pull_mem;
  KVPairs<Val> data;
  const size_t n = msg.data.size();
  if (n) {
    CHECK_GE(n, (size_t)2);
    data.keys = msg.data[0];
    data.vals = msg.data[1];
    if (n > 2) {
      CHECK_EQ(n, (size_t)3);
      data.lens = msg.data[2];
      CHECK_EQ(data.lens.size(), data.keys.size());
    }
  }
  if (!handle_ready_.load(std::memory_order_acquire)) {
    std::unique_lock<std::mutex> lk(handle_mu_);
    handle_cv_.wait_for(lk, std::chrono::seconds(30),
                        [this] { return handle_ready_.load(std::memory_order_acquire); });
  }
  CHECK(handle_ready_.load(std::memory_order_acquire)) << "KVServer got a request but no request handle was set";
  request_handle_(meta, data, this);
}

template <typename Val>
void KVServer<Val>::Response(const KVMeta& req, const KVPairs<Val>& res, const SendOpts& opts) {
  // answer the instance of the worker group that pairs with this server instance
  const int worker_rank = Postoffice::IDtoRank(req.sender);
  Message msg;
  msg.meta.app_id = obj_->app_id();
  msg.meta.customer_id = req.customer_id;
  msg.meta.request = false;
  msg.meta.push = req.push;
  msg.meta.head = req.cmd;
  msg.meta.timestamp = req.timestamp;
  msg.meta.recver = postoffice_->GroupWorkerRankToInstanceID(worker_rank, instance_idx_);
  msg.meta.key = req.key;
  msg.meta.addr = req.addr;
  msg.meta.val_len = req.val_len;
  msg.meta.option = req.option;
  msg.meta.mem = req.mem;
  if (req.push && req.pull) {
    // fused push-pull: the one reply is a pull response aimed at the worker's destination
    CHECK(res.keys.size()) << "a push-pull request must be answered with the values";
    msg.meta.push = false;
    msg.meta.addr = req.pull_addr;
    msg.meta.val_len = req.pull_len;
    msg.meta.mem = req.pull_mem;
  }
  msg.meta.codec = opts.codec;
  msg.meta.scale = opts.scale;
  msg.wait_event = opts.wait_event;
  if (res.keys.size()) {
    msg.AddData(res.keys);
    msg.AddData(res.vals);
    if (res.lens.size()) msg.AddData(res.lens);
  }
  postoffice_->van()->Send(msg);
}

// ---------------------------------------------------------------------------
// KVWorker
// ---------------------------------------------------------------------------

template <typename Val>
void KVWorker<Val>::DefaultSlicer(const KVPairs<Val>& send, const std::vector<Range>& ranges,
                                  typename KVWorker<Val>::SlicedKVs* sliced) {
  const size_t n = ranges.size();
  sliced->assign(n, std::make_pair(false, KVPairs<Val>()));
  if (send.keys.empty()) return;

  if (send.keys.size() == 1) {
    // one key (a tensor per request, the common case): no cut table, no binary searches
    const Key key = send.keys[0];
    for (size_t i = 0; i < n; ++i) {
      const bool open_end = i + 1 == n && static_cast<Key>(ranges[i].end()) == kMaxKey;
      if (key < static_cast<Key>(ranges[i].begin()) || !(key < static_cast<Key>(ranges[i].end()) || open_end)) continue;
      auto& out = (*sliced)[i];
      out.first = true;
      out.second.keys = send.keys;
      if (send.lens.empty()) {
        out.second.vals = send.vals;
      } else {
        CHECK_EQ(send.lens.size(), (size_t)1);
        out.second.lens = send.lens;
        const size_t val_to = static_cast<size_t>(send.lens[0]);
        if (val_to <= send.vals.size()) out.second.vals = send.vals.segment(0, val_to);  // a pull carries none yet
      }
      return;
    }
    LOG(FATAL) << "key " << key << " lies outside every server range";
  }

  // cut[i] = index of the first key owned by server i; keys are sorted
  std::vector<size_t> cut(n + 1, 0);
  const Key* kb = send.keys.begin();
  const Key* ke = send.keys.end();
  cut[0] = static_cast<size_t>(std::lower_bound(kb, ke, static_cast<Key>(ranges[0].begin())) - kb);
  for (size_t i = 0; i < n; ++i) {
    if (i) CHECK_EQ(ranges[i - 1].end(), ranges[i].begin());
    // the last range ends at kMaxKey, which no valid key equals or exceeds... except
    // kMaxKey itself; lower_bound on the inclusive end keeps it in the last slice
    const Key* from = kb + cut[i];
    const Key hi = static_cast<Key>(ranges[i].end());
    const Key* to = (i + 1 == n && hi == kMaxKey) ? ke : std::lower_bound(from, ke, hi);
    cut[i + 1] = static_cast<size_t>(to - kb);
  }
  CHECK_EQ(cut[0], (size_t)0) << "keys below the first server range";
  CHECK_EQ(cut[n], send.keys.size());

  size_t k = 0;  // fixed value length, when lens is absent
  if (send.lens.empty()) {
    k = send.vals.size() / send.keys.size();
    CHECK_EQ(k * send.keys.size(), send.vals.size());
  } else {
    CHECK_EQ(send.keys.size(), send.lens.size());
  }
  size_t val_at = 0;
  for (size_t i = 0; i < n; ++i) {
    if (cut[i + 1] == cut[i]) continue;
    auto& out = (*sliced)[i];
    out.first = true;
    out.second.keys = send.keys.segment(cut[i], cut[i + 1]);
    if (!send.lens.empty()) {
      out.second.lens = send.lens.segment(cut[i], cut[i + 1]);
      size_t val_to = val_at;
      for (int l : out.second.lens) val_to += static_cast<size_t>(l);
      // a pull request carries no values yet
      if (val_to <= send.vals.size()) out.second.vals = send.vals.segment(val_at, val_to);
      val_at = val_to;
    } else {
      out.second.vals = send.vals.segment(cut[i] * k, cut[i + 1] * k);
    }
  }
}

template <typename Val>
void KVWorker<Val>::Send(int timestamp, bool push, int cmd, KVPairs<Val>& kvs,
                         const SendOpts& opts, const SArray<Val>* pull_dest) {
  SlicedKVs sliced;
  slicer_(kvs, postoffice_->GetServerKeyRanges(), &sliced);

  // servers that get nothing are accounted for up front
  int skipped = 0;
  for (const auto& s : sliced) skipped += s.first ? 0 : 1;
  if (skipped) obj_->AddResponse(timestamp, skipped);
  if (static_cast<size_t>(skipped) == sliced.size()) RunCallback(timestamp);

  for (size_t i = 0; i < sliced.size(); ++i) {
    auto& s = sliced[i];
    if (!s.first) continue;
    auto& part = s.second;
    Message msg;
    msg.meta.app_id = obj_->app_id();
    msg.meta.customer_id = obj_->customer_id();
    msg.meta.request = true;
    msg.meta.push = push;
    msg.meta.head = cmd;
    msg.meta.timestamp = timestamp;
    // worker instance i of a group talks to server instance i of every group
    msg.meta.recver = postoffice_->GroupServerRankToInstanceID(static_cast<int>(i), instance_idx_);
    msg.meta.addr = reinterpret_cast<uint64_t>(part.vals.data());
    msg.meta.val_len = static_cast<int64_t>(part.vals.size());
    if (part.keys.size()) msg.meta.key = part.keys[0];
    if (pull_dest) {
      // fused push-pull: the reply lands in the slice of *pull_dest that mirrors this slice of
      // vals — or in all of it when this server gets the whole request
      CHECK(push);
      size_t off = 0, cnt = pull_dest->size();
      if (static_cast<size_t>(skipped) + 1 != sliced.size()) {
        CHECK_EQ(pull_dest->size(), kvs.vals.size()) << "ZPushPull over several servers: *outs must mirror vals";
        off = static_cast<size_t>(part.vals.data() - kvs.vals.data());
        cnt = part.vals.size();
      }
      msg.meta.pull = true;
      msg.meta.pull_addr = reinterpret_cast<uint64_t>(pull_dest->data() + off);
      msg.meta.pull_len = static_cast<int64_t>(cnt);
      if (opts.pull_dest_mem.valid()) msg.meta.pull_mem = opts.pull_dest_mem;
    }
    msg.meta.codec = opts.codec;
    msg.meta.scale = opts.scale;
    msg.meta.option = opts.option;
    msg.wait_event = opts.wait_event;
    msg.slot_bytes = opts.slot_bytes;
    if (opts.dest_mem.valid()) {
      msg.meta.mem = opts.dest_mem;
      if (push) msg.stage = opts.stage;
    }
    const SArray<Val> dest = part.vals;  // placement of the pull destination
    if (!push) part.vals.clear();
    if (part.keys.size()) {
      msg.AddData(part.keys);
      msg.AddData(part.vals);
      if (part.lens.size()) msg.AddData(part.lens);
    }
    if (!push) {
      msg.meta.src_dev_type = dest.src_device_type_;
      msg.meta.src_dev_id = dest.src_device_id_;
      msg.meta.dst_dev_type = dest.dst_device_type_;
      msg.meta.dst_dev_id = dest.dst_device_id_;
    }
    postoffice_->van()->Send(msg);
  }
}

template <typename Val>
void KVWorker<Val>::Process(const Message& msg) {
  if (msg.meta.simple_app) {
    SimpleApp::Process(msg);
    return;
  }
  const int ts = msg.meta.timestamp;
  if (!msg.meta.push && msg.data.size()) {
    CHECK_GE(msg.data.size(), (size_t)2);
    KVPairs<Val> kvs;
    kvs.keys = msg.data[0];
    kvs.vals = msg.data[1];
    if (msg.data.size() > 2) kvs.lens = msg.data[2];
    std::lock_guard<SpinMutex> lk(mu_);
    recv_kvs_[ts].push_back(kvs);
  }
  // the tracker counts this response *after* the handler returns, hence the -1
  if (obj_->NumResponse(ts) == postoffice_->num_servers() - 1) RunCallback(ts);
}

template <typename Val>
void KVWorker<Val>::RunCallback(int timestamp) {
  Callback cb;
  {
    std::lock_guard<SpinMutex> lk(mu_);
    auto it = callbacks_.find(timestamp);
    if (it == callbacks_.end()) return;
    cb = std::move(it->second);
    callbacks_.erase(it);
  }
  if (cb) cb();
}

template <typename Val>
template <typename C, typename D>
int KVWorker<Val>::Pull_(const SArray<Key>& keys, C* vals, D* lens, int cmd, const Callback& cb,
                         const SendOpts& opts, const SArray<Val>* push_vals) {
  CHECK_NOTNULL(vals);
  const int ts = obj_->NewRequest(kServerGroup);
  AddCallback(ts, [this, ts, keys, vals, lens, cb]() mutable {
    std::vector<KVPairs<Val>> parts;
    {
      std::lock_guard<SpinMutex> lk(mu_);
      auto it = recv_kvs_.find(ts);
      if (it != recv_kvs_.end()) {
        parts.swap(it->second);
        recv_kvs_.erase(it);
      }
    }
    // every key must come back exactly once
    size_t total_key = 0, total_val = 0;
    for (const auto& s : parts) {
      Range r = FindRange(keys, s.keys.front(), static_cast<Key>(s.keys.back() + 1));
      CHECK_EQ(r.size(), s.keys.size()) << "unmatched keys size from one server";
      if (lens) CHECK_EQ(s.lens.size(), s.keys.size());
      total_key += s.keys.size();
      total_val += s.vals.size();
    }
    CHECK_EQ(total_key, keys.size()) << "lost some servers?";
    std::sort(parts.begin(), parts.end(), [](const KVPairs<Val>& a, const KVPairs<Val>& b) {
      return a.keys.front() < b.keys.front();
    });
    if (vals->empty()) {
      vals->resize(total_val);
    } else {
      CHECK_GE(vals->size(), total_val);
    }
    {
      // stitch the per-server slices into the caller's buffers. A slice that landed in place
      // (zero-copy pull of a one-sided van, or TcpVan's direct landing) is skipped by the
      // pointer test, so this is also right when a one-sided van had to fall back to a
      // two-sided transfer for a buffer it could not export.
      Val* out = vals->data();
      int* out_len = nullptr;
      if (lens) {
        if (lens->empty()) {
          lens->resize(keys.size());
        } else {
          CHECK_EQ(lens->size(), keys.size());
        }
        out_len = lens->data();
      }
      for (const auto& s : parts) {
        if (s.vals.data() != out && s.vals.size()) {
          CHECK(!s.vals.on_gpu()) << "pulled values are in device memory but did not land in the "
                                     "destination; pull into an exportable device buffer";
          // memmove: a slice that landed further right in the same buffer may overlap its final place
          memmove(out, s.vals.data(), s.vals.size() * sizeof(Val));
        }
        out += s.vals.size();
        if (out_len) {
          memcpy(out_len, s.lens.data(), s.lens.size() * sizeof(int));
          out_len += s.lens.size();
        }
      }
    }
    if (cb) cb();
  });

  KVPairs<Val> kvs;
  kvs.keys = keys;
  if (push_vals) {
    // fused push-pull: the request carries the values to push, the completion above stitches
    // the reply into *vals exactly as for a pull
    kvs.vals = *push_vals;
    if (lens && !lens->empty()) kvs.lens = kv_detail::ViewOf(lens);  // in: push lengths, out: pulled lengths
    const SArray<Val> dest = kv_detail::ViewOf(vals);
    Send(ts, true, cmd, kvs, opts, &dest);
    return ts;
  }
  // the destination is cut per server so that replies can land in place — possible when its
  // size says how many values each key has. A buffer merely pre-sized "large enough" (allowed:
  // only the front is written) does not: then the replies are gathered and stitched afterwards.
  const bool lens_known = lens && !lens->empty();
  if (lens_known || (keys.size() && vals->size() % keys.size() == 0)) kvs.vals = kv_detail::ViewOf(vals);
  if (lens_known) kvs.lens = kv_detail::ViewOf(lens);
  Send(ts, false, cmd, kvs, opts);
  return ts;
}

}  // namespace ps
#endif  // PS_KV_APP_H_
