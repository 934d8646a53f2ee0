/**
 * \file onesided_van.h
 * \brief OneSidedVan: push / pull payloads are *written into the receiver's
 *        memory by the sender*; only a small descriptor travels over TCP.
 *
 * This is the B200 counterpart of the reference's RDMA-class vans (RDMAVan
 * src/rdma_van.h:26-950 + RDMATransport src/rdma_transport.h:198-467, and the
 * CUDA-aware UCXVan src/ucx_van.h:874-1339): same protocol shape, different
 * fabric. Mapping:
 *   ibv_reg_mr / rkey            -> MemDomain::Export -> RegionDesc (CUDA IPC / shm)
 *   rendezvous start / reply     -> ADDR_REQUEST / ADDR_RESOLVED control messages,
 *                                   result cached per (peer, key)   [push landing slot]
 *   RDMA WRITE of the payload    -> MemDomain::CopyAsync: an sm_100a kernel storing
 *                                   straight into peer HBM over NVLink, optionally
 *                                   fused with scale / bf16 cast / fp8 block quant
 *   WRITE_WITH_IMM of the meta   -> the descriptor (Meta with MemRef): same-host peers get
 *                                   it in their shared-memory ring at once, GATED on a
 *                                   completion word the copy itself stores (PollCQ = the
 *                                   receiver polling that word); other peers get it over
 *                                   TCP after the copy's ticket completes
 *   zero-copy pull               -> the pull request carries the MemRef of the
 *                                   worker's destination tensor; the server's copy
 *                                   kernel writes the values there
 *   registered recv buffers      -> RegisterRecvBuffer'd SArrays become the landing
 *                                   slots (pointer identity preserved)
 *   IPCTransport (same host)     -> same-process peers skip IPC and use raw pointers
 * The TCP side (connection setup, control plane, CPU payloads) is inherited
 * from TcpVan. The memory backend is a MemDomain: CudaDomain ("nvl") or
 * ShmDomain ("shm", the GPU-less twin that keeps this protocol testable on CPU).
 */
#ifndef PS_VAN_ONESIDED_VAN_H_
#define PS_VAN_ONESIDED_VAN_H_
#include <chrono>
#include <condition_variable>
#include <deque>
#include <atomic>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <thread>
#include <tuple>
#include <utility>
#include <vector>

#include "core/nvtx.h"
#include "van/mem_domain.h"
#include "van/tcp_van.h"

namespace ps {

class OneSidedVan : public TcpVan {
 public:
  OneSidedVan(Postoffice* postoffice, MemDomain* domain, const std::string& type_name)
      : TcpVan(postoffice), domain_(domain), type_(type_name) {}
  ~OneSidedVan() override { StopCompleter(); }

  std::string GetType() const override { return type_; }

  void Start(int customer_id, bool standalone) override {
    {
      std::lock_guard<SpinMutex> lk(cq_mu_);
      if (!completer_) {
        cq_stop_ = false;
        completer_.reset(new std::thread(&OneSidedVan::CompletionLoop, this));
      }
    }
    TcpVan::Start(customer_id, standalone);
  }

  void Stop() override {
    StopCompleter();
    TcpVan::Stop();
    domain_->ReleaseNames();
    if (coalesce_) {
      PS_VLOG(1) << type_ << " van " << my_node_.id << ": " << coalesced_copies_.load() << " copies in "
                 << coalesced_batches_.load() << " coalesced batches";
    }
    PS_VLOG(1) << type_ << " van " << my_node_.id << ": " << copies_.load() << " one-sided copies, "
               << gated_frames_.load() << " descriptors gated by the copy engine";
    PS_VLOG(1) << type_ << " van: receive thread slept " << num_blocking_waits() << " times, " << num_deferred_sends()
               << " of its sends went through the outbox";
    std::lock_guard<SpinMutex> lk(rv_mu_);
    push_slots_.clear();
    landing_.clear();
    peer_regions_.clear();
    announced_.clear();
  }

  void SetNode(const Node& node) override {
    Node n = node;
    n.dev_id = domain_->device();
    Van::SetNode(n);
  }

  void RegisterRecvBuffer(Message& msg) override {
    CHECK_GE(msg.data.size(), (size_t)2);
    if (!domain_->Handles(msg.data[1].src_device_type_, msg.data[1].data())) {
      TcpVan::RegisterRecvBuffer(msg);  // plain host buffer: two-sided path
      return;
    }
    std::lock_guard<SpinMutex> lk(rv_mu_);
    registered_slots_[std::make_pair(msg.meta.sender, msg.meta.key)] = msg.data[1];
    registered_count_.store(static_cast<int>(registered_slots_.size()), std::memory_order_release);
  }

  /*!
   * \brief a node id that is connected AGAIN belongs to a NEW process: after a recovery the
   *        replacement takes over the dead node's id but brings its own regions and knows none of
   *        ours. Everything cached under that id — mappings of its regions (region ids start from
   *        0 again over there), the slots it granted, what we announced to it — is forgotten, or a
   *        pull reply would be written into the dead process's memory (the reference re-creates
   *        the endpoint and its memory-region tables on reconnect, src/rdma_van.h:759-777).
   */
  void Connect(const Node& node) override {
    if (HasPeer(node.id)) {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      const int id = node.id;
      for (auto it = peer_regions_.begin(); it != peer_regions_.end();) {
        it = it->first.first == id ? peer_regions_.erase(it) : std::next(it);
      }
      for (auto it = push_slots_.begin(); it != push_slots_.end();) {
        it = it->first.first == id ? push_slots_.erase(it) : std::next(it);
      }
      for (auto it = announced_.begin(); it != announced_.end();) {
        it = it->first == id ? announced_.erase(it) : std::next(it);
      }
    }
    // a peer on another host cannot map our memory, nor we its: everything for it travels in frames
    static const bool across = GetEnv("PS_ONESIDED_ACROSS_HOSTS", 0) != 0;  // (hosts sharing /dev/shm, for tests)
    if (node.id >= 0 && static_cast<size_t>(node.id) < kNegotiated) {
      negotiated_[node.id].store(false, std::memory_order_release);
    }
    if (node.id != my_node_.id) {
      const bool foreign = !across && !my_node_.hostname.empty() && node.hostname != my_node_.hostname;
      std::lock_guard<SpinMutex> lk(rv_mu_);
      if (foreign) {
        foreign_.insert(node.id);
        any_foreign_.store(true, std::memory_order_release);
      } else {
        foreign_.erase(node.id);
      }
    }
    TcpVan::Connect(node);
  }

  void PinMemory(void* addr, size_t /*length*/, bool /*gpu*/, int /*dev*/ = 0) override {
    RegionDesc d;
    if (domain_->Export(addr, &d)) RegionIdFor(&d);
  }

  void UnpinMemory(void* addr) override {
    RegionDesc d;
    if (!domain_->Export(addr, &d)) return;
    {
      // the region id stays reserved (peers may still hold its mapping) but is never handed out again:
      // the next export of this base gets a fresh id and a fresh announcement
      std::lock_guard<SpinMutex> lk(rv_mu_);
      region_of_base_.erase(d.base);
    }
    domain_->Unexport(d.base);
  }
  void* AllocExportable(size_t bytes) override { return domain_->Alloc(bytes); }
  void* AllocExportableOn(size_t bytes, int device) override { return domain_->AllocOn(bytes, device); }
  int NumDevices() override { return domain_->num_devices(); }
  void FreeExportable(void* p) override { domain_->Free(p); }
  void* DataStream() override { return domain_->Stream(); }

  bool AllocSymmetric(const std::string& tag, size_t bytes, SymmetricBuffer* out) override {
    // process-wide: the worker van and the server van of a joint process share ONE block
    // (a device joins a multicast team once, and both roles must see the same bytes)
    static std::mutex mu;
    static std::map<std::string, SymmetricBuffer> done;
    const int job_port = GetEnv("DMLC_PS_ROOT_PORT", 0);
    const std::string key = std::to_string(job_port) + "/" + type_ + "/" + tag;
    std::lock_guard<std::mutex> lk(mu);
    auto it = done.find(key);
    if (it != done.end()) {
      *out = it->second;
      return true;
    }
    // the participants: one entry per PROCESS that runs a worker or a server on this host, ordered by
    // its smallest node id (every process derives the same list from the scheduler's node table)
    std::vector<Node> nodes = ClusterNodes();
    std::sort(nodes.begin(), nodes.end(), [](const Node& a, const Node& b) { return a.id < b.id; });
    SymmetricGroup g;
    g.job_port = job_port;
    for (const Node& n : nodes) {
      if (n.hostname != my_node_.hostname || n.pid == 0) continue;
      if (std::find(g.pids.begin(), g.pids.end(), n.pid) == g.pids.end()) g.pids.push_back(n.pid);
    }
    const int me = static_cast<int>(getpid());
    for (size_t i = 0; i < g.pids.size(); ++i) {
      if (g.pids[i] == me) g.index = static_cast<int>(i);
    }
    if (g.index < 0) {
      LOG(WARNING) << type_ << " van: AllocSymmetric before the node table arrived (or from a process that is "
                   << "neither worker nor server)";
      return false;
    }
    if (!domain_->SymmetricAlloc(g, tag, bytes, out)) return false;
    for (const Node& n : nodes) {
      for (size_t i = 0; i < g.pids.size(); ++i) {
        if (n.hostname == my_node_.hostname && n.pid == g.pids[i]) out->node_member.emplace_back(n.id, static_cast<int>(i));
      }
    }
    done[key] = *out;
    PS_VLOG(1) << type_ << " van: symmetric buffer '" << tag << "' " << out->bytes << " B, member " << out->index
               << " of " << out->count << ", multicast " << (out->mc ? "yes" : "no");
    return true;
  }

  void TransportStats(std::vector<std::pair<std::string, uint64_t>>* out) override {
    uint64_t launches = 0, items = 0;
    domain_->EngineStats(&launches, &items);
    out->emplace_back("onesided_copies", copies_.load());
    out->emplace_back("onesided_bytes", copy_bytes_.load());
    out->emplace_back("gated_frames", gated_frames_.load());
    out->emplace_back("staged_copies", staged_copies_.load());
    out->emplace_back("push_slot_rendezvous", slot_rendezvous_.load());
    out->emplace_back("recv_thread_sleeps", num_blocking_waits());
    out->emplace_back("deferred_sends", num_deferred_sends());
    out->emplace_back("engine_launches", launches);
    out->emplace_back("engine_items", items);
  }
  MemDomain* domain() { return domain_.get(); }

  /*! \brief local address of `mem` inside a region node `peer` announced, or null */
  void* ResolvePeerMem(int peer, const MemRef& mem) override {
    std::lock_guard<SpinMutex> lk(rv_mu_);
    auto it = peer_regions_.find(std::make_pair(peer, mem.region));
    return it == peer_regions_.end() ? nullptr : it->second + mem.offset;
  }

  /*! \brief one-sided transfers issued / bytes moved (for tests and benchmarks) */
  uint64_t num_onesided_copies() const { return copies_.load(); }
  uint64_t onesided_bytes() const { return copy_bytes_.load(); }

 protected:
  int SendMsg(Message& msg) override {
    if (!msg.meta.control.empty() || msg.meta.simple_app) return TcpVan::SendMsg(msg);
    const bool has_vals = msg.data.size() >= 2 && msg.data[1].size() > 0;
    AwaitNegotiation(msg.meta.recver);
    if (any_foreign_.load(std::memory_order_acquire) && IsForeign(msg.meta.recver)) return SendTwoSided(msg, true);
    if (msg.meta.request && msg.meta.push && has_vals &&
        domain_->Handles(msg.data[1].src_device_type_, msg.data[1].data())) {
      return SendPush(msg);
    }
    if (msg.meta.request && !msg.meta.push && msg.meta.addr != 0 &&
        domain_->Handles(msg.meta.src_dev_type, reinterpret_cast<void*>(msg.meta.addr))) {
      // a caller-named destination (symmetric buffer) needs no export / announcement
      if (!msg.meta.mem.valid()) AttachPullDestination(&msg);
      if (msg.meta.mem.valid()) return Submit(msg, nullptr, false);
      return SendTwoSided(msg, false);  // memory that cannot be exported: the reply comes in a frame
    }
    if (!msg.meta.request && !msg.meta.push && msg.meta.mem.valid() && has_vals) {
      if (msg.meta.codec == kCodecPlaced) return SendPlacedResponse(msg);
      return SendPullResponse(msg);
    }
    if (msg.meta.request && msg.meta.push && msg.meta.pull && !msg.meta.pull_mem.valid() &&
        msg.meta.pull_addr != 0) {
      // fused push-pull whose values travel two-sided (e.g. a gradient tensor that cannot be
      // exported): the reply can still be written in place if its destination can
      const size_t esz = msg.meta.data_type.size() > 1 ? DataTypeSize(msg.meta.data_type[1]) : 1;
      DescribeDestination(msg.meta.recver, msg.meta.pull_addr,
                          static_cast<uint64_t>(msg.meta.pull_len) * esz, &msg.meta.pull_mem);
    }
    // nothing was placed one-sidedly: do not let the receiver rebuild a payload
    if (!msg.meta.request) msg.meta.mem = MemRef();
    if (!msg.meta.request && msg.meta.codec == kCodecPlaced) {
      // a value-less reply marked "placed" (e.g. the ack of a push whose slot a queued kernel
      // still reads): gate it on the work already enqueued on the data stream
      msg.meta.codec = kCodecRaw;
      MemDomain::CopyItem gate;
      gate.wait_event = msg.wait_event;
      return Submit(msg, &gate, true);
    }
    // whatever is left travels two-sided: device memory cannot ride in a frame, nor receive one
    return SendTwoSided(msg, false);
  }

  /*! \brief a descriptor handed over in-process still has to be turned into its payload view */
  void OnLocalDeliver(Message* msg) override {
    if (msg->meta.control.empty() && !msg->meta.simple_app && msg->meta.mem.valid()) RebuildPayload(msg);
  }

  /*! \brief rendezvous messages of an in-process peer are served on the caller's thread */
  bool OnLocalControl(Message* msg) override {
    if (msg->meta.control.cmd == Control::ADDR_REQUEST) {
      OnSlotRequest(*msg);
      return true;
    }
    if (msg->meta.control.cmd == Control::ADDR_RESOLVED) {
      OnRegionMessage(*msg);
      return true;
    }
    return false;
  }

  int RecvMsg(Message* msg) override {
    for (;;) {
      const int n = TcpVan::RecvMsg(msg);
      if (n < 0) return n;
      const auto cmd = msg->meta.control.cmd;
      if (cmd == Control::ADDR_REQUEST) {
        OnSlotRequest(*msg);
        continue;
      }
      if (cmd == Control::ADDR_RESOLVED) {
        OnRegionMessage(*msg);
        continue;
      }
      if (msg->meta.control.empty() && !msg->meta.simple_app && msg->meta.mem.valid()) {
        RebuildPayload(msg);
      } else if (staged_pulls_pending_.load(std::memory_order_acquire) > 0 && msg->meta.control.empty() &&
                 !msg->meta.simple_app && !msg->meta.request && !msg->meta.push) {
        LandStagedPull(msg);
      } else if (registered_count_.load(std::memory_order_acquire) > 0 && msg->meta.control.empty() &&
                 !msg->meta.simple_app && msg->meta.request && msg->meta.push) {
        LandInRegisteredBuffer(msg);
      }
      return n;
    }
  }

 private:
  struct Slot {
    char* ptr = nullptr;      // address usable by this process (local or peer-mapped)
    uint64_t capacity = 0;
    int32_t region = -1;      // id in the owner's table
    uint64_t offset = 0;
  };
  using PeerKey = std::pair<int, uint64_t>;

  /*! \brief a slot more than 1.5x (+4 KB) larger than what is pushed now is re-made to size */
  static bool Oversized(uint64_t capacity, uint64_t bytes) {
    return capacity > bytes + bytes / 2 + 4096;
  }

  static size_t DataTypeSize(DataType t) {
    switch (t) {
      case INT16: case UINT16: return 2;
      case INT32: case UINT32: case FLOAT: return 4;
      case INT64: case UINT64: case DOUBLE: return 8;
      default: return 1;
    }
  }

  // -- peers on other hosts: two-sided, device memory staged through the host ------------------

  /*! \brief a same-host peer could not map our ring, or we could not map its ring: no shared memory */
  void OnPipeVerdict(int peer_id, bool accepted) override {
    if (accepted) return;
    std::lock_guard<SpinMutex> lk(rv_mu_);
    foreign_.insert(peer_id);
    any_foreign_.store(true, std::memory_order_release);
  }

  /*!
   * \brief before the first data message for a peer: wait until the ring negotiation with it has a
   *        verdict (milliseconds at start-up; bounded, because a peer configured without rings never
   *        offers one). Afterwards `foreign_` says whether the peer shares memory with us.
   */
  void AwaitNegotiation(int recver) {
    const size_t slot = static_cast<size_t>(recver);
    if (slot < kNegotiated && negotiated_[slot].load(std::memory_order_acquire)) return;
    // the receive thread is the one that processes offers and answers: it cannot wait for them. What it
    // sends are replies, and a reply that cannot travel one-sidedly is staged into a frame (SendTwoSided).
    if (OnReceiveThread()) return;
    static const int limit_ms = GetEnv("PS_NEGOTIATION_TIMEOUT_MS", 3000);
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::milliseconds(limit_ms);
    while (NegotiationOpen(recver) && std::chrono::steady_clock::now() < deadline) {
      std::this_thread::sleep_for(std::chrono::microseconds(200));
    }
    if (slot < kNegotiated) negotiated_[slot].store(true, std::memory_order_release);
  }

  bool IsForeign(int node_id) {
    std::lock_guard<SpinMutex> lk(rv_mu_);
    return foreign_.count(node_id) > 0;
  }

  /*!
   * \brief send `msg` two-sided (its payload inside the frame): the peer lives on another host
   *        (`foreign`: nothing can be written into its memory, every MemRef is dropped), or this
   *        particular message cannot go one-sidedly (memory that cannot be exported, a request that
   *        named no destination). Values in device memory are copied to the host first; the
   *        destination of a pull that lies in device memory and is not described by a MemRef is
   *        remembered, and the reply is copied into it on arrival (LandStagedPull). The reference's
   *        vans do the same whenever the fabric cannot reach the memory (ZMQ van for CPU tensors,
   *        UCX without GPUDirect).
   */
  int SendTwoSided(Message& msg, bool foreign) {
    if (foreign) {
      msg.meta.mem = MemRef();
      msg.meta.pull_mem = MemRef();
    }
    if (msg.meta.request) {
      const bool fused = msg.meta.push && msg.meta.pull;
      const bool described = fused ? msg.meta.pull_mem.valid() : msg.meta.mem.valid();
      const uint64_t addr = fused ? msg.meta.pull_addr : (msg.meta.push ? 0 : msg.meta.addr);
      // (a fused push-pull does not tag its destination: it lives where the pushed values live)
      const int dev_type = fused && msg.data.size() >= 2 ? msg.data[1].src_device_type_ : msg.meta.src_dev_type;
      const int dev_id = fused && msg.data.size() >= 2 ? msg.data[1].src_device_id_ : msg.meta.src_dev_id;
      if (!described && addr != 0 && domain_->NeedsStaging(dev_type, reinterpret_cast<void*>(addr))) {
        const size_t esz = msg.meta.data_type.size() > 1 ? DataTypeSize(msg.meta.data_type[1]) : 1;
        StagedPull rec;
        rec.addr = addr;
        rec.bytes = static_cast<uint64_t>(fused ? msg.meta.pull_len : msg.meta.val_len) * esz;
        rec.dev_type = dev_type;
        rec.dev_id = dev_id;
        {
          std::lock_guard<SpinMutex> lk(rv_mu_);
          if (staged_pulls_.size() >= (1u << 16)) staged_pulls_.erase(staged_pulls_.begin());
          staged_pulls_[std::make_tuple(msg.meta.recver, msg.meta.app_id, msg.meta.customer_id,
                                        msg.meta.timestamp)] = rec;
          staged_pulls_pending_.store(static_cast<int>(staged_pulls_.size()), std::memory_order_release);
        }
        // the address means nothing to the peer, and no socket may land bytes at it over here
        if (fused) msg.meta.pull_addr = 0; else msg.meta.addr = 0;
      }
    }
    if (msg.data.size() >= 2 && msg.data[1].size() > 0 &&
        domain_->NeedsStaging(msg.data[1].src_device_type_, msg.data[1].data())) {
      const SArray<char>& dev = msg.data[1];
      SArray<char> host(dev.size());
      domain_->CopyToHost(host.data(), dev.data(), dev.size(), msg.wait_event);
      host.src_device_type_ = CPU;
      host.src_device_id_ = 0;
      host.dst_device_type_ = dev.dst_device_type_;
      host.dst_device_id_ = dev.dst_device_id_;
      msg.data[1] = host;
      msg.wait_event = nullptr;
      ++staged_copies_;
    }
    if (!msg.meta.request && msg.meta.codec == kCodecPlaced) msg.meta.codec = kCodecRaw;
    return Submit(msg, nullptr, false);
  }

  /*! \brief a pull reply arrived in host memory (frame): copy it to the device destination its request named */
  void LandStagedPull(Message* msg) {
    if (msg->data.size() < 2 || msg->data[1].size() == 0) return;
    StagedPull rec;
    {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      auto it = staged_pulls_.find(std::make_tuple(msg->meta.sender, msg->meta.app_id, msg->meta.customer_id,
                                                   msg->meta.timestamp));
      if (it == staged_pulls_.end()) return;
      rec = it->second;
      staged_pulls_.erase(it);
      staged_pulls_pending_.store(static_cast<int>(staged_pulls_.size()), std::memory_order_release);
    }
    const SArray<char>& got = msg->data[1];
    CHECK_LE(got.size(), rec.bytes) << "pull reply larger than the destination it was requested for";
    domain_->CopyFromHost(reinterpret_cast<void*>(rec.addr), got.data(), got.size());
    SArray<char> placed;
    placed.reset(reinterpret_cast<char*>(rec.addr), got.size(), [](char*) {}, static_cast<DeviceType>(rec.dev_type),
                 rec.dev_id, static_cast<DeviceType>(rec.dev_type), rec.dev_id);
    msg->data[1] = placed;
    ++staged_copies_;
  }

  /*!
   * \brief a push arrived IN a frame (its sender is on another host, or could not go one-sidedly) for a
   *        (sender, key) the application registered a receive buffer for: the contract is that the
   *        handler sees the values in THAT buffer (KVServer::RegisterRecvBuffer, reference
   *        src/rdma_van.h:293-319), so they are copied there — host to device if the buffer is in HBM.
   */
  void LandInRegisteredBuffer(Message* msg) {
    if (msg->data.size() < 2 || msg->data[1].size() == 0) return;
    SArray<char> reg;
    {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      auto it = registered_slots_.find(std::make_pair(msg->meta.sender, static_cast<uint64_t>(msg->meta.key)));
      if (it == registered_slots_.end()) return;
      reg = it->second;
    }
    const SArray<char>& got = msg->data[1];
    if (got.data() == reg.data() || got.size() > reg.size() || got.on_gpu()) return;
    if (domain_->NeedsStaging(reg.src_device_type_, reg.data())) {
      domain_->CopyFromHost(reg.data(), got.data(), got.size());
      ++staged_copies_;
    } else {
      memcpy(reg.data(), got.data(), got.size());
    }
    msg->data[1] = reg.segment(0, got.size());
  }

  // -- region bookkeeping -----------------------------------------------------

  /*! \brief id of the exported region with d->base (assigned on first sight); fills d */
  int32_t RegionIdFor(RegionDesc* d) {
    std::lock_guard<SpinMutex> lk(rv_mu_);
    auto it = region_of_base_.find(d->base);
    if (it == region_of_base_.end()) {
      const int32_t id = static_cast<int32_t>(my_regions_.size());
      d->region = id;
      d->owner = my_node_.id;
      strncpy(d->host, my_node_.hostname.c_str(), sizeof(d->host) - 1);
      my_regions_.push_back(*d);
      region_of_base_[d->base] = id;
      return id;
    }
    *d = my_regions_[it->second];
    d->owner = my_node_.id;
    return it->second;
  }

  char* ImportPeerRegion(int peer, const RegionDesc& d) {
    {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      auto it = peer_regions_.find(std::make_pair(peer, d.region));
      if (it != peer_regions_.end()) return it->second;
    }
    char* base = static_cast<char*>(domain_->Import(d));
    std::lock_guard<SpinMutex> lk(rv_mu_);
    peer_regions_[std::make_pair(peer, d.region)] = base;
    return base;
  }

  // -- push: sender side -------------------------------------------------------

  int SendPush(Message& msg) {
    NvtxRange nvtx("ps.push");
    const int recver = msg.meta.recver;
    const SArray<char>& vals = msg.data[1];
    const uint64_t wire = WireBytes(msg.meta.codec, vals.size());
    Slot slot;
    if (msg.meta.mem.region == kSymmetricRegion) {
      // symmetric push: encode into the sender's OWN copy of the job-wide buffer; the
      // receiver reads every worker's copy at this offset through the multicast mapping
      CHECK(msg.stage != nullptr) << "symmetric push without a staging address";
      slot.ptr = static_cast<char*>(msg.stage);
      slot.region = kSymmetricRegion;
      slot.offset = msg.meta.mem.offset;
    } else {
      slot = AcquirePushSlot(recver, msg.meta.key, wire, vals.dst_device_type_ == GPU ? vals.dst_device_id_ : -1,
                             msg.slot_bytes);
    }
    MemDomain::CopyItem item;
    item.dst = slot.ptr;
    item.src = vals.data();
    item.n_src_bytes = vals.size();
    item.codec = msg.meta.codec;
    item.scale = msg.meta.scale;
    item.wait_event = msg.wait_event;
    item.src_device_type = vals.src_device_type_;
    item.src_device_id = vals.src_device_type_ == GPU ? vals.src_device_id_ : -1;
    ++copies_;
    copy_bytes_ += wire;
    Message desc;
    desc.meta = msg.meta;
    desc.meta.mem.region = slot.region;
    desc.meta.mem.offset = slot.offset;
    desc.meta.mem.bytes = wire;
    if (msg.meta.pull && !msg.meta.pull_mem.valid() && msg.meta.pull_addr != 0) {
      // fused push-pull: tell the server where the reply goes, as a pull request would
      const size_t esz = msg.meta.data_type.size() > 1 ? DataTypeSize(msg.meta.data_type[1]) : 1;
      DescribeDestination(recver, msg.meta.pull_addr, static_cast<uint64_t>(msg.meta.pull_len) * esz,
                          &desc.meta.pull_mem);
    }
    desc.data = msg.data;
    desc.data[1] = vals.segment(0, 0);  // payload already placed; keep the segment slot
    desc.meta.data_size = msg.meta.data_size - static_cast<int64_t>(vals.size());
    // keep the source alive until the copy has completed
    return Submit(desc, &item, false, vals) + static_cast<int>(std::min<uint64_t>(wire, 0x3fffffff));
  }

  /*!
   * \brief landing slot at `recver` for `key`; rendezvous on first use or growth. With `slot_bytes`
   *        (SendOpts::slot_bytes) the slot is requested at that capacity and kept while pushes fit.
   */
  Slot AcquirePushSlot(int recver, uint64_t key, uint64_t bytes, int dst_device = -1, uint64_t slot_bytes = 0) {
    std::unique_lock<SpinMutex> lk(rv_mu_);
    const PeerKey pk(recver, key);
    auto it = push_slots_.find(pk);
    if (it != push_slots_.end() && it->second.capacity >= bytes &&
        (slot_bytes != 0 || !Oversized(it->second.capacity, bytes))) {
      return it->second;
    }
    bytes = std::max(bytes, slot_bytes);
    ++slot_rendezvous_;
    push_slots_.erase(pk);  // too small, or far too large (e.g. bf16 init, then fp8 gradients)
    lk.unlock();
    Message req;
    req.meta.recver = recver;
    req.meta.request = true;
    req.meta.control.cmd = Control::ADDR_REQUEST;
    req.meta.key = key;
    req.meta.val_len = static_cast<int64_t>(bytes);
    req.meta.dst_dev_id = dst_device;  // a receiver that drives several devices cuts the slot on this one
    req.meta.timestamp = GetTimestamp();
    CHECK_GT(TcpVan::SendMsg(req), 0);
    lk.lock();
    // bounded: a receiver that never answers (dead, or out of memory for the slot) must not hang the
    // sender forever. PS_RENDEZVOUS_TIMEOUT_S (default 300, 0 = wait for ever) — past it the push
    // fails loudly (dmlc::Error from CHECK), which the application can catch and act upon.
    static const int limit_s = GetEnv("PS_RENDEZVOUS_TIMEOUT_S", 300);
    int waited_s = 0;
    while (!rv_cv_.wait_for(lk, std::chrono::seconds(30), [&] { return push_slots_.count(pk) > 0; })) {
      waited_s += 30;
      LOG(WARNING) << type_ << " van " << my_node_.id << ": no landing slot from node " << recver
                   << " for key " << key << " (" << bytes << " B) after " << waited_s << " s";
      CHECK(limit_s <= 0 || waited_s < limit_s)
          << type_ << " van " << my_node_.id << ": node " << recver << " never granted a landing slot for key "
          << key << " (" << bytes << " B): giving up after " << waited_s << " s (PS_RENDEZVOUS_TIMEOUT_S)";
    }
    return push_slots_[pk];
  }

  // -- push: receiver side -----------------------------------------------------

  void OnSlotRequest(const Message& req) {
    const int sender = req.meta.sender;
    const uint64_t key = req.meta.key;
    const uint64_t bytes = static_cast<uint64_t>(req.meta.val_len);
    const PeerKey pk(sender, key);
    char* ptr = nullptr;
    uint64_t cap = 0;
    {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      auto reg = registered_slots_.find(pk);
      auto have = landing_.find(pk);
      if (reg != registered_slots_.end()) {
        CHECK_GE(reg->second.size(), bytes) << "registered buffer smaller than the push";
        ptr = reg->second.data();
        cap = reg->second.size();
      } else if (have != landing_.end() && have->second.second >= bytes &&
                 !Oversized(have->second.second, bytes)) {
        ptr = have->second.first;
        cap = have->second.second;
      } else if (have != landing_.end()) {
        // wrong size: give the old slot back (Free synchronises with kernels still reading it)
        domain_->Free(have->second.first);
        landing_.erase(have);
      }
    }
    if (!ptr) {
      cap = AlignUp(bytes, 256);
      const int want_dev = req.meta.dst_dev_id;
      ptr = static_cast<char*>(want_dev >= 0 && domain_->num_devices() > 1 ? domain_->AllocOn(cap, want_dev)
                                                                           : domain_->Alloc(cap));
      CHECK(ptr) << "out of " << domain_->name() << " memory for a " << cap << " B landing slot";
    }
    RegionDesc d;
    CHECK(domain_->Export(ptr, &d)) << "landing slot is not exportable";
    RegionIdFor(&d);
    {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      landing_[pk] = std::make_pair(ptr, cap);
    }
    Message rep;
    rep.meta.recver = sender;
    rep.meta.request = false;
    rep.meta.control.cmd = Control::ADDR_RESOLVED;
    rep.meta.head = kReplySlot;
    rep.meta.key = key;
    rep.meta.val_len = static_cast<int64_t>(cap);
    rep.meta.addr = reinterpret_cast<uint64_t>(ptr) - d.base;  // offset inside the region
    rep.meta.body = d.Serialize();
    rep.meta.timestamp = GetTimestamp();
    CHECK_GT(TcpVan::SendMsg(rep), 0);
  }

  /*! \brief ADDR_RESOLVED: either a slot reply or a region announcement */
  void OnRegionMessage(const Message& m) {
    RegionDesc d;
    CHECK(RegionDesc::Parse(m.meta.body, 0, &d)) << "malformed region descriptor";
    char* base = ImportPeerRegion(m.meta.sender, d);
    if (m.meta.head == kReplySlot) {
      Slot s;
      s.ptr = base + m.meta.addr;
      s.capacity = static_cast<uint64_t>(m.meta.val_len);
      s.region = d.region;
      s.offset = m.meta.addr;
      {
        std::lock_guard<SpinMutex> lk(rv_mu_);
        push_slots_[PeerKey(m.meta.sender, m.meta.key)] = s;
      }
      rv_cv_.notify_all();
    }
  }

  // -- pull ----------------------------------------------------------------------

  /*!
   * \brief describe [addr, addr+bytes) of this process so that `recver` can write into it:
   *        export the containing allocation (announcing it to that peer once) and fill `out`.
   *        False if the memory cannot be exported (the reply then travels two-sided).
   */
  bool DescribeDestination(int recver, uint64_t addr, uint64_t bytes, MemRef* out) {
    RegionDesc d;
    if (!domain_->Export(reinterpret_cast<void*>(addr), &d)) return false;
    const int32_t id = RegionIdFor(&d);
    bool known = false;
    {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      known = announced_.count(std::make_pair(recver, id)) > 0;
    }
    if (!known) {
      // the announcement must be in the peer's ring BEFORE any request that names the region — also
      // a request of another application thread that finds the region "already announced": the
      // entry is made only after the send, under a lock that serialises announcers
      std::lock_guard<std::mutex> alk(announce_mu_);
      bool still_unknown;
      {
        std::lock_guard<SpinMutex> lk(rv_mu_);
        still_unknown = announced_.count(std::make_pair(recver, id)) == 0;
      }
      if (still_unknown) {
        Message ann;
        ann.meta.recver = recver;
        ann.meta.request = true;
        ann.meta.control.cmd = Control::ADDR_RESOLVED;
        ann.meta.head = kAnnounceRegion;
        ann.meta.body = d.Serialize();
        ann.meta.timestamp = GetTimestamp();
        CHECK_GT(TcpVan::SendMsg(ann), 0);
        std::lock_guard<SpinMutex> lk(rv_mu_);
        announced_.insert(std::make_pair(recver, id));
      }
    }
    out->region = id;
    out->offset = addr - d.base;
    out->bytes = bytes;
    return true;
  }

  /*! \brief name the pull destination so the server can write into it */
  void AttachPullDestination(Message* msg) {
    const size_t esz = msg->meta.data_type.size() > 1 ? DataTypeSize(msg->meta.data_type[1]) : 1;
    DescribeDestination(msg->meta.recver, msg->meta.addr,
                        static_cast<uint64_t>(msg->meta.val_len) * esz, &msg->meta.mem);
  }

  int SendPullResponse(Message& msg) {
    NvtxRange nvtx("ps.pull_reply");
    const int recver = msg.meta.recver;
    char* base = nullptr;
    {
      std::lock_guard<SpinMutex> lk(rv_mu_);
      auto it = peer_regions_.find(std::make_pair(recver, msg.meta.mem.region));
      CHECK(it != peer_regions_.end()) << "pull destination region " << msg.meta.mem.region
                                       << " of node " << recver << " was never announced";
      base = it->second;
    }
    const SArray<char>& vals = msg.data[1];
    const uint64_t wire = WireBytes(msg.meta.codec, vals.size());
    if (msg.meta.mem.bytes) {
      CHECK_LE(wire, msg.meta.mem.bytes) << "pull response larger than the destination";
    }
    MemDomain::CopyItem item;
    item.dst = base + msg.meta.mem.offset;
    item.src = vals.data();
    item.n_src_bytes = vals.size();
    item.codec = msg.meta.codec;
    item.scale = msg.meta.scale;
    item.wait_event = msg.wait_event;
    item.src_device_type = vals.src_device_type_;
    item.src_device_id = -1;  // a landing slot or a store: the domain finds the device by address
    ++copies_;
    copy_bytes_ += wire;
    Message desc;
    desc.meta = msg.meta;
    desc.meta.mem.bytes = wire;
    desc.data = msg.data;
    desc.data[1] = vals.segment(0, 0);
    desc.meta.data_size = msg.meta.data_size - static_cast<int64_t>(vals.size());
    return Submit(desc, &item, false, vals) + static_cast<int>(std::min<uint64_t>(wire, 0x3fffffff));
  }

  /*!
   * \brief the application already wrote the values into the destination (e.g. the
   *        fused update kernel stores the new parameters straight into every
   *        worker's buffer); only gate the descriptor on `wait_event`.
   */
  int SendPlacedResponse(Message& msg) {
    MemDomain::CopyItem gate;  // no bytes to move: only wait for the stream (and the event)
    gate.wait_event = msg.wait_event;
    Message desc;
    desc.meta = msg.meta;
    desc.meta.codec = kCodecRaw;
    desc.meta.mem.bytes = msg.data[1].size();
    desc.data = msg.data;
    desc.data[1] = msg.data[1].segment(0, 0);
    desc.meta.data_size = msg.meta.data_size - static_cast<int64_t>(msg.data[1].size());
    return Submit(desc, &gate, true);
  }

  // -- receive-side payload reconstruction -----------------------------------------

  void RebuildPayload(Message* msg) {
    const MemRef& mem = msg->meta.mem;
    char* ptr = nullptr;
    if (msg->meta.request && msg->meta.push) {
      if (mem.region == kSymmetricRegion) return;  // the handler resolves the offset itself
      std::lock_guard<SpinMutex> lk(rv_mu_);
      CHECK_LT(static_cast<size_t>(mem.region), my_regions_.size());
      ptr = reinterpret_cast<char*>(my_regions_[mem.region].base + mem.offset);
    } else if (!msg->meta.request && !msg->meta.push) {
      ptr = reinterpret_cast<char*>(msg->meta.addr);
    } else {
      return;  // pull request: the MemRef is for the handler, there is no payload
    }
    if (msg->data.size() < 2) return;  // e.g. an empty ack that merely echoes the MemRef
    const int dev = domain_->device();
    SArray<char> vals;
    vals.reset(ptr, mem.bytes, [](char*) {}, dev >= 0 ? GPU : CPU, dev >= 0 ? dev : 0,
               dev >= 0 ? GPU : CPU, dev >= 0 ? dev : 0);
    msg->data[1] = vals;
    msg->meta.data_size += static_cast<int64_t>(mem.bytes);
  }

  // -- ordered, completion-gated descriptor sends -----------------------------------

  struct Pending {
    Message msg;
    Ticket ticket;
    SArray<char> keep_alive;
  };

  // -- launch coalescing ------------------------------------------------------------------

  struct Held {
    Message msg;
    SArray<char> keep_alive;
  };
  struct CorkState {
    int depth = 0;
    bool gate = false;  // some message must wait for the data stream even without a copy
    std::vector<MemDomain::CopyItem> items;
    std::vector<Held> held;
  };
  /*! \brief this thread's cork on this van */
  CorkState& MyCork() {
    thread_local std::map<const OneSidedVan*, CorkState> per_van;
    return per_van[this];
  }

  /*!
   * \brief the one way out for data messages: `item` (may be null) is the copy that must
   *        complete before `msg` may leave; `gate_only` marks an item that moves no bytes.
   *        Corked: remember both; otherwise issue the copy now and queue the message behind it.
   */
  int Submit(Message& msg, const MemDomain::CopyItem* item, bool gate_only,
             const SArray<char>& keep_alive = SArray<char>()) {
    if (coalesce_) {
      CorkState& c = MyCork();
      if (c.depth > 0) {
        if (item && !gate_only) c.items.push_back(*item);
        if (item && gate_only) {
          c.gate = true;
          if (item->wait_event) c.items.push_back(*item);  // zero bytes: only its event matters
        }
        Held h;
        h.msg = msg;
        h.keep_alive = keep_alive;
        c.held.push_back(std::move(h));
        return 1 + static_cast<int>(msg.meta.data_size & 0x3fffffff);
      }
    }
    if (signal_ && PeerGated(msg.meta.recver)) {
      // this peer's ring was accepted only a moment ago and earlier messages for it may still sit in
      // the completion queue (ticket path): they must leave first, or a pull could overtake its push
      std::atomic<int>& in_flight = TicketsFor(msg.meta.recver);
      while (in_flight.load(std::memory_order_acquire) != 0) std::this_thread::yield();
      // same-host peer with a descriptor ring: the frame goes into the ring NOW and the copy
      // kernel itself opens its gate (st.release.sys on the ring's completion word) — no event,
      // no completion thread, no second hop for the descriptor. Frames without a copy simply
      // queue behind the gated ones in the ring, which keeps the order of the SendMsg calls.
      if (!item) return TcpVan::SendMsg(msg);  // (encodes host-resident values that asked for a wire codec)
      MemDomain::CopyItem it = *item;
      if (gate_only) it.n_src_bytes = 0;
      const GateIssue issue = [this, &it](void* word, uint64_t seq) { return domain_->CopySignal(it, word, seq); };
      const int rc = TcpVan::SendFrame(msg, &issue, &keep_alive);
      CHECK_NE(rc, kNotGated) << type_ << " van: the copy engine refused to signal a gated frame";
      ++gated_frames_;
      return rc;
    }
    Ticket t;
    if (item) {
      t = domain_->CopyAsync(item->dst, item->src, gate_only ? 0 : item->n_src_bytes, item->codec,
                             item->scale, item->wait_event, item->src_device_type);
    }
    return Ordered(msg, t, keep_alive);
  }

  void* MapGateWord(ShmPipe* pipe) override {
    if (!signal_) return nullptr;
    return domain_->MapSignalWord(pipe->map_base(), 4096, pipe->gate_word());
  }
  void ReleaseGateWord(ShmPipe* pipe) override { domain_->UnmapSignalWord(pipe->map_base()); }

 public:
  void Cork() override {
    if (coalesce_) ++MyCork().depth;
  }
  void Uncork() override {
    if (!coalesce_) return;
    CorkState& c = MyCork();
    if (c.depth == 0 || --c.depth > 0) return;
    if (c.held.empty()) return;
    NvtxRange nvtx("ps.uncork");
    Ticket t;
    if (!c.items.empty() || c.gate) {
      t = domain_->CopyBatchAsync(c.items);
      ++coalesced_batches_;
      coalesced_copies_ += c.items.size();
    }
    // the first message carries the ticket; the queue is FIFO, so the others (and their
    // keep-alive references) follow it out only after the whole batch has completed
    for (size_t i = 0; i < c.held.size(); ++i) {
      Ordered(c.held[i].msg, i == 0 ? t : Ticket(), c.held[i].keep_alive);
    }
    c.items.clear();
    c.held.clear();
    c.gate = false;
  }
  /*! \brief descriptors whose delivery was gated on a completion signalled by the copy engine */
  uint64_t num_gated_frames() const { return gated_frames_.load(); }
  /*! \brief batches flushed by Uncork / copies that shared a batch (tests, benchmarks) */
  uint64_t num_coalesced_batches() const { return coalesced_batches_.load(); }
  uint64_t num_coalesced_copies() const { return coalesced_copies_.load(); }

 private:
  /*!
   * \brief send `msg` after `t` completes, preserving the order of SendMsg calls.
   *        With nothing in flight and no ticket the send happens inline.
   */
  int Ordered(Message& msg, Ticket t, const SArray<char>& keep_alive = SArray<char>()) {
    {
      std::lock_guard<SpinMutex> lk(cq_mu_);
      if (t.event != nullptr || !cq_.empty() || cq_busy_) {
        Pending p;
        p.msg = msg;
        p.ticket = t;
        p.keep_alive = keep_alive;
        TicketsFor(msg.meta.recver).fetch_add(1, std::memory_order_acq_rel);
        cq_.push_back(std::move(p));
        cq_size_.fetch_add(1, std::memory_order_release);
        cq_cv_.notify_one();
        return 1 + static_cast<int>(msg.meta.data_size & 0x3fffffff);
      }
    }
    return TcpVan::SendMsg(msg);
  }

  void CompletionLoop() {
    std::unique_lock<SpinMutex> lk(cq_mu_);
    std::vector<Pending> batch;
    // a sleeping thread takes 100+ us to come back on a virtual machine: between the bursts of a
    // round stay on the CPU as long as the recent gaps suggest before giving it up
    SpinBudget budget(GetEnv("PS_QUEUE_SPIN_US", 20), GetEnv("PS_SPIN_MAX_US", 1000));
    for (;;) {
      const auto t0 = std::chrono::steady_clock::now();
      const bool was_idle = cq_.empty();
      if (was_idle && !cq_stop_) {
        lk.unlock();
        SpinPoll([this] { return cq_size_.load(std::memory_order_acquire) != 0; }, budget.floor_us(),
                 budget.window_us());
        lk.lock();
      }
      cq_cv_.wait(lk, [this] { return cq_stop_ || !cq_.empty(); });
      if (cq_.empty()) {
        if (cq_stop_) return;
        continue;
      }
      if (was_idle) {
        budget.Observe(
            std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count());
      }
      batch.clear();
      batch.push_back(std::move(cq_.front()));
      cq_.pop_front();
      cq_size_.fetch_sub(1, std::memory_order_release);
      cq_busy_ = true;
      lk.unlock();
      domain_->Wait(batch[0].ticket);  // payload is globally visible after this
      // everything queued behind it whose copy has also finished leaves in the same flush:
      // one sendmsg per peer instead of one per descriptor
      lk.lock();
      while (!cq_.empty() && batch.size() < 48 && domain_->Ready(cq_.front().ticket)) {
        batch.push_back(std::move(cq_.front()));
        cq_.pop_front();
        cq_size_.fetch_sub(1, std::memory_order_release);
      }
      lk.unlock();
      for (size_t i = 1; i < batch.size(); ++i) domain_->Wait(batch[i].ticket);  // recycle tickets
      if (batch.size() == 1) {
        if (TcpVan::SendMsg(batch[0].msg) < 0) {
          LOG(WARNING) << "failed to send descriptor: " << batch[0].msg.DebugString();
        }
      } else {
        // group by peer, preserving the per-peer order
        std::map<int, std::vector<Message*>> per_peer;
        for (Pending& p : batch) per_peer[p.msg.meta.recver].push_back(&p.msg);
        for (auto& kv : per_peer) {
          if (TcpVan::SendMsgBatch(kv.first, kv.second) < 0) {
            LOG(WARNING) << "failed to send " << kv.second.size() << " descriptors to node "
                         << kv.first;
          }
        }
      }
      for (Pending& p : batch) {
        TicketsFor(p.msg.meta.recver).fetch_sub(1, std::memory_order_acq_rel);
      }
      batch.clear();  // drops the keep-alive references
      lk.lock();
      cq_busy_ = false;
    }
  }

  void StopCompleter() {
    std::unique_ptr<std::thread> t;
    {
      std::lock_guard<SpinMutex> lk(cq_mu_);
      cq_stop_ = true;
      t.swap(completer_);
    }
    cq_cv_.notify_all();
    if (t) t->join();
  }

  enum { kReplySlot = 1, kAnnounceRegion = 2 };

  std::unique_ptr<MemDomain> domain_;
  std::string type_;

  std::mutex announce_mu_;  // serialises region announcements (see DescribeDestination)
  SpinMutex rv_mu_;  // slot / region tables: looked up on every push, pull reply and received descriptor
  std::condition_variable_any rv_cv_;
  std::map<PeerKey, Slot> push_slots_;                          // sender: where my pushes land
  std::map<PeerKey, std::pair<char*, uint64_t>> landing_;       // receiver: slots I handed out
  std::map<PeerKey, SArray<char>> registered_slots_;            // receiver: user-registered
  std::vector<RegionDesc> my_regions_;                          // regions I exported, by id
  std::map<uint64_t, int32_t> region_of_base_;
  std::map<std::pair<int, int32_t>, char*> peer_regions_;       // (peer, region) -> mapping
  std::set<std::pair<int, int32_t>> announced_;                 // (peer, my region) announced
  /*! \brief peers on other hosts, the device destinations of pulls sent to them, staging copies made */
  struct StagedPull {
    uint64_t addr = 0;
    uint64_t bytes = 0;
    int dev_type = UNK;
    int dev_id = 0;
  };
  std::set<int> foreign_;
  static constexpr size_t kNegotiated = 4096;
  std::atomic<bool> negotiated_[kNegotiated] = {};  // by node id: the first data message has waited for the verdict
  std::atomic<bool> any_foreign_{false};
  std::map<std::tuple<int, int, int, int>, StagedPull> staged_pulls_;
  std::atomic<int> staged_pulls_pending_{0};
  std::atomic<int> registered_count_{0};  // size of registered_slots_ (checked without the lock per frame)
  std::atomic<uint64_t> staged_copies_{0};
  std::atomic<uint64_t> slot_rendezvous_{0};  // ADDR_REQUESTs sent for push landing slots

  SpinMutex cq_mu_;
  std::condition_variable_any cq_cv_;
  std::atomic<int> cq_size_{0};  // lets the idle completer poll without the lock
  std::deque<Pending> cq_;
  bool cq_stop_ = false;
  bool cq_busy_ = false;
  std::unique_ptr<std::thread> completer_;

  /*! \brief descriptors queued on the ticket path and not yet sent, by receiver id modulo the table
   *  size (a collision only makes a gated send wait a little longer than it has to) */
  static constexpr size_t kTicketSlots = 256;
  std::atomic<int> tickets_in_flight_[kTicketSlots] = {};
  std::atomic<int>& TicketsFor(int recver) { return tickets_in_flight_[static_cast<size_t>(recver) % kTicketSlots]; }
  std::atomic<uint64_t> copies_{0};
  std::atomic<uint64_t> copy_bytes_{0};
  /*! \brief PS_COALESCE_LAUNCHES: honour Cork / Uncork (off: every copy is its own launch) */
  bool coalesce_ = GetEnv("PS_COALESCE_LAUNCHES", 0) != 0;
  /*! \brief PS_GATED_FRAMES (default 1): completion signalled by the copy engine into the peer's
   *  descriptor ring; 0 = cudaEvent + completion thread for every message (round-1 behaviour) */
  bool signal_ = GetEnv("PS_GATED_FRAMES", 1) != 0;
  std::atomic<uint64_t> gated_frames_{0};
  std::atomic<uint64_t> coalesced_batches_{0};
  std::atomic<uint64_t> coalesced_copies_{0};
};

}  // namespace ps
#endif  // PS_VAN_ONESIDED_VAN_H_
