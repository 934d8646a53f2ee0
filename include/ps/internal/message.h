/**
 * \file message.h
 * \brief The in-memory message model: Node, Control, Meta, Message.
 *
 * Field names follow the reference so application code ports unchanged
 * (parity: include/ps/internal/message.h:14-18,37-62,66-134,139-173,177-258,
 * 262-300). Differences, on purpose:
 *   - byte counts (data_size, val_len) are 64-bit: a single B200 message may
 *     exceed 2 GiB (the reference caps at INT_MAX, SURVEY appendix C);
 *   - Meta carries a MemRef: {region, offset, flag_seq} names a span inside a
 *     peer-mapped memory region (HBM exported over CUDA IPC / VMM, or POSIX shm),
 *     which is what replaces the reference's (addr, rkey) pair on RDMA;
 *   - Node carries pid + device ordinal so co-located endpoints can skip IPC.
 */
#ifndef PS_INTERNAL_MESSAGE_H_
#define PS_INTERNAL_MESSAGE_H_
#include <array>
#include <climits>
#include <cstdint>
#include <sstream>
#include <string>
#include <vector>
#include "ps/internal/inline_vec.h"
#include "ps/sarray.h"

namespace ps {

/*! \brief element types that can travel in Message::data */
enum DataType {
  CHAR, INT8, INT16, INT32, INT64, UINT8, UINT16, UINT32, UINT64, FLOAT, DOUBLE, OTHER
};
static const char* const DataTypeName[] = {"CHAR",  "INT8",   "INT16",  "INT32",  "INT64", "UINT8",
                                           "UINT16", "UINT32", "UINT64", "FLOAT", "DOUBLE", "OTHER"};

namespace msg_detail {
template <typename V> struct TypeTag { static constexpr DataType value = OTHER; };
#define PS_TYPE_TAG_(T, E) template <> struct TypeTag<T> { static constexpr DataType value = E; }
PS_TYPE_TAG_(char, CHAR);
PS_TYPE_TAG_(int8_t, INT8);
PS_TYPE_TAG_(int16_t, INT16);
PS_TYPE_TAG_(int32_t, INT32);
PS_TYPE_TAG_(int64_t, INT64);
PS_TYPE_TAG_(uint8_t, UINT8);
PS_TYPE_TAG_(uint16_t, UINT16);
PS_TYPE_TAG_(uint32_t, UINT32);
PS_TYPE_TAG_(uint64_t, UINT64);
PS_TYPE_TAG_(float, FLOAT);
PS_TYPE_TAG_(double, DOUBLE);
#undef PS_TYPE_TAG_
}  // namespace msg_detail

template <typename V>
DataType GetDataType() {
  return msg_detail::TypeTag<V>::value;
}

/*! \brief maximum ports / devices one node may advertise */
static const int kMaxNodePorts = 32;

/*! \brief identity and addressing of one postoffice instance */
struct Node {
  /*! \brief "unset" sentinel for ids and ports */
  static const int kEmpty;
  enum Role { SERVER, WORKER, SCHEDULER, JOINT };

  Node() : role(SERVER), id(kEmpty), customer_id(0), num_ports(1), port(kEmpty),
           is_recovery(false), endpoint_name_len(0), aux_id(-1), pid(0), dev_id(-1) {
    ports.fill(0);
    dev_types.fill(UNK);
    dev_ids.fill(0);
    memset(endpoint_name, 0, sizeof(endpoint_name));
  }

  static const char* RoleName(Role r) {
    switch (r) {
      case SERVER: return "server";
      case WORKER: return "worker";
      case SCHEDULER: return "scheduler";
      default: return "joint";
    }
  }
  std::string DebugString() const {
    std::ostringstream os;
    os << "[role=" << RoleName(role);
    if (id != kEmpty) os << ", id=" << id;
    os << ", ip=" << hostname << ", port=" << port << ", is_recovery=" << is_recovery
       << ", aux_id=" << aux_id << ", num_ports=" << num_ports;
    if (num_ports > 1) {
      os << ", ports=[";
      for (int i = 0; i < num_ports; ++i) os << ports[i] << ",";
      os << "], devices=[";
      for (int i = 0; i < num_ports; ++i)
        os << DeviceTypeName[dev_types[i]] << "[" << dev_ids[i] << "],";
      os << "]";
    }
    if (dev_id >= 0) os << ", gpu=" << dev_id;
    if (pid) os << ", pid=" << pid;
    if (endpoint_name_len) os << ", endpoint_name_len=" << endpoint_name_len;
    os << "]";
    return os.str();
  }
  std::string ShortDebugString() const {
    std::string s = role == SERVER ? "S" : (role == WORKER ? "W" : "H");
    if (id != kEmpty) s += "[" + std::to_string(id) + "]";
    return s;
  }
  /*! \brief "host:port" — the identity the scheduler dedups on */
  std::string Address() const { return hostname + ":" + std::to_string(port); }

  Role role;
  int id;
  int customer_id;
  std::string hostname;
  int num_ports;
  std::array<int, kMaxNodePorts> ports;
  std::array<int, kMaxNodePorts> dev_types;
  std::array<int, kMaxNodePorts> dev_ids;
  int port;
  bool is_recovery;
  /*! \brief opaque transport endpoint blob (a CUDA IPC handle is exactly 64 B) */
  char endpoint_name[64];
  size_t endpoint_name_len;
  /*! \brief preferred rank on registration; transport scratch afterwards */
  int aux_id;
  /*! \brief OS process id: equal (hostname, pid) means "same address space" */
  int pid;
  /*! \brief CUDA device ordinal this instance is bound to, -1 if CPU-only */
  int dev_id;
};

/*! \brief system-level command riding in Meta::control */
struct Control {
  enum Command {
    EMPTY, TERMINATE, ADD_NODE, BARRIER, ACK, HEARTBEAT, BOOTSTRAP, ADDR_REQUEST,
    ADDR_RESOLVED, INSTANCE_BARRIER
  };
  Control() : cmd(EMPTY), barrier_group(0), msg_sig(0) {}
  bool empty() const { return cmd == EMPTY; }
  static const char* CommandName(Command c) {
    static const char* const names[] = {"EMPTY", "TERMINATE", "ADD_NODE", "BARRIER", "ACK",
                                        "HEARTBEAT", "BOOTSTRAP", "ADDR_REQUEST",
                                        "ADDR_RESOLVED", "INSTANCE_BARRIER"};
    return names[c];
  }
  std::string DebugString() const {
    if (empty()) return "";
    std::ostringstream os;
    os << "cmd=" << CommandName(cmd);
    if (!node.empty()) {
      os << ", node={";
      for (const Node& n : node) os << " " << n.DebugString();
      os << " }";
    }
    if (cmd == BARRIER || cmd == INSTANCE_BARRIER) os << ", barrier_group=" << barrier_group;
    if (cmd == ACK) os << ", msg_sig=" << msg_sig;
    return os.str();
  }
  Command cmd;
  std::vector<Node> node;
  int barrier_group;
  uint64_t msg_sig;
};

/*!
 * \brief a span inside a memory region that the receiver can (or already does)
 *        map: the B200 replacement for RDMA's (remote address, rkey).
 */
struct MemRef {
  /*! \brief region id unique per exporting node; -1 = none */
  int32_t region = -1;
  /*! \brief byte offset of the span inside the region */
  uint64_t offset = 0;
  /*! \brief bytes of payload placed at the span (wire form) */
  uint64_t bytes = 0;
  /*! \brief value the producer will store to the span's ready-flag; 0 = no flag */
  uint64_t flag_seq = 0;
  bool valid() const { return region >= 0; }
};

/*! \brief everything about a message except its bulk payload */
struct Meta {
  static const int kEmpty;
  Meta()
      : head(kEmpty), app_id(kEmpty), customer_id(kEmpty), timestamp(kEmpty), sender(kEmpty),
        recver(kEmpty), request(false), push(false), simple_app(false) {}

  std::string DebugString() const {
    std::ostringstream os;
    if (sender == kEmpty) os << "?"; else os << sender;
    os << " => " << recver << ". Meta: request=" << request;
    if (timestamp != kEmpty) os << ", timestamp=" << timestamp;
    if (!control.empty()) {
      os << ", control={ " << control.DebugString() << " }";
    } else {
      os << ", app_id=" << app_id << ", customer_id=" << customer_id
         << ", simple_app=" << simple_app << ", push=" << push << (pull ? "+pull" : "") << ", sid=" << sid;
    }
    if (head != kEmpty) os << ", head=" << head;
    if (control.empty() && !simple_app) os << ", key=" << key;
    if (!body.empty()) os << ", body=" << body;
    if (!data_type.empty()) {
      os << ", dtype={";
      for (auto d : data_type) os << " " << DataTypeName[static_cast<int>(d)];
      os << " }";
    }
    if (mem.valid()) os << ", mem={r" << mem.region << "+" << mem.offset << " bytes=" << mem.bytes << "}";
    if (codec) os << ", codec=" << codec << ", scale=" << scale;
    if (!control.empty() || simple_app) os << ". NOT DATA MSG!";
    return os.str();
  }

  int head;
  int app_id;
  int customer_id;
  int timestamp;
  int sender;
  int recver;
  bool request;
  bool push;
  bool simple_app;
  std::string body;
  InlineVec<DataType, 4> data_type;
  DeviceType src_dev_type = UNK;
  int src_dev_id = -1;
  DeviceType dst_dev_type = UNK;
  int dst_dev_id = -1;
  Control control;
  /*! \brief total payload bytes over all data segments */
  int64_t data_size = 0;
  /*! \brief first key of the message (one key per message on the one-sided paths) */
  uint64_t key = 0;
  /*! \brief address of the sender-side value buffer (pull destination) */
  uint64_t addr = 0;
  /*! \brief number of value elements */
  int64_t val_len = 0;
  /*!
   * \brief fused push-pull: a push request that also asks for the (updated) values. The reply
   *        is a pull response that lands at `pull_addr` (`pull_len` elements) / `pull_mem`;
   *        there is no separate push ack. Halves the messages of a push + pull pair.
   */
  bool pull = false;
  uint64_t pull_addr = 0;
  int64_t pull_len = 0;
  MemRef pull_mem;
  /*! \brief free 4-byte field for applications / transports */
  int option = 0;
  /*! \brief per-peer sequence id (ordered delivery) */
  int sid = 0;
  /*! \brief peer-mappable location of the value buffer, if any */
  MemRef mem;
  /*! \brief transform the sender's copy engine applied to the values (WireCodec) */
  int codec = 0;
  /*! \brief scale folded into the transform (e.g. 1/num_workers on gradient push) */
  float scale = 1.0f;
};

/*! \brief optional transform applied by the copy engine while it moves the bytes */
enum WireCodec : int {
  kCodecRaw = 0,           // byte copy
  kCodecF32ToBf16 = 1,     // dst_bf16[i] = src_f32[i] * scale
  kCodecBf16Scale = 2,     // dst_bf16[i] = src_bf16[i] * scale
  kCodecF32ToFp8Block = 3, // block-scaled e4m3: 32 elements share one e8m0 exponent
  kCodecBf16ToFp8Block = 4,
  kCodecPlaced = 5,        // payload already written by the application; send descriptor only
  kCodecNumCodecs
};

/*! \brief bytes the wire form of `n_src_bytes` of source occupies */
inline uint64_t WireBytes(int codec, uint64_t n_src_bytes) {
  switch (codec) {
    case kCodecF32ToBf16: return n_src_bytes / 2;
    case kCodecBf16Scale: return n_src_bytes;
    case kCodecF32ToFp8Block: {  // n elements -> n bytes of e4m3 + n/32 scale bytes
      const uint64_t n = n_src_bytes / 4;
      return ((n + 31) & ~uint64_t(31)) + ((n + 31) & ~uint64_t(31)) / 32;
    }
    case kCodecBf16ToFp8Block: {
      const uint64_t n = n_src_bytes / 2;
      return ((n + 31) & ~uint64_t(31)) + ((n + 31) & ~uint64_t(31)) / 32;
    }
    default: return n_src_bytes;
  }
}

/*! \brief per-send options that never travel on the wire */
struct SendOpts {
  /*! \brief WireCodec applied while copying the values into peer memory */
  int codec = 0;
  float scale = 1.0f;
  /*! \brief cudaEvent_t the copy must wait for (producer of the values), or null */
  void* wait_event = nullptr;
  /*!
   * \brief the remote side already knows this buffer under a name (e.g. an offset inside a
   *        symmetric / multicast-bound buffer), so the van must not export or rendezvous.
   *        Pull: where the reply lands. Push: where the (encoded) values are staged — in the
   *        SENDER's own symmetric buffer, at `stage`; the server then reads all workers'
   *        copies at that offset through the multicast address (in-switch reduction).
   */
  MemRef dest_mem;
  /*! \brief push with a symmetric `dest_mem`: local address the values are encoded into */
  void* stage = nullptr;
  /*! \brief fused push-pull: caller-named destination of the reply (like `dest_mem` for a pull) */
  MemRef pull_dest_mem;
  /*! \brief value of Meta::option / KVMeta::option (application-defined flags) */
  int option = 0;
  /*!
   * \brief push over a one-sided van: request the landing slot at this capacity and reuse it for
   *        every push of the key that fits, however much smaller (pushes whose size changes every
   *        step, e.g. row-sparse gradients). 0: the slot is re-made when a push outgrows it or
   *        shrinks far below it.
   */
  uint64_t slot_bytes = 0;
};

/*! \brief MemRef::region value meaning "offset inside the job-wide symmetric buffer" */
static const int32_t kSymmetricRegion = 0x40000000;

/*! \brief meta + zero-copy payload segments */
struct Message {
  Meta meta;
  InlineVec<SArray<char>, 4> data;
  /*! \brief local-only: event gating the one-sided copy of data[1] */
  void* wait_event = nullptr;
  /*! \brief local-only: staging address of a symmetric push (see SendOpts::stage) */
  void* stage = nullptr;
  /*! \brief local-only: landing-slot capacity to request (see SendOpts::slot_bytes) */
  uint64_t slot_bytes = 0;

  /*! \brief append a segment; the second one (the values) sets the placement fields */
  template <typename V>
  void AddData(const SArray<V>& val) {
    CHECK_EQ(data.size(), meta.data_type.size());
    meta.data_type.push_back(GetDataType<V>());
    SArray<char> bytes(val);
    meta.data_size += static_cast<int64_t>(bytes.size());
    data.push_back(bytes);
    if (data.size() == 2) {
      meta.src_dev_type = val.src_device_type_;
      meta.src_dev_id = val.src_device_id_;
      meta.dst_dev_type = val.dst_device_type_;
      meta.dst_dev_id = val.dst_device_id_;
    }
  }
  std::string DebugString() const {
    std::ostringstream os;
    os << meta.DebugString();
    if (!data.empty()) {
      os << " Body: { " << DeviceTypeName[meta.src_dev_type] << "(" << meta.src_dev_id << ")->"
         << DeviceTypeName[meta.dst_dev_type] << "(" << meta.dst_dev_id << ") data_size=[";
      for (const auto& d : data) os << d.size() << ",";
      os << "] }";
    }
    return os.str();
  }
};

}  // namespace ps
#endif  // PS_INTERNAL_MESSAGE_H_
