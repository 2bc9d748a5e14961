// bag_reader.cpp -- rosbag v2.0 /tf reader + offline replay (see include/target_estimation_b200/bag_reader.hpp)
#include "target_estimation_b200/bag_reader.hpp"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <stdexcept>

#include "target_estimation_b200/target_manager.hpp"

namespace target_estimation_b200 {

namespace {

struct Cursor {
  const uint8_t* p;
  size_t n, pos = 0;
  Cursor(const uint8_t* p_, size_t n_) : p(p_), n(n_) {}
  bool done() const { return pos >= n; }
  void need(size_t k) const {
    if (k > n - pos) throw std::runtime_error("rosbag: truncated record");
  }
  uint32_t u32() {
    need(4);
    uint32_t v;
    std::memcpy(&v, p + pos, 4);   // little-endian on disk and on every host this builds for
    pos += 4;
    return v;
  }
  double f64() {
    need(8);
    double v;
    std::memcpy(&v, p + pos, 8);
    pos += 8;
    return v;
  }
  Cursor sub(size_t k) {
    need(k);
    Cursor c(p + pos, k);
    pos += k;
    return c;
  }
  std::string str() {
    const uint32_t l = u32();
    need(l);
    std::string s(reinterpret_cast<const char*>(p + pos), l);
    pos += l;
    return s;
  }
};

using Fields = std::map<std::string, std::string>;

// record header / connection header: repeated <uint32 len><name>=<value>
Fields parseFields(Cursor c) {
  Fields f;
  while (!c.done()) {
    const uint32_t l = c.u32();
    c.need(l);
    const char* s = reinterpret_cast<const char*>(c.p + c.pos);
    const void* eq = std::memchr(s, '=', l);
    if (!eq) throw std::runtime_error("rosbag: header field without '='");
    const size_t k = (size_t)(static_cast<const char*>(eq) - s);
    f[std::string(s, k)] = std::string(s + k + 1, l - k - 1);
    c.pos += l;
  }
  return f;
}
uint32_t fieldU32(const Fields& f, const char* name) {
  auto it = f.find(name);
  if (it == f.end() || it->second.size() < 4) throw std::runtime_error(std::string("rosbag: missing header field ") + name);
  uint32_t v;
  std::memcpy(&v, it->second.data(), 4);
  return v;
}

struct Parser {
  std::string topic;
  std::map<uint32_t, bool> conn_wanted;   // connection id -> (topic matches and the type is a TF message)
  std::vector<TfRecord> out;
  uint32_t n_msgs = 0;

  void message(const Fields& h, Cursor body) {
    const uint32_t conn = fieldU32(h, "conn");
    auto it = conn_wanted.find(conn);
    if (it == conn_wanted.end() || !it->second) return;
    auto t = h.find("time");
    if (t == h.end() || t->second.size() < 8) throw std::runtime_error("rosbag: message record without time");
    uint32_t rs, rn;
    std::memcpy(&rs, t->second.data(), 4);
    std::memcpy(&rn, t->second.data() + 4, 4);
    const uint32_t count = body.u32();
    for (uint32_t i = 0; i < count; ++i) {
      TfRecord r;
      r.rec_sec = rs;
      r.rec_nsec = rn;
      r.msg = n_msgs;
      r.seq = body.u32();
      r.sec = body.u32();
      r.nsec = body.u32();
      r.frame_id = body.str();
      r.child_frame_id = body.str();
      for (int e = 0; e < 7; ++e) r.pose[e] = body.f64();
      out.push_back(std::move(r));
    }
    ++n_msgs;
  }

  void records(Cursor c, bool top_level) {
    while (!c.done()) {
      const uint32_t hl = c.u32();
      const Fields h = parseFields(c.sub(hl));
      const uint32_t dl = c.u32();
      Cursor data = c.sub(dl);
      auto op = h.find("op");
      if (op == h.end() || op->second.size() < 1) throw std::runtime_error("rosbag: record without op");
      switch ((uint8_t)op->second[0]) {
        case 0x02: message(h, data); break;
        case 0x05: {   // chunk
          if (!top_level) throw std::runtime_error("rosbag: nested chunk");
          auto comp = h.find("compression");
          if (comp == h.end() || comp->second != "none")
            throw std::runtime_error("rosbag: compressed chunks (" + (comp == h.end() ? std::string("?") : comp->second) + ") are not supported");
          records(data, false);
          break;
        }
        case 0x07: {   // connection: header {conn, topic}, data = connection header {topic, type, md5sum, ...}
          const uint32_t conn = fieldU32(h, "conn");
          const Fields ch = parseFields(data);
          auto tp = h.find("topic");
          auto ty = ch.find("type");
          const bool is_tf = ty != ch.end() && (ty->second == "tf2_msgs/TFMessage" || ty->second == "tf/tfMessage");
          conn_wanted[conn] = tp != h.end() && tp->second == topic && is_tf;
          break;
        }
        default: break;   // 0x03 bag header, 0x04 index data, 0x06 chunk info: not needed for a sequential read
      }
    }
  }
};

}  // namespace

std::vector<TfRecord> readBagTf(const std::string& path, const std::string& topic) {
  std::FILE* f = std::fopen(path.c_str(), "rb");
  if (!f) throw std::runtime_error("rosbag: cannot open " + path);
  std::vector<uint8_t> buf;
  uint8_t tmp[1 << 16];
  size_t k;
  while ((k = std::fread(tmp, 1, sizeof(tmp), f)) > 0) buf.insert(buf.end(), tmp, tmp + k);
  std::fclose(f);
  static const char magic[] = "#ROSBAG V2.0\n";
  const size_t ml = sizeof(magic) - 1;
  if (buf.size() < ml || std::memcmp(buf.data(), magic, ml) != 0) throw std::runtime_error("rosbag: not a V2.0 bag: " + path);
  Parser p;
  p.topic = topic;
  p.records(Cursor(buf.data() + ml, buf.size() - ml), true);
  return std::move(p.out);
}

ReplayStats replayBag(TickFrontEnd& mgr, const std::vector<TfRecord>& rec, double frequency, long long extra_ticks) {
  if (!(frequency > 0.0)) throw std::invalid_argument("frequency must be > 0");
  ReplayStats st;
  if (rec.empty()) return st;
  const double dt = 1.0 / frequency;                                  // src/target_node.cpp:32
  const long long period_ns = std::llround(1e9 / frequency);
  const long long t0 = (long long)rec[0].rec_sec * 1000000000LL + rec[0].rec_nsec;
  size_t next = 0;
  long long left_after_last = extra_ticks;
  std::vector<const char*> frames;
  std::vector<uint32_t> sec, nsec;
  std::vector<double> poses;
  std::vector<unsigned> erased;
  for (long long k = 0;; ++k) {
    const long long now = t0 + k * period_ns;
    erased.clear();
    mgr.tick(dt, (uint32_t)(now / 1000000000LL), (uint32_t)(now % 1000000000LL), &erased);   // ros_target_manager.update(dt)
    st.erased += (long long)erased.size();
    ++st.ticks;
    // ros::spinOnce(): every message received so far, one callback per message
    while (next < rec.size() && (long long)rec[next].rec_sec * 1000000000LL + rec[next].rec_nsec <= now) {
      const uint32_t m = rec[next].msg;
      frames.clear(); sec.clear(); nsec.clear(); poses.clear();
      while (next < rec.size() && rec[next].msg == m) {
        frames.push_back(rec[next].child_frame_id.c_str());
        sec.push_back(rec[next].sec);
        nsec.push_back(rec[next].nsec);
        poses.insert(poses.end(), rec[next].pose, rec[next].pose + 7);
        ++next;
      }
      mgr.measurementCallBack((long long)frames.size(), frames.data(), sec.data(), nsec.data(), poses.data());
      ++st.messages;
      st.transforms += (long long)frames.size();
    }
    if (next >= rec.size() && left_after_last-- <= 0) break;
  }
  return st;
}

}  // namespace target_estimation_b200
