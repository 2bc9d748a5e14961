// bag_reader.hpp -- minimal rosbag v2.0 reader for /tf recordings and the offline replay loop of the node.
//
// The reference is fed by a /tf subscriber (tf2_msgs/TFMessage -> transformStampedToPose7d,
// /root/reference/include/target_estimation/target_manager_ros.hpp:36-46, src/target_manager_ros.cpp:26-39) and ships one
// recording, test/test_multiple_targets.bag (frames target_0..2), to be played against target_node.  This reader takes
// such a bag without ROS: file header, chunk records (uncompressed), connection records, message-data records; the
// message body is the ROS1 serialisation of TFMessage (uint32 count, then per transform: header {seq, stamp, frame_id},
// child_frame_id, translation xyz, rotation xyzw as little-endian doubles).
// replayBag() is the node's main loop (src/target_node.cpp:36-44: update(dt); spinOnce(); sleep) on the bag's clock.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace target_estimation_b200 {

class TickFrontEnd;

struct TfRecord {
  uint32_t rec_sec = 0, rec_nsec = 0;   // receive time of the message record (what `rosbag play --clock` publishes as now)
  uint32_t msg = 0;                     // index of the TFMessage this transform belongs to (one callback per message)
  uint32_t seq = 0, sec = 0, nsec = 0;  // header.seq, header.stamp
  std::string frame_id, child_frame_id;
  double pose[7] = {0, 0, 0, 0, 0, 0, 1};   // transformStampedToPose7d: translation xyz, rotation xyzw
};

// every transform of every message on `topic`, in record order.  Throws std::runtime_error on a malformed or
// compressed bag (bz2 / lz4 chunks are not supported: re-record with `rosbag compress -j` undone, `rosbag decompress`).
std::vector<TfRecord> readBagTf(const std::string& path, const std::string& topic = "/tf");

struct ReplayStats {
  long long ticks = 0, messages = 0, transforms = 0, erased = 0;
};
// target_node's loop on the recording: tick k runs at now_k = (first record time) + k / frequency (integer nanoseconds);
// after each tick the messages received up to now_k are delivered, one measurementCallBack per message.  Ends
// `extra_ticks` ticks after the last message was delivered.
ReplayStats replayBag(TickFrontEnd& mgr, const std::vector<TfRecord>& records, double frequency, long long extra_ticks = 0);

}  // namespace target_estimation_b200
