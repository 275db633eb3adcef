// Host-side readers for the reference's input files (no Boost / urdfdom / Pinocchio in the product):
//   * boost-property-tree INFO files — task.info, reference.info, gait.info as loaded by
//     QMInterface::QMInterface (qm_interface/src/QMInterface.cpp:37-74) through ocs2::loadData
//   * the URDF consumed by QMInterface::setupModel (QMInterface.cpp:408-439)
// and the model constants derived from them (CentroidalModelInfo, cost weights, limits).
#pragma once
#include <map>
#include <stdexcept>
#include <string>
#include <vector>

#include "../kernels/dev_common.cuh"

namespace qmb {

// Flat view of an INFO file: "a.b.c" → value; children order preserved for list-like nodes.
class InfoFile {
 public:
  explicit InfoFile(const std::string& path);
  bool has(const std::string& key) const { return values_.count(key) != 0; }
  double number(const std::string& key) const;
  double number(const std::string& key, double fallback) const { return has(key) ? number(key) : fallback; }
  std::string text(const std::string& key) const;
  // boolean leaf as ocs2::loadData::loadPtreeValue<bool> reads it ("true" / "false", "1" / "0"); a missing key gives `fallback`, any other value throws
  bool boolean(const std::string& key, bool fallback) const;
  // ocs2::loadData::loadEigenMatrix semantics ("(i,j) value" entries times optional "scaling")
  std::vector<double> matrix(const std::string& key, int rows, int cols) const;
  // "[i] value" children of a node, in index order
  std::vector<std::string> list(const std::string& key) const;
  bool has_node(const std::string& key) const { return nodes_.count(key) != 0; }
 private:
  std::map<std::string, std::string> values_;
  std::map<std::string, std::vector<std::string>> nodes_;   // node path → child keys (in file order)
};

struct UrdfJoint { std::string name, type, parent, child; double xyz[3] = {0, 0, 0}, rpy[3] = {0, 0, 0}, axis[3] = {1, 0, 0}; double lower = 0, upper = 0, effort = 0, velocity = 0; };
struct UrdfLink { std::string name; bool has_inertial = false; double mass = 0, com[3] = {0, 0, 0}, rpy[3] = {0, 0, 0}, inertia[6] = {0, 0, 0, 0, 0, 0}; /* ixx ixy ixz iyy iyz izz */ };
struct UrdfRobot { std::map<std::string, UrdfLink> links; std::map<std::string, UrdfJoint> joints; };
UrdfRobot read_urdf(const std::string& path);

struct HostFrame { std::string name; int body; double R[9]; double p[3]; };

// Everything the kernels need, on the host (mirrors DevModel) plus names for the API layer.
struct HostModel {
  DevModel dev;
  std::vector<std::string> joint_names;
  std::vector<HostFrame> frames;
  double initial_state[NX];
  double default_joint_state[NJ];
};

// Build the model exactly as the reference does: composite floating root, joints in name-sorted depth-first
// order, fixed joints lumped, SRBD CentroidalModelInfo from reference.info:defaultJointState, cost weights
// from task.info (Q, R with the leg-velocity block mapped through the foot Jacobians, QMInterface.cpp:274-299).
HostModel build_host_model(const std::string& task_file, const std::string& urdf_file, const std::string& reference_file, const std::string& gains_file);

// gait.info / reference.info mode-sequence templates (ocs2 ModeSequenceTemplate) and name → mode number
struct ModeTemplate { std::vector<double> switching_times; std::vector<int> modes; };
int mode_from_name(const std::string& name);
ModeTemplate read_mode_template(const InfoFile& f, const std::string& key);

}  // namespace qmb
