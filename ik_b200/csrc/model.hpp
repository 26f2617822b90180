// Host-side flat kinematic model and IK problem description (internal to libikb200.so).
//
// HostModel is what the reference gets from pinocchio::Model (common.hpp:17): joints in Pinocchio's
// depth-first order with parent indices, joint placements, configuration / tangent offsets, position
// limits and the frame table.  HostProblem mirrors ik::InverseKinematicsProblem (problem.hpp:9-206)
// restricted to the task kinds the DLS hot path evaluates.
#pragma once
#include <array>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/ikb200.h"
#include "joint_types.hpp"

namespace ikb {

using SE3d = std::array<double, 12>;  // R row-major (9) then p (3)

inline SE3d se3_identity() { return SE3d{1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0}; }
SE3d se3_mul(const SE3d &a, const SE3d &b);

enum FrameType { FRAME_OP = 0, FRAME_JOINT = 1, FRAME_FIXED_JOINT = 2, FRAME_BODY = 3 };

struct HostModel {
    std::vector<std::string> joint_names;
    std::vector<int32_t> parent, jtype, idx_q, idx_v;
    std::vector<SE3d> placement;
    std::vector<std::array<double, 3>> axis;
    std::vector<double> lower, upper;
    // per joint: total mass of the bodies it supports (bodies behind fixed joints included) and their centre of mass in
    // the joint frame -- Pinocchio's model.inertias[j].mass() / .lever(), read by CentreOfMassTask only
    std::vector<double> mass;
    std::vector<std::array<double, 3>> com;
    std::vector<std::string> frame_names;
    std::vector<int32_t> frame_parent, frame_type;
    std::vector<SE3d> frame_placement;
    int nq = 0, nv = 0;

    int njoints() const { return (int)parent.size(); }
    int nframes() const { return (int)frame_parent.size(); }
    int frame_id(const std::string &name) const;  // model.getFrameId: nframes() when absent
    int add_joint(const std::string &name, int type, int parent_joint, const SE3d &pl, const std::array<double, 3> &ax,
                  const std::vector<double> &lo, const std::vector<double> &hi);
    int add_frame(const std::string &name, int parent_joint, const SE3d &pl, int type);
};

// URDF text -> HostModel following urdfdom + Pinocchio's traversal (SURVEY.md 8c.1).  Throws
// std::runtime_error with a message on malformed input / unsupported joints.
HostModel model_from_urdf(const std::string &xml, bool free_flyer);

struct HostTask {
    int kind = IKB_TASK_FRAME;
    int frame = 0, ref = 0;
    int type = IKB_FULL;  // FRAME: kinematic type; ALIGN_AXIS: axis; POSTURE: nj
    int priority = 0;
    int dim = 0;
    int target_size = 0;
    std::vector<double> weight;  // dim
    std::vector<double> mask;    // posture only
};

// FrameConstraint (frame.hpp:333-465): ik::dls projects its step into the null space of the stacked constraint Jacobian
struct HostConstraint {
    int frame = 0, ref = 0;
    int type = IKB_FULL;
    int dim = 6;
};

struct HostProblem {
    HostModel model;  // by value, like the reference (problem.hpp:183)
    int max_priority_level = 0;
    std::vector<HostTask> tasks;  // insertion order
    std::vector<HostConstraint> constraints;  // insertion order
    int c_size() const {  // problem.hpp:47-53
        int n = 0;
        for (const auto &c : constraints) n += c.dim;
        return n;
    }

    int levels() const {  // one more than the highest priority any task uses
        int n = 0;
        for (const auto &t : tasks) n = t.priority + 1 > n ? t.priority + 1 : n;
        return n;
    }

    int rows() const;
    int e_size(int priority) const;
    int target_size() const;
    int target_offset(int task) const;
};

}  // namespace ikb
