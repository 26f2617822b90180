// What a joint type means, for host and device code alike: its configuration and tangent sizes and the kind of motion it
// has.  Every test of a joint type outside the flattener goes through these helpers, so that a new type cannot fall
// silently into the branch of another one (the codes are public ABI values, include/ikb200.h, and not ordered by kind).
//
//   universe            nq 0, nv 0
//   free-flyer          nq 7 (x y z, qx qy qz qw), nv 6
//   revolute            nq 1 (angle), nv 1                  RX RY RZ, unaligned
//   continuous          nq 2 (cos, sin of the angle), nv 1  RUBX RUBY RUBZ, unaligned (Pinocchio's RevoluteUnbounded)
//   prismatic           nq 1, nv 1                          PX PY PZ, unaligned
#pragma once
#include "../../include/ikb200.h"

#if defined(__CUDACC__)
#define IKB_JT_HD __host__ __device__ __forceinline__ constexpr
#else
#define IKB_JT_HD inline constexpr
#endif

namespace ikb {

IKB_JT_HD bool is_continuous(int t) { return t >= IKB_J_RUBX && t <= IKB_J_RUB_UNALIGNED; }
IKB_JT_HD bool is_revolute(int t) { return t >= IKB_J_RX && t <= IKB_J_REV_UNALIGNED; }   // bounded revolute only
IKB_JT_HD bool is_revolute_like(int t) { return is_revolute(t) || is_continuous(t); }
IKB_JT_HD bool is_prismatic(int t) { return t >= IKB_J_PX && t <= IKB_J_PRIS_UNALIGNED; }
IKB_JT_HD int joint_nq(int t) { return t == IKB_J_UNIVERSE ? 0 : (t == IKB_J_FREEFLYER ? 7 : (is_continuous(t) ? 2 : 1)); }
IKB_JT_HD int joint_nv(int t) { return t == IKB_J_UNIVERSE ? 0 : (t == IKB_J_FREEFLYER ? 6 : 1); }
// 0 / 1 / 2 for a joint along the x / y / z axis of its frame, -1 for an unaligned one (axis in the model) and for the
// universe and free-flyer joints
IKB_JT_HD int axis_index(int t) {
    return (t == IKB_J_RX || t == IKB_J_PX || t == IKB_J_RUBX) ? 0
         : (t == IKB_J_RY || t == IKB_J_PY || t == IKB_J_RUBY) ? 1
         : (t == IKB_J_RZ || t == IKB_J_PZ || t == IKB_J_RUBZ) ? 2 : -1;
}
// the revolute type with the same axis as a continuous one (their placement and Jacobian column are the same), other
// types unchanged
IKB_JT_HD int as_revolute(int t) { return is_continuous(t) ? t - (IKB_J_RUBX - IKB_J_RX) : t; }

}  // namespace ikb

#undef IKB_JT_HD
