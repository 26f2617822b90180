// TEST-ONLY: spec_harness.cpp's kernel-shaped loop, plus the Cassie specialisation whose pelvis task is folded into the
// two leg roles (ik_b200/specs/cassie_feet_pelvis_fold.json), so that it can be compared with the three-role arrow body
// (exported by spec_harness.cpp too) in one library.
#include "../../ik_b200/csrc/gen/cassie_feet_pelvis_fold.cuh"
#include "spec_harness.cpp"

IKB_SPEC_EXPORT(h_spec_cassie_feet_pelvis_fold, SpecCassieFeetPelvisFold)
