// TEST-ONLY: the generated body of a plugin specialisation (a header written by tools/gen_kernel.py for one URDF and task
// list, named by -DIKB_PLUGIN_HEADER="..." with its struct -DIKB_PLUGIN_STRUCT=...) driven on the CPU by spec_harness.cpp's
// loop, exported as h_spec_plugin_{d,f,pd,eval}.  Never linked into libikb200.so.
#include "spec_harness.cpp"
#include IKB_PLUGIN_HEADER

IKB_SPEC_EXPORT(h_spec_plugin, IKB_PLUGIN_STRUCT)
