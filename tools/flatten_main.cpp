// Build-time helper: dumps the product's flattened model (ik_b200/csrc/urdf_model.cpp) as JSON so that
// tools/gen_kernel.py can specialise a kernel on it.  Usage: ikb_flatten <urdf> <free_flyer 0|1>
#include <cstdio>
#include <fstream>
#include <iostream>
#include <sstream>

#include "../ik_b200/csrc/model.hpp"

int main(int argc, char **argv) {
    if (argc < 3) {
        std::fprintf(stderr, "usage: %s <urdf> <free_flyer>\n", argv[0]);
        return 2;
    }
    std::ifstream f(argv[1]);
    std::stringstream ss;
    ss << f.rdbuf();
    ikb::HostModel m;
    try {
        m = ikb::model_from_urdf(ss.str(), argv[2][0] == '1');
    } catch (const std::exception &e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 1;
    }
    std::printf("{\n\"nq\": %d, \"nv\": %d,\n\"joints\": [\n", m.nq, m.nv);
    for (int j = 0; j < m.njoints(); ++j) {
        std::printf("{\"name\": \"%s\", \"parent\": %d, \"type\": %d, \"idx_q\": %d, \"idx_v\": %d, \"placement\": [",
                    m.joint_names[j].c_str(), m.parent[j], m.jtype[j], m.idx_q[j], m.idx_v[j]);
        for (int k = 0; k < 12; ++k) std::printf("%s%.17g", k ? ", " : "", m.placement[j][k]);
        std::printf("], \"axis\": [%.17g, %.17g, %.17g], \"mass\": %.17g, \"com\": [%.17g, %.17g, %.17g]}%s\n", m.axis[j][0],
                    m.axis[j][1], m.axis[j][2], m.mass[j], m.com[j][0], m.com[j][1], m.com[j][2], j + 1 < m.njoints() ? "," : "");
    }
    std::printf("],\n\"frames\": [\n");
    for (int i = 0; i < m.nframes(); ++i) {
        std::printf("{\"name\": \"%s\", \"parent\": %d, \"placement\": [", m.frame_names[i].c_str(), m.frame_parent[i]);
        for (int k = 0; k < 12; ++k) std::printf("%s%.17g", k ? ", " : "", m.frame_placement[i][k]);
        std::printf("]}%s\n", i + 1 < m.nframes() ? "," : "");
    }
    std::printf("]\n}\n");
    return 0;
}
