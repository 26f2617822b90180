// URDF -> flat kinematic tree (host).  Replaces pinocchio::urdf::buildModelFromXML as used by the
// reference (ik_ros/src/cassie.cpp:34-35).  Neither urdfdom nor Pinocchio exist in this build, so the
// rules they apply are re-implemented here from their documented behaviour (SURVEY.md 8c.1):
//   * children of a link are visited in byte-wise order of JOINT name (urdfdom keeps joints in a
//     std::map<std::string, ...>), the tree is walked depth-first, movable joints are numbered in visit
//     order, fixed joints collapse into frames on the supporting joint;
//   * rpy -> quaternion (urdfdom Rotation::setFromRPY, normalised) -> matrix (Eigen), literals verbatim;
//   * a unit axis selects RX/RY/RZ (PX/PY/PZ, RUBX/RUBY/RUBZ), anything else is an unaligned joint with a normalised axis;
//   * a continuous joint is Pinocchio's unbounded revolute: q = (cos, sin), both entries bounded by +-1.01;
//   * the optional free-flyer root joint is "root_joint" with limits +-DBL_MAX.
// The XML reader below is a minimal non-validating parser (elements, attributes, comments, PIs, CDATA).
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>

#include "model.hpp"

namespace ikb {

SE3d se3_mul(const SE3d &a, const SE3d &b) {
    SE3d c;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) c[3 * i + j] = a[3 * i] * b[j] + a[3 * i + 1] * b[3 + j] + a[3 * i + 2] * b[6 + j];
        c[9 + i] = a[9 + i] + (a[3 * i] * b[9] + a[3 * i + 1] * b[10] + a[3 * i + 2] * b[11]);
    }
    return c;
}

int HostModel::frame_id(const std::string &name) const {
    for (size_t i = 0; i < frame_names.size(); ++i)
        if (frame_names[i] == name) return (int)i;
    return nframes();
}

int HostModel::add_joint(const std::string &name, int type, int parent_joint, const SE3d &pl,
                         const std::array<double, 3> &ax, const std::vector<double> &lo, const std::vector<double> &hi) {
    joint_names.push_back(name);
    parent.push_back(parent_joint);
    jtype.push_back(type);
    idx_q.push_back(nq);
    idx_v.push_back(nv);
    placement.push_back(pl);
    axis.push_back(ax);
    mass.push_back(0.0);
    com.push_back({0.0, 0.0, 0.0});
    lower.insert(lower.end(), lo.begin(), lo.end());
    upper.insert(upper.end(), hi.begin(), hi.end());
    nq += joint_nq(type);
    nv += joint_nv(type);
    return njoints() - 1;
}

int HostModel::add_frame(const std::string &name, int parent_joint, const SE3d &pl, int type) {
    frame_names.push_back(name);
    frame_parent.push_back(parent_joint);
    frame_placement.push_back(pl);
    frame_type.push_back(type);
    return nframes() - 1;
}

int HostProblem::rows() const {
    int s = 0;
    for (const auto &t : tasks) s += t.dim;
    return s;
}
int HostProblem::e_size(int priority) const {
    int s = 0;
    for (const auto &t : tasks)
        if (t.priority == priority) s += t.dim;
    return s;
}
int HostProblem::target_size() const {
    int s = 0;
    for (const auto &t : tasks) s += t.target_size;
    return s;
}
int HostProblem::target_offset(int task) const {
    int s = 0;
    for (int i = 0; i < task; ++i) s += tasks[i].target_size;
    return s;
}

// ---------------------------------------------------------------------------------------------------
// minimal XML reader
// ---------------------------------------------------------------------------------------------------
namespace {

struct XmlNode {
    std::string name;
    std::vector<std::pair<std::string, std::string>> attrs;
    std::vector<std::unique_ptr<XmlNode>> children;
    const std::string *attr(const char *key) const {
        for (const auto &kv : attrs)
            if (kv.first == key) return &kv.second;
        return nullptr;
    }
    const XmlNode *child(const char *tag) const {
        for (const auto &c : children)
            if (c->name == tag) return c.get();
        return nullptr;
    }
};

class XmlReader {
   public:
    explicit XmlReader(const std::string &s) : s_(s) {}
    std::unique_ptr<XmlNode> parse_document() {
        skip_misc();
        if (eof() || s_[i_] != '<') fail("no root element");
        auto root = parse_element();
        return root;
    }

   private:
    const std::string &s_;
    size_t i_ = 0;
    bool eof() const { return i_ >= s_.size(); }
    [[noreturn]] void fail(const std::string &why) const {
        throw std::runtime_error("URDF parse error at byte " + std::to_string(i_) + ": " + why);
    }
    bool starts(const char *lit) const { return s_.compare(i_, std::strlen(lit), lit) == 0; }
    void skip_until(const char *lit) {
        size_t p = s_.find(lit, i_);
        if (p == std::string::npos) fail(std::string("unterminated construct, expected ") + lit);
        i_ = p + std::strlen(lit);
    }
    void skip_ws() {
        while (!eof() && (s_[i_] == ' ' || s_[i_] == '\t' || s_[i_] == '\n' || s_[i_] == '\r')) ++i_;
    }
    // whitespace, text, comments, processing instructions, doctype
    void skip_misc() {
        for (;;) {
            while (!eof() && s_[i_] != '<') ++i_;
            if (eof()) return;
            if (starts("<!--")) skip_until("-->");
            else if (starts("<?")) skip_until("?>");
            else if (starts("<![CDATA[")) skip_until("]]>");
            else if (starts("<!")) skip_until(">");
            else return;
        }
    }
    std::string parse_name() {
        size_t b = i_;
        while (!eof()) {
            char c = s_[i_];
            if (c == ' ' || c == '\t' || c == '\n' || c == '\r' || c == '/' || c == '>' || c == '=') break;
            ++i_;
        }
        if (i_ == b) fail("expected a name");
        return s_.substr(b, i_ - b);
    }
    static std::string unescape(const std::string &v) {
        if (v.find('&') == std::string::npos) return v;
        static const std::pair<const char *, char> ents[] = {{"&amp;", '&'}, {"&lt;", '<'}, {"&gt;", '>'},
                                                            {"&quot;", '"'}, {"&apos;", '\''}};
        std::string o;
        for (size_t k = 0; k < v.size();) {
            bool hit = false;
            if (v[k] == '&')
                for (const auto &e : ents)
                    if (v.compare(k, std::strlen(e.first), e.first) == 0) {
                        o.push_back(e.second);
                        k += std::strlen(e.first);
                        hit = true;
                        break;
                    }
            if (!hit) o.push_back(v[k++]);
        }
        return o;
    }
    std::unique_ptr<XmlNode> parse_element() {
        ++i_;  // '<'
        auto node = std::make_unique<XmlNode>();
        node->name = parse_name();
        for (;;) {
            skip_ws();
            if (eof()) fail("unterminated start tag <" + node->name);
            if (s_[i_] == '/') {
                if (!starts("/>")) fail("malformed empty-element tag");
                i_ += 2;
                return node;
            }
            if (s_[i_] == '>') {
                ++i_;
                break;
            }
            std::string key = parse_name();
            skip_ws();
            if (eof() || s_[i_] != '=') fail("attribute " + key + " has no value");
            ++i_;
            skip_ws();
            if (eof() || (s_[i_] != '"' && s_[i_] != '\'')) fail("attribute value must be quoted");
            char quote = s_[i_++];
            size_t e = s_.find(quote, i_);
            if (e == std::string::npos) fail("unterminated attribute value");
            node->attrs.emplace_back(key, unescape(s_.substr(i_, e - i_)));
            i_ = e + 1;
        }
        for (;;) {
            skip_misc();
            if (eof()) fail("missing </" + node->name + ">");
            if (starts("</")) {
                i_ += 2;
                std::string close = parse_name();
                if (close != node->name) fail("mismatched </" + close + ">, expected </" + node->name + ">");
                skip_ws();
                if (eof() || s_[i_] != '>') fail("malformed end tag");
                ++i_;
                return node;
            }
            node->children.push_back(parse_element());
        }
    }
};

std::vector<double> parse_floats(const std::string *s, size_t n, const std::vector<double> &dflt, const char *what) {
    if (!s) return dflt;
    std::vector<double> v;
    const char *c = s->c_str();
    for (;;) {
        while (*c == ' ' || *c == '\t' || *c == '\n' || *c == '\r') ++c;
        if (!*c) break;
        char *end = nullptr;
        double x = std::strtod(c, &end);
        if (end == c) throw std::runtime_error(std::string("URDF: bad number in ") + what + "=\"" + *s + "\"");
        v.push_back(x);
        c = end;
    }
    if (v.size() != n) throw std::runtime_error(std::string("URDF: ") + what + " needs " + std::to_string(n) + " numbers");
    return v;
}

// urdfdom Rotation::setFromRPY (+normalize) then Eigen Quaternion::toRotationMatrix
SE3d origin_to_se3(const std::vector<double> &xyz, const std::vector<double> &rpy) {
    const double phi = rpy[0] / 2.0, the = rpy[1] / 2.0, psi = rpy[2] / 2.0;
    double x = std::sin(phi) * std::cos(the) * std::cos(psi) - std::cos(phi) * std::sin(the) * std::sin(psi);
    double y = std::cos(phi) * std::sin(the) * std::cos(psi) + std::sin(phi) * std::cos(the) * std::sin(psi);
    double z = std::cos(phi) * std::cos(the) * std::sin(psi) - std::sin(phi) * std::sin(the) * std::cos(psi);
    double w = std::cos(phi) * std::cos(the) * std::cos(psi) + std::sin(phi) * std::sin(the) * std::sin(psi);
    const double s = std::sqrt(x * x + y * y + z * z + w * w);
    x /= s; y /= s; z /= s; w /= s;
    const double tx = 2 * x, ty = 2 * y, tz = 2 * z;
    const double twx = tx * w, twy = ty * w, twz = tz * w;
    const double txx = tx * x, txy = ty * x, txz = tz * x;
    const double tyy = ty * y, tyz = tz * y, tzz = tz * z;
    return SE3d{1 - (tyy + tzz), txy - twz, txz + twy,
                txy + twz, 1 - (txx + tzz), tyz - twx,
                txz - twy, tyz + twx, 1 - (txx + tyy),
                xyz[0], xyz[1], xyz[2]};
}

struct UrdfJoint {
    std::string name, type, parent, child;
    SE3d placement;
    std::array<double, 3> axis;
    double lower = 0, upper = 0;
};

// Eigen isApprox(unit vector), default precision 1e-12
bool approx_unit(const std::array<double, 3> &a, int k) {
    double d2 = 0, n2 = 0;
    for (int i = 0; i < 3; ++i) {
        const double u = (i == k) ? 1.0 : 0.0;
        d2 += (a[i] - u) * (a[i] - u);
        n2 += a[i] * a[i];
    }
    return d2 <= 1e-24 * std::min(n2, 1.0);
}

struct Builder {
    HostModel m;
    std::map<std::string, std::vector<const UrdfJoint *>> children;  // parent link -> joints (sorted by name)
    std::map<std::string, int> body_frame;                           // link name -> BODY frame index

    void visit(const UrdfJoint &j) {
        auto pf = body_frame.find(j.parent);
        if (pf == body_frame.end()) throw std::runtime_error("URDF: joint " + j.name + " has unknown parent link " + j.parent);
        const int pframe = pf->second;
        const int support = m.frame_parent[pframe];
        const SE3d placement = se3_mul(m.frame_placement[pframe], j.placement);
        if (j.type == "fixed") {
            m.add_frame(j.name, support, placement, FRAME_FIXED_JOINT);
            body_frame[j.child] = m.add_frame(j.child, support, placement, FRAME_BODY);
        } else if (j.type == "revolute" || j.type == "prismatic" || j.type == "continuous") {
            const bool rev = j.type == "revolute", cont = j.type == "continuous";
            const int first = rev ? IKB_J_RX : (cont ? IKB_J_RUBX : IKB_J_PX);   // X, Y, Z, unaligned follow in that order
            int type = first + 3;
            std::array<double, 3> ax = j.axis;
            bool aligned = false;
            for (int k = 0; k < 3 && !aligned; ++k)
                if (approx_unit(j.axis, k)) {
                    type = first + k;
                    ax = {0, 0, 0};
                    ax[k] = 1.0;
                    aligned = true;
                }
            if (!aligned) {
                const double n = std::sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
                if (!(n > 0)) throw std::runtime_error("URDF: joint " + j.name + " has a zero axis");
                for (auto &v : ax) v /= n;
            }
            // continuous: Pinocchio's URDF parser bounds both entries of (cos, sin) by -1.01 / +1.01 and ignores <limit>
            const int jid = cont ? m.add_joint(j.name, type, support, placement, ax, {-1.01, -1.01}, {1.01, 1.01})
                                 : m.add_joint(j.name, type, support, placement, ax, {j.lower}, {j.upper});
            m.add_frame(j.name, jid, se3_identity(), FRAME_JOINT);
            body_frame[j.child] = m.add_frame(j.child, jid, se3_identity(), FRAME_BODY);
        } else {
            throw std::runtime_error("URDF: joint type \"" + j.type + "\" (joint " + j.name + ") is not supported");
        }
        auto it = children.find(j.child);
        if (it != children.end())
            for (const UrdfJoint *c : it->second) visit(*c);
    }
};

}  // namespace

HostModel model_from_urdf(const std::string &xml, bool free_flyer) {
    XmlReader reader(xml);
    std::unique_ptr<XmlNode> root = reader.parse_document();
    if (root->name != "robot") throw std::runtime_error("URDF: root element is <" + root->name + ">, expected <robot>");

    std::vector<std::string> links;
    std::map<std::string, std::array<double, 4>> inertials;  // link -> mass, centre of mass in the link frame
    std::map<std::string, UrdfJoint> joints;  // std::map: byte-wise name order, as in urdfdom
    for (const auto &c : root->children) {
        if (c->name == "link") {
            const std::string *n = c->attr("name");
            if (!n) throw std::runtime_error("URDF: <link> without a name");
            links.push_back(*n);
            if (const XmlNode *ine = c->child("inertial"))
                if (const XmlNode *ms = ine->child("mass")) {
                    const XmlNode *o = ine->child("origin");
                    const auto xyz = parse_floats(o ? o->attr("xyz") : nullptr, 3, {0, 0, 0}, "inertial xyz");
                    inertials[*n] = {parse_floats(ms->attr("value"), 1, {0}, "mass value")[0], xyz[0], xyz[1], xyz[2]};
                }
        } else if (c->name == "joint") {
            UrdfJoint j;
            const std::string *n = c->attr("name"), *t = c->attr("type");
            if (!n || !t) throw std::runtime_error("URDF: <joint> needs name and type");
            j.name = *n;
            j.type = *t;
            const XmlNode *par = c->child("parent"), *chi = c->child("child");
            if (!par || !chi || !par->attr("link") || !chi->attr("link"))
                throw std::runtime_error("URDF: joint " + j.name + " needs <parent link> and <child link>");
            j.parent = *par->attr("link");
            j.child = *chi->attr("link");
            const XmlNode *o = c->child("origin");
            j.placement = origin_to_se3(parse_floats(o ? o->attr("xyz") : nullptr, 3, {0, 0, 0}, "xyz"),
                                        parse_floats(o ? o->attr("rpy") : nullptr, 3, {0, 0, 0}, "rpy"));
            const XmlNode *a = c->child("axis");
            auto av = parse_floats(a ? a->attr("xyz") : nullptr, 3, {1, 0, 0}, "axis xyz");
            j.axis = {av[0], av[1], av[2]};
            if (const XmlNode *l = c->child("limit")) {
                if (l->attr("lower")) j.lower = parse_floats(l->attr("lower"), 1, {0}, "lower")[0];
                if (l->attr("upper")) j.upper = parse_floats(l->attr("upper"), 1, {0}, "upper")[0];
            }
            if (!joints.emplace(j.name, j).second) throw std::runtime_error("URDF: duplicate joint " + j.name);
        }
    }
    if (links.empty()) throw std::runtime_error("URDF: no links");

    Builder b;
    std::map<std::string, bool> is_child;
    for (const auto &kv : joints) {
        b.children[kv.second.parent].push_back(&kv.second);
        is_child[kv.second.child] = true;
    }
    std::string root_link;
    int nroots = 0;
    for (const auto &l : links)
        if (!is_child.count(l)) {
            root_link = l;
            ++nroots;
        }
    if (nroots != 1) throw std::runtime_error("URDF: expected exactly one root link, found " + std::to_string(nroots));

    HostModel &m = b.m;
    m.add_joint("universe", IKB_J_UNIVERSE, 0, se3_identity(), {0, 0, 0}, {}, {});
    m.add_frame("universe", 0, se3_identity(), FRAME_OP);
    if (free_flyer) {
        const std::vector<double> hi(7, DBL_MAX), lo(7, -DBL_MAX);
        const int jid = m.add_joint("root_joint", IKB_J_FREEFLYER, 0, se3_identity(), {0, 0, 0}, lo, hi);
        m.add_frame("root_joint", jid, se3_identity(), FRAME_JOINT);
        b.body_frame[root_link] = m.add_frame(root_link, jid, se3_identity(), FRAME_BODY);
    } else {
        b.body_frame[root_link] = m.add_frame(root_link, 0, se3_identity(), FRAME_BODY);
    }
    auto it = b.children.find(root_link);
    if (it != b.children.end())
        for (const UrdfJoint *c : it->second) b.visit(*c);
    // Pinocchio appends every body's inertia to its supporting joint: mass and first moment in the joint frame
    std::vector<std::array<double, 3>> moment(m.njoints(), {0.0, 0.0, 0.0});
    for (const auto &kv : inertials) {
        auto bf = b.body_frame.find(kv.first);
        if (bf == b.body_frame.end()) continue;
        const SE3d &pl = m.frame_placement[bf->second];
        const int j = m.frame_parent[bf->second];
        const double ml = kv.second[0];
        m.mass[j] += ml;
        for (int i = 0; i < 3; ++i)
            moment[j][i] += ml * (pl[9 + i] + pl[3 * i] * kv.second[1] + pl[3 * i + 1] * kv.second[2] + pl[3 * i + 2] * kv.second[3]);
    }
    for (int j = 0; j < m.njoints(); ++j)
        if (m.mass[j] > 0)
            for (int i = 0; i < 3; ++i) m.com[j][i] = moment[j][i] / m.mass[j];
    return std::move(b.m);
}

}  // namespace ikb
