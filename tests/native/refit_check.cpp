// The BVH refit of b200rt_scene_update (csrc/prim_box.hpp: node_links, refit_links_host, refit_host — the host twin of
// csrc/refit.cuh) against the host SAH builder (csrc/bvh_build.hpp) and the node packing (csrc/node_layout.hpp), with g++:
//   links   every inner node but the root has exactly the parent (node, side) whose reference names it, and every leaf's hit
//           id the slot that holds it; primitives without a leaf (invalid boxes, the up-front one) have none
//   noop    refitting from the records the tree was built from reproduces the builder's nodes byte for byte
//   moved   after random moves that keep each primitive's validity, every child box is pack_node of the exact union of its
//           subtree's padded leaf boxes, over several successive refits
//   karras  the same on a small hand-built Karras-numbered tree (children numbered below their parents, leaves in Morton order)
// over random and degenerate primitives: coincident, thin, huge, inverted and NaN.  Prints one line per check; exit 1 on failure.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include "../../shirley_raytracing_rs_b200/csrc/bvh_build.hpp"
#include "../../shirley_raytracing_rs_b200/csrc/node_layout.hpp"
#include "../../shirley_raytracing_rs_b200/csrc/prim_box.hpp"

using namespace b200rt;

struct F4 { float x, y, z, w; };
struct Geom { F4 g0, g1; };

static int failures = 0;
#define CHECK(cond, ...) do { if (!(cond)) { if (failures++ < 20) { printf("FAIL %s:%d: ", __FILE__, __LINE__); printf(__VA_ARGS__); printf("\n"); } } } while (0)

struct Scene {
    std::vector<uint32_t> type;
    std::vector<Geom> geom;
};

// one random primitive of `type` near centre c with scale s; `kind` picks a degenerate case
static Geom random_geom(std::mt19937& rng, uint32_t type, const float c[3], float s, int kind) {
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    Geom g{};
    const float t = kind == 1 ? 0.f : (kind == 2 ? 1e-7f * s : s * (0.05f + 0.5f * std::fabs(u(rng))));   // thin: zero or sub-pad thickness
    if (type == B200RT_PRIM_SPHERE) g.g0 = {c[0], c[1], c[2], kind == 3 ? -t - 0.1f : t};                 // kind 3: negative radius
    else if (type == B200RT_PRIM_BOX) {
        g.g0 = {c[0], c[1], c[2], 0.f};
        g.g1 = {c[0] + t, c[1] + (kind == 3 ? -1.f : t + 0.01f * s), c[2] + t * 0.5f, 0.f};                // kind 3: inverted y
    } else {
        g.g0 = {c[0] - t, c[0] + t, c[1] - 2 * t, kind == 3 ? c[1] - 3 * t - 1.f : c[1] + 2 * t};
        g.g1 = {c[2], 0.f, 0.f, 0.f};
    }
    if (kind == 4) g.g0.x = NAN;
    return g;
}

static Scene random_scene(std::mt19937& rng, int n, float spread) {
    Scene sc;
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    std::vector<float> centres;
    for (int i = 0; i < n; ++i) {
        float c[3] = {spread * u(rng), spread * u(rng), spread * u(rng)};
        if (i > 0 && rng() % 6 == 0) { const int j = rng() % i; for (int k = 0; k < 3; ++k) c[k] = centres[3 * j + k]; }   // coincident
        centres.insert(centres.end(), c, c + 3);
        const uint32_t type = rng() % 5;
        const int kind = rng() % 10 < 6 ? 0 : 1 + rng() % 4;
        const float s = rng() % 20 == 0 ? spread * 1e3f : 1.f;                                                                // huge
        sc.type.push_back(type);
        sc.geom.push_back(random_geom(rng, type, c, s, kind));
    }
    return sc;
}

// b200rt_scene_create's tree: valid boxes only, the first valid primitive kept out (as an up-front one is), padded, host SAH,
// packed with pack_node.  Returns the nodes as 16 floats each.
struct Tree { std::vector<float> nodes; std::vector<uint8_t> valid; int up_front = -1; };
static float scene_pad(const Scene& sc, std::vector<uint8_t>* valid) {
    float max_abs = 0.f;
    valid->assign(sc.type.size(), 0);
    for (size_t i = 0; i < sc.type.size(); ++i) {
        float lo[3], hi[3];
        prim_box(sc.type[i], sc.geom[i].g0, sc.geom[i].g1, lo, hi);
        (*valid)[i] = box_valid(lo, hi);
        if ((*valid)[i]) max_abs = std::max(max_abs, box_max_abs(lo, hi));
    }
    return box_pad_for(max_abs);
}
static Tree build_tree(const Scene& sc) {
    Tree t;
    const float pad = scene_pad(sc, &t.valid);
    std::vector<BuildPrim> bp;
    for (size_t i = 0; i < sc.type.size(); ++i) {
        if (!t.valid[i]) continue;
        if (t.up_front < 0 && sc.type.size() > 3) { t.up_front = (int)i; continue; }
        BuildPrim p;
        prim_box(sc.type[i], sc.geom[i].g0, sc.geom[i].g1, p.box.lo, p.box.hi);
        for (int k = 0; k < 3; ++k) p.centroid[k] = 0.5f * (p.box.lo[k] + p.box.hi[k]);
        pad_box(p.box.lo, p.box.hi, pad);
        p.code = (int)((sc.type[i] << 28) | i);
        bp.push_back(p);
    }
    BvhBuildResult r = build_bvh(std::move(bp));
    t.nodes.resize(r.nodes.size() * 16);
    for (size_t i = 0; i < r.nodes.size(); ++i) {
        const float* q = r.nodes[i].q;
        int ref0, ref1;
        memcpy(&ref0, &q[12], 4); memcpy(&ref1, &q[13], 4);
        pack_node(q, q + 3, q + 6, q + 9, ref0, ref1, &t.nodes[16 * i]);
    }
    return t;
}

static void check_links(const std::vector<float>& nodes, size_t n_prims, const std::vector<uint8_t>& has_leaf, const char* what) {
    const uint32_t n_nodes = (uint32_t)(nodes.size() / 16);
    std::vector<int> parent, leaf;
    refit_links_host(nodes.data(), n_nodes, (uint32_t)n_prims, &parent, &leaf);
    CHECK(n_nodes == 0 || parent[0] == -1, "%s: root has a parent", what);
    for (uint32_t i = 1; i < n_nodes; ++i) {
        CHECK(parent[i] >= 0, "%s: node %u has no parent", what, i);
        if (parent[i] >= 0) CHECK(node_ref(&nodes[16 * (parent[i] >> 1)], parent[i] & 1) == (int)i, "%s: node %u: parent slot does not name it", what, i);
    }
    for (size_t id = 0; id < n_prims; ++id) {
        CHECK((leaf[id] >= 0) == (has_leaf[id] != 0), "%s: hit id %zu: leaf slot %d, has_leaf %d", what, id, leaf[id], has_leaf[id]);
        if (leaf[id] >= 0) {
            const int r = node_ref(&nodes[16 * (leaf[id] >> 1)], leaf[id] & 1);
            CHECK(r < 0 && ((uint32_t)~r & LEAF_ID_MASK) == id, "%s: hit id %zu: slot holds ref %d", what, id, r);
        }
    }
}

// expected node array: each child box the builders' way (box_grow over the subtree's padded leaf boxes), packed
static void subtree_box(const std::vector<float>& nodes, int ref, const std::vector<Geom>& geom, float pad, HostBox& b) {
    if (ref == EMPTY_CHILD) return;
    if (ref < 0) {
        const uint32_t code = (uint32_t)~ref;
        HostBox p;
        prim_box(code >> 28, geom[code & LEAF_ID_MASK].g0, geom[code & LEAF_ID_MASK].g1, p.lo, p.hi);
        pad_box(p.lo, p.hi, pad);
        detail::box_grow(b, p);
        return;
    }
    for (int s = 0; s < 2; ++s) subtree_box(nodes, node_ref(&nodes[16 * ref], s), geom, pad, b);
}
static std::vector<float> expected_nodes(const std::vector<float>& nodes, const std::vector<Geom>& geom, float pad) {
    std::vector<float> out(nodes.size());
    for (size_t i = 0; i < nodes.size() / 16; ++i) {
        HostBox b[2];
        for (int s = 0; s < 2; ++s) { detail::box_init(b[s]); subtree_box(nodes, node_ref(&nodes[16 * i], s), geom, pad, b[s]); }
        pack_node(b[0].lo, b[0].hi, b[1].lo, b[1].hi, node_ref(&nodes[16 * i], 0), node_ref(&nodes[16 * i], 1), &out[16 * i]);
    }
    return out;
}

// moves and resizes every primitive, keeping whether its box is valid
static void move_scene(std::mt19937& rng, Scene& sc, float spread) {
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    for (size_t i = 0; i < sc.type.size(); ++i) {
        std::vector<uint8_t> was;
        Scene one{{sc.type[i]}, {sc.geom[i]}};
        scene_pad(one, &was);
        for (int attempt = 0; attempt < 50; ++attempt) {
            float c[3] = {spread * u(rng), spread * u(rng), spread * u(rng)};
            Scene cand{{sc.type[i]}, {random_geom(rng, sc.type[i], c, rng() % 20 == 0 ? spread * 1e3f : 1.f, rng() % 10 < 6 ? 0 : 1 + rng() % 4)}};
            std::vector<uint8_t> now;
            scene_pad(cand, &now);
            if (now[0] == was[0]) { sc.geom[i] = cand.geom[0]; break; }
        }
    }
}

int main() {
    std::mt19937 rng(12345);
    int trees = 0;
    for (int round = 0; round < 60; ++round) {
        const int sizes[] = {0, 1, 2, 3, 5, 17, 64, 300, 2500};
        const int n = sizes[round % 9];
        const float spread = round % 3 == 0 ? 3.f : (round % 3 == 1 ? 30.f : 2000.f);
        Scene sc = random_scene(rng, n, spread);
        Tree t = build_tree(sc);
        std::vector<uint8_t> has_leaf(t.valid);
        if (t.up_front >= 0) has_leaf[t.up_front] = 0;
        check_links(t.nodes, sc.type.size(), has_leaf, "sah");

        std::vector<uint8_t> v;
        float pad = scene_pad(sc, &v);
        std::vector<float> refit(t.nodes);
        refit_host(refit.data(), (uint32_t)(refit.size() / 16), sc.geom.data(), pad);
        CHECK(refit.size() == t.nodes.size() && memcmp(refit.data(), t.nodes.data(), refit.size() * 4) == 0, "noop: round %d (n %d) nodes differ", round, n);

        for (int step = 0; step < 4; ++step) {
            move_scene(rng, sc, spread * (step + 1));
            pad = scene_pad(sc, &v);
            CHECK(v == t.valid, "round %d: a move changed validity", round);
            refit_host(refit.data(), (uint32_t)(refit.size() / 16), sc.geom.data(), pad);
            const std::vector<float> want = expected_nodes(t.nodes, sc.geom, pad);
            CHECK(memcmp(refit.data(), want.data(), want.size() * 4) == 0, "moved: round %d step %d (n %d) nodes differ", round, step, n);
        }
        ++trees;
    }
    if (failures == 0) printf("links ok\n");
    if (failures == 0) printf("noop ok\n");
    if (failures == 0) printf("moved ok\n");

    {   // Karras numbering: 5 leaves in Morton order (hit ids 3 0 4 1 2); node 0 = root, its children 2 and 3, node 1 under node 2
        Scene sc;
        std::mt19937 r2(7);
        for (int i = 0; i < 5; ++i) { float c[3] = {(float)i, 0.5f * i, -1.f * i}; sc.type.push_back(i % 5); sc.geom.push_back(random_geom(r2, i % 5, c, 1.f, 0)); }
        const int order[5] = {3, 0, 4, 1, 2};
        auto leaf = [&](int k) { return ~(int)((sc.type[order[k]] << 28) | (uint32_t)order[k]); };
        const int refs[4][2] = {{2, 3}, {leaf(1), leaf(2)}, {leaf(0), 1}, {leaf(3), leaf(4)}};
        std::vector<float> nodes(4 * 16, 0.f);
        for (int i = 0; i < 4; ++i) { memcpy(&nodes[16 * i + NODE_REF], &refs[i][0], 4); memcpy(&nodes[16 * i + NODE_REF + 1], &refs[i][1], 4); }
        std::vector<int> parent, slot;
        refit_links_host(nodes.data(), 4, 5, &parent, &slot);
        CHECK(parent[0] == -1 && parent[2] == 0 && parent[3] == 1 && parent[1] == 2 * 2 + 1, "karras: parents %d %d %d %d", parent[0], parent[1], parent[2], parent[3]);
        const int want_slot[5] = {2 * 1 + 0, 2 * 3 + 0, 2 * 3 + 1, 2 * 2 + 0, 2 * 1 + 1};   // by hit id 0..4
        for (int id = 0; id < 5; ++id) CHECK(slot[id] == want_slot[id], "karras: hit id %d slot %d, want %d", id, slot[id], want_slot[id]);
        check_links(nodes, 5, std::vector<uint8_t>(5, 1), "karras");
        std::vector<uint8_t> v;
        for (int step = 0; step < 3; ++step) {
            const float pad = scene_pad(sc, &v);
            refit_host(nodes.data(), 4, sc.geom.data(), pad);
            const std::vector<float> want = expected_nodes(nodes, sc.geom, pad);
            CHECK(memcmp(nodes.data(), want.data(), want.size() * 4) == 0, "karras: step %d nodes differ", step);
            move_scene(r2, sc, 10.f);
        }
        if (failures == 0) printf("karras ok\n");
    }
    printf("%d trees\n", trees);
    return failures ? 1 : 0;
}
