// scene_host.cpp - the host-side scene of libptap (C ABI ptap_scene_*): replaces class Scene
// (Scene.h:21-39, Scene.cpp:3-396) including the mesh import the reference delegates to Assimp.
//
// What is kept: the seven public arrays and their layouts, one-vertex-per-face-corner import scaled by
// BASE_MODEL_SCALE, per-mesh bounding boxes, the 25^3 grid binning rule, and the scene hard-coded in
// Scene::Scene.  What is new: an in-repo Wavefront reader (Assimp is not vendored and not installed), a parser for
// the Config.txt schema the reference only sketched, synthetic meshes for the large-scene configs, and a counting
// (two-pass, CSR) grid build instead of vector<vector<int>>.
#include <algorithm>
#include <array>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/ptap.h"
#include "bvh_build.h"

namespace {

constexpr float kFloatMax = 9999999.0f, kFloatMin = -9999990.0f;   // Config.h:5-6
constexpr float kBaseModelScale = 1000;                            // Config.h:17

}  // namespace

struct ptap_scene {
    std::vector<PtapModel> models;
    std::vector<PtapMesh> meshes;
    std::vector<PtapVertex> vertices;
    std::vector<PtapTriangle> triangles;
    std::vector<PtapGrid> grids;
    std::vector<PtapVoxel> voxels;
    std::vector<int32_t> refs;
    int32_t grid_dim[3] = {25, 25, 25};
    // Config.txt extensions (not part of the reference's Scene)
    int32_t cfg_width = 0, cfg_height = 0, cfg_iter = 0, cfg_depth = 0;
    bool cfg_has_camera = false;
    PtapCamera cfg_camera{{0.0f, 0.0f, 920.0f}, {-10.0f, -4.0f, 900.0f}, {20.0f, 16.0f}, 0, 0u};
    // optional BVH (ptap_scene_build_bvh); invalidated by any mesh edit
    ptap::BvhBuildResult bvh;
    bool have_bvh = false;
    bool have_recs = false;       // st_recs holds the triangle records of the current meshes (ptap_scene_pack_triangles / ptap_scene_build_bvh)
    int bvh_nnodes = 0;
    // upload-bound copies of the BVH arrays and the triangle records, page-locked when a CUDA device exists (plain malloc otherwise)
    struct Staging {
        void* p = nullptr; size_t bytes = 0; bool pinned = false;
        void release() { if (p) { if (pinned) cudaFreeHost(p); else free(p); } p = nullptr; bytes = 0; pinned = false; }
        void* fill(const void* src, size_t n)
        {
            release();
            if (n == 0) return nullptr;
            if (cudaHostAlloc(&p, n, cudaHostAllocDefault) == cudaSuccess) pinned = true;
            else { (void)cudaGetLastError(); p = malloc(n); pinned = false; }
            if (p) { memcpy(p, src, n); bytes = n; }
            return p;
        }
        ~Staging() { release(); }
    } st_nodes, st_tri_id, st_recs;
    std::string err;
};

namespace {

// ---- glm 0.9.6.3 restated (column-major float[16], m(c,r) = M[4c+r]); evaluation order as in
// external/include/glm/gtc/matrix_transform.inl:40-134 and glm/detail/type_mat4x4.inl:37-92, 686-704 ------------

struct M4 { float v[16]; };

M4 identity() { M4 m{}; m.v[0] = m.v[5] = m.v[10] = m.v[15] = 1.0f; return m; }

M4 mul(const M4& a, const M4& b)           // type_mat4x4.inl:686-704: ((A0*b0 + A1*b1) + A2*b2) + A3*b3 per column
{
    M4 r;
    for (int c = 0; c < 4; ++c)
        for (int k = 0; k < 4; ++k)
            r.v[4 * c + k] = ((a.v[k] * b.v[4 * c] + a.v[4 + k] * b.v[4 * c + 1]) + a.v[8 + k] * b.v[4 * c + 2]) + a.v[12 + k] * b.v[4 * c + 3];
    return r;
}

M4 scaleM(const float s[3])                // matrix_transform.inl:122-134 on the identity
{
    M4 m = identity(), r;
    for (int k = 0; k < 4; ++k) { r.v[k] = m.v[k] * s[0]; r.v[4 + k] = m.v[4 + k] * s[1]; r.v[8 + k] = m.v[8 + k] * s[2]; r.v[12 + k] = m.v[12 + k]; }
    return r;
}

M4 translateM(const float t[3])            // matrix_transform.inl:40-49: m[0]*v0 + m[1]*v1 + m[2]*v2 + m[3]
{
    M4 m = identity(), r = m;
    for (int k = 0; k < 4; ++k) r.v[12 + k] = ((m.v[k] * t[0] + m.v[4 + k] * t[1]) + m.v[8 + k] * t[2]) + m.v[12 + k];
    return r;
}

M4 rotateM(float angle, const float axis_in[3])   // matrix_transform.inl:52-85 on the identity
{
    const float c = std::cos(angle), s = std::sin(angle);
    const float len2 = (axis_in[0] * axis_in[0] + axis_in[1] * axis_in[1]) + axis_in[2] * axis_in[2];
    const float il = 1.0f / std::sqrt(len2);
    const float ax[3] = {axis_in[0] * il, axis_in[1] * il, axis_in[2] * il};
    const float t[3] = {(1.0f - c) * ax[0], (1.0f - c) * ax[1], (1.0f - c) * ax[2]};
    float R[3][3];
    R[0][0] = c + t[0] * ax[0];
    R[0][1] = 0 + t[0] * ax[1] + s * ax[2];
    R[0][2] = 0 + t[0] * ax[2] - s * ax[1];
    R[1][0] = 0 + t[1] * ax[0] - s * ax[2];
    R[1][1] = c + t[1] * ax[1];
    R[1][2] = 0 + t[1] * ax[2] + s * ax[0];
    R[2][0] = 0 + t[2] * ax[0] + s * ax[1];
    R[2][1] = 0 + t[2] * ax[1] - s * ax[0];
    R[2][2] = c + t[2] * ax[2];
    M4 m = identity(), r;
    for (int col = 0; col < 3; ++col)
        for (int k = 0; k < 4; ++k)
            r.v[4 * col + k] = (m.v[k] * R[col][0] + m.v[4 + k] * R[col][1]) + m.v[8 + k] * R[col][2];
    for (int k = 0; k < 4; ++k) r.v[12 + k] = m.v[12 + k];
    return r;
}

M4 inverseM(const M4& M)                   // type_mat4x4.inl:37-92
{
    auto m = [&](int c, int r) { return M.v[4 * c + r]; };
    const float C00 = m(2, 2) * m(3, 3) - m(3, 2) * m(2, 3), C02 = m(1, 2) * m(3, 3) - m(3, 2) * m(1, 3), C03 = m(1, 2) * m(2, 3) - m(2, 2) * m(1, 3);
    const float C04 = m(2, 1) * m(3, 3) - m(3, 1) * m(2, 3), C06 = m(1, 1) * m(3, 3) - m(3, 1) * m(1, 3), C07 = m(1, 1) * m(2, 3) - m(2, 1) * m(1, 3);
    const float C08 = m(2, 1) * m(3, 2) - m(3, 1) * m(2, 2), C10 = m(1, 1) * m(3, 2) - m(3, 1) * m(1, 2), C11 = m(1, 1) * m(2, 2) - m(2, 1) * m(1, 2);
    const float C12 = m(2, 0) * m(3, 3) - m(3, 0) * m(2, 3), C14 = m(1, 0) * m(3, 3) - m(3, 0) * m(1, 3), C15 = m(1, 0) * m(2, 3) - m(2, 0) * m(1, 3);
    const float C16 = m(2, 0) * m(3, 2) - m(3, 0) * m(2, 2), C18 = m(1, 0) * m(3, 2) - m(3, 0) * m(1, 2), C19 = m(1, 0) * m(2, 2) - m(2, 0) * m(1, 2);
    const float C20 = m(2, 0) * m(3, 1) - m(3, 0) * m(2, 1), C22 = m(1, 0) * m(3, 1) - m(3, 0) * m(1, 1), C23 = m(1, 0) * m(2, 1) - m(2, 0) * m(1, 1);
    const float F0[4] = {C00, C00, C02, C03}, F1[4] = {C04, C04, C06, C07}, F2[4] = {C08, C08, C10, C11};
    const float F3[4] = {C12, C12, C14, C15}, F4[4] = {C16, C16, C18, C19}, F5[4] = {C20, C20, C22, C23};
    const float V0[4] = {m(1, 0), m(0, 0), m(0, 0), m(0, 0)}, V1[4] = {m(1, 1), m(0, 1), m(0, 1), m(0, 1)};
    const float V2[4] = {m(1, 2), m(0, 2), m(0, 2), m(0, 2)}, V3[4] = {m(1, 3), m(0, 3), m(0, 3), m(0, 3)};
    const float SA[4] = {+1, -1, +1, -1}, SB[4] = {-1, +1, -1, +1};
    M4 inv;
    for (int k = 0; k < 4; ++k) {
        inv.v[0 + k] = ((V1[k] * F0[k] - V2[k] * F1[k]) + V3[k] * F2[k]) * SA[k];
        inv.v[4 + k] = ((V0[k] * F0[k] - V2[k] * F3[k]) + V3[k] * F4[k]) * SB[k];
        inv.v[8 + k] = ((V0[k] * F1[k] - V1[k] * F3[k]) + V3[k] * F5[k]) * SA[k];
        inv.v[12 + k] = ((V0[k] * F2[k] - V1[k] * F4[k]) + V2[k] * F5[k]) * SB[k];
    }
    const float d0 = m(0, 0) * inv.v[0], d1 = m(0, 1) * inv.v[4], d2 = m(0, 2) * inv.v[8], d3 = m(0, 3) * inv.v[12];
    const float ood = 1.0f / ((d0 + d1) + (d2 + d3));
    for (float& x : inv.v) x = x * ood;
    return inv;
}

// ---- meshes ---------------------------------------------------------------------------------------------------

void bbUpdate(PtapMesh& mesh, const float* p)      // BoundingBox::update, Primitive.h:49-58
{
    for (int k = 0; k < 3; ++k) {
        mesh.bb_min[k] = mesh.bb_min[k] > p[k] ? p[k] : mesh.bb_min[k];
        mesh.bb_max[k] = mesh.bb_max[k] < p[k] ? p[k] : mesh.bb_max[k];
    }
}

PtapMesh emptyMesh()
{
    PtapMesh m{};
    for (int k = 0; k < 3; ++k) { m.bb_min[k] = kFloatMax; m.bb_max[k] = kFloatMin; }   // Primitive.h:38-47
    return m;
}

// Appends a mesh given final (already scaled) vertices and local indices, the way processMesh does (Scene.cpp:264-291).
int appendMesh(ptap_scene* s, const PtapVertex* verts, int nverts, const int32_t* idx, int ntris)
{
    PtapMesh mesh = emptyMesh();
    mesh.v_start = (int)s->vertices.size();
    for (int i = 0; i < nverts; ++i) { s->vertices.push_back(verts[i]); bbUpdate(mesh, verts[i].position); }
    mesh.v_end = (int)s->vertices.size();
    mesh.t_start = (int)s->triangles.size();
    for (int t = 0; t < ntris; ++t) {
        PtapTriangle tri;
        for (int k = 0; k < 3; ++k) tri.v[k] = mesh.v_start + idx[3 * t + k];
        s->triangles.push_back(tri);
    }
    mesh.t_end = (int)s->triangles.size();
    s->meshes.push_back(mesh);
    s->have_bvh = false; s->have_recs = false;
    return (int)s->meshes.size() - 1;
}

// Wavefront reader reproducing Assimp's default import for the subset the reference uses (no JoinIdenticalVertices):
// one vertex per face corner in file order; polygons are fan-triangulated; missing normals become the face normal.
int loadObj(ptap_scene* s, const std::string& path_in, int32_t* mesh_index)
{
    std::string path = path_in;
    for (char& c : path) if (c == '\\') c = '/';        // the reference uses Windows separators (Scene.cpp:7-27)
    FILE* f = fopen(path.c_str(), "r");
    if (!f) { s->err = "Unable to open file \"" + path_in + "\"."; return PTAP_E_IO; }
    std::vector<float> v, vn;
    std::vector<PtapVertex> verts;
    std::vector<int32_t> idx;
    std::vector<char> line(1 << 16);
    int lineno = 0;
    while (fgets(line.data(), (int)line.size(), f)) {
        ++lineno;
        const char* p = line.data();
        while (*p == ' ' || *p == '\t') ++p;
        if (p[0] == 'v' && (p[1] == ' ' || p[1] == '\t')) {
            float x, y, z;
            if (sscanf(p + 2, "%f %f %f", &x, &y, &z) != 3) { fclose(f); s->err = path + ": bad vertex at line " + std::to_string(lineno); return PTAP_E_PARSE; }
            v.push_back(x); v.push_back(y); v.push_back(z);
        } else if (p[0] == 'v' && p[1] == 'n') {
            float x, y, z;
            if (sscanf(p + 3, "%f %f %f", &x, &y, &z) != 3) { fclose(f); s->err = path + ": bad normal at line " + std::to_string(lineno); return PTAP_E_PARSE; }
            vn.push_back(x); vn.push_back(y); vn.push_back(z);
        } else if (p[0] == 'f' && (p[1] == ' ' || p[1] == '\t')) {
            char* q = const_cast<char*>(p + 2);
            std::vector<PtapVertex> corner;
            std::vector<bool> has_n;
            for (;;) {
                while (*q == ' ' || *q == '\t') ++q;
                if (*q == '\0' || *q == '\n' || *q == '\r' || *q == '#') break;
                char* e;
                long iv = strtol(q, &e, 10), in = 0;
                if (e == q) { fclose(f); s->err = path + ": bad face at line " + std::to_string(lineno); return PTAP_E_PARSE; }
                q = e;
                if (*q == '/') { ++q; if (*q != '/') strtol(q, &q, 10); if (*q == '/') { ++q; in = strtol(q, &q, 10); } }
                const long nv = (long)v.size() / 3, nn = (long)vn.size() / 3;
                if (iv < 0) iv = nv + 1 + iv;
                if (in < 0) in = nn + 1 + in;
                if (iv < 1 || iv > nv || in > nn) { fclose(f); s->err = path + ": index out of range at line " + std::to_string(lineno); return PTAP_E_PARSE; }
                PtapVertex pv{};
                for (int k = 0; k < 3; ++k) {
                    pv.position[k] = v[3 * (iv - 1) + k] * kBaseModelScale;                       // convertFromVector3D, Scene.cpp:255-262
                    pv.normal[k] = in > 0 ? vn[3 * (in - 1) + k] * kBaseModelScale : 0.0f;
                }
                corner.push_back(pv); has_n.push_back(in > 0);
            }
            if (corner.size() < 3) { fclose(f); s->err = path + ": face with fewer than 3 corners at line " + std::to_string(lineno); return PTAP_E_PARSE; }
            for (size_t k = 1; k + 1 < corner.size(); ++k) {
                PtapVertex tri[3] = {corner[0], corner[k], corner[k + 1]};
                const bool hn[3] = {has_n[0], has_n[k], has_n[k + 1]};
                if (!(hn[0] && hn[1] && hn[2])) {        // no vn: use the geometric normal, scaled like imported ones
                    const float* a = tri[0].position; const float* b = tri[1].position; const float* c = tri[2].position;
                    const double e1[3] = {(double)b[0] - a[0], (double)b[1] - a[1], (double)b[2] - a[2]}, e2[3] = {(double)c[0] - a[0], (double)c[1] - a[1], (double)c[2] - a[2]};
                    double n[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
                    const double l = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
                    for (int j = 0; j < 3; ++j) if (!hn[j]) for (int d = 0; d < 3; ++d) tri[j].normal[d] = l > 0 ? (float)(n[d] / l * kBaseModelScale) : 0.0f;
                }
                for (int j = 0; j < 3; ++j) { idx.push_back((int32_t)verts.size()); verts.push_back(tri[j]); }
            }
        }
    }
    fclose(f);
    if (verts.empty()) { s->err = path + ": no faces"; return PTAP_E_PARSE; }
    const int mi = appendMesh(s, verts.data(), (int)verts.size(), idx.data(), (int)idx.size() / 3);
    if (mesh_index) *mesh_index = mi;
    return PTAP_OK;
}

uint32_t hash32(uint32_t a)        // integer hash for the synthetic displacement (not the reference's utilHash)
{
    a ^= a >> 16; a *= 0x7feb352du; a ^= a >> 15; a *= 0x846ca68bu; a ^= a >> 16;
    return a;
}

// Displaced icosphere: 20 * 4^level triangles, shared vertices displaced radially by 1 + displacement * noise, where
// the noise is a smooth sum of a few sinusoids plus a small per-vertex hash term (SURVEY.md 8d configs 2 and 4).
int addIcosphere(ptap_scene* s, int level, float radius, float displacement, uint32_t seed, int32_t* mesh_index)
{
    if (level < 0 || level > 10) { s->err = "icosphere level must be in [0, 10]"; return PTAP_E_INVALID; }
    std::vector<double> pos;
    std::vector<int> tri;
    const double t = (1.0 + std::sqrt(5.0)) / 2.0;
    const double base[12][3] = {{-1, t, 0}, {1, t, 0}, {-1, -t, 0}, {1, -t, 0}, {0, -1, t}, {0, 1, t}, {0, -1, -t}, {0, 1, -t}, {t, 0, -1}, {t, 0, 1}, {-t, 0, -1}, {-t, 0, 1}};
    for (auto& b : base) { const double l = std::sqrt(b[0] * b[0] + b[1] * b[1] + b[2] * b[2]); pos.push_back(b[0] / l); pos.push_back(b[1] / l); pos.push_back(b[2] / l); }
    const int faces[20][3] = {{0, 11, 5}, {0, 5, 1}, {0, 1, 7}, {0, 7, 10}, {0, 10, 11}, {1, 5, 9}, {5, 11, 4}, {11, 10, 2}, {10, 7, 6}, {7, 1, 8},
                              {3, 9, 4}, {3, 4, 2}, {3, 2, 6}, {3, 6, 8}, {3, 8, 9}, {4, 9, 5}, {2, 4, 11}, {6, 2, 10}, {8, 6, 7}, {9, 8, 1}};
    for (auto& fc : faces) { tri.push_back(fc[0]); tri.push_back(fc[1]); tri.push_back(fc[2]); }
    for (int l = 0; l < level; ++l) {
        std::unordered_map<uint64_t, int> mid;
        mid.reserve(tri.size() * 2);
        auto midpoint = [&](int a, int b) {
            const uint64_t key = a < b ? ((uint64_t)a << 32) | (uint32_t)b : ((uint64_t)b << 32) | (uint32_t)a;
            auto it = mid.find(key);
            if (it != mid.end()) return it->second;
            double m[3] = {pos[3 * a] + pos[3 * b], pos[3 * a + 1] + pos[3 * b + 1], pos[3 * a + 2] + pos[3 * b + 2]};
            const double len = std::sqrt(m[0] * m[0] + m[1] * m[1] + m[2] * m[2]);
            const int id = (int)pos.size() / 3;
            pos.push_back(m[0] / len); pos.push_back(m[1] / len); pos.push_back(m[2] / len);
            mid.emplace(key, id);
            return id;
        };
        std::vector<int> next; next.reserve(tri.size() * 4);
        for (size_t i = 0; i < tri.size(); i += 3) {
            const int a = tri[i], b = tri[i + 1], c = tri[i + 2];
            const int ab = midpoint(a, b), bc = midpoint(b, c), ca = midpoint(c, a);
            const int sub[12] = {a, ab, ca, b, bc, ab, c, ca, bc, ab, bc, ca};
            next.insert(next.end(), sub, sub + 12);
        }
        tri.swap(next);
    }
    const int nv = (int)pos.size() / 3;
    std::vector<double> disp(nv);
    const double ph = (seed % 1000) * 0.01;
    for (int i = 0; i < nv; ++i) {
        const double x = pos[3 * i], y = pos[3 * i + 1], z = pos[3 * i + 2];
        const double smooth = 0.5 * std::sin(5 * x + ph) * std::cos(4 * y - ph) + 0.3 * std::sin(9 * z + 2 * ph) * std::sin(7 * x) + 0.2 * std::cos(13 * y + 3 * z);
        const double rough = (hash32((uint32_t)i * 2654435761u + seed) & 0xffff) / 65535.0 - 0.5;
        disp[i] = 1.0 + displacement * (smooth + 0.1 * rough);
    }
    // per-vertex normals of the displaced surface (area-weighted), then one vertex per face corner like the OBJ import
    std::vector<double> P(3 * (size_t)nv), Nrm(3 * (size_t)nv, 0.0);
    for (int i = 0; i < nv; ++i) for (int k = 0; k < 3; ++k) P[3 * i + k] = pos[3 * i + k] * disp[i];
    for (size_t i = 0; i < tri.size(); i += 3) {
        const double* a = &P[3 * tri[i]]; const double* b = &P[3 * tri[i + 1]]; const double* c = &P[3 * tri[i + 2]];
        const double e1[3] = {b[0] - a[0], b[1] - a[1], b[2] - a[2]}, e2[3] = {c[0] - a[0], c[1] - a[1], c[2] - a[2]};
        const double n[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
        for (int j = 0; j < 3; ++j) for (int k = 0; k < 3; ++k) Nrm[3 * tri[i + j] + k] += n[k];
    }
    std::vector<PtapVertex> verts(tri.size());
    std::vector<int32_t> idx(tri.size());
    const double unit = (double)radius / kBaseModelScale;     // OBJ-space radius; the import scales by BASE_MODEL_SCALE
    for (size_t i = 0; i < tri.size(); ++i) {
        const int vi = tri[i];
        const double l = std::sqrt(Nrm[3 * vi] * Nrm[3 * vi] + Nrm[3 * vi + 1] * Nrm[3 * vi + 1] + Nrm[3 * vi + 2] * Nrm[3 * vi + 2]);
        PtapVertex pv{};
        for (int k = 0; k < 3; ++k) {
            pv.position[k] = (float)(P[3 * vi + k] * unit) * kBaseModelScale;
            pv.normal[k] = (float)(l > 0 ? Nrm[3 * vi + k] / l : pos[3 * vi + k]) * kBaseModelScale;
        }
        verts[i] = pv; idx[i] = (int32_t)i;
    }
    const int mi = appendMesh(s, verts.data(), (int)verts.size(), idx.data(), (int)tri.size() / 3);
    if (mesh_index) *mesh_index = mi;
    return PTAP_OK;
}

// ---- grid build: Scene::addMeshesToGrid (Scene.cpp:318-396) + computeVoxelIndex (Scene.cpp:293-316) as a counting sort -------

int f2iX86(float x) { return (x >= -2147483648.0f && x < 2147483648.0f) ? (int)x : (-2147483647 - 1); }
int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

// Fails (PTAP_E_INVALID, s->err names the count, the scene's previous grids kept) when the grids would hold more than 2^31 - 1 cells or
// references in all: voxels and reference positions are 32-bit.  Both counts are taken before any per-cell work.
int buildGrids(ptap_scene* s, int gx, int gy, int gz)
{
    const int gd[3] = {gx, gy, gz};
    const size_t ncell = (size_t)gx * gy * gz;
    // grid list (Scene.cpp:322-339) and every listed triangle's voxel index box
    std::vector<int> grid_of_mesh(s->meshes.size(), -1), grid_model;
    std::vector<std::array<float, 3>> widths;
    std::vector<std::vector<int>> lohis;
    long long total = 0;
    for (size_t i = 0; i < s->models.size(); ++i) {
        const int mi = s->models[i].mesh_index;
        if (grid_of_mesh[mi] >= 0) continue;                                                // Scene.cpp:325-329
        grid_of_mesh[mi] = (int)grid_model.size();
        grid_model.push_back((int)i);
        const PtapMesh& mesh = s->meshes[mi];
        std::array<float, 3> w;
        for (int k = 0; k < 3; ++k) w[k] = (mesh.bb_max[k] - mesh.bb_min[k]) / gd[k];   // Scene.cpp:341-347
        std::vector<int> lohi((size_t)std::max(0, mesh.t_end - mesh.t_start) * 6);
        for (int t = mesh.t_start; t < mesh.t_end; ++t) {
            float tmn[3] = {kFloatMax, kFloatMax, kFloatMax}, tmx[3] = {kFloatMin, kFloatMin, kFloatMin};
            for (int k = 0; k < 3; ++k) {
                const float* p = s->vertices[s->triangles[t].v[k]].position;
                for (int d = 0; d < 3; ++d) { tmn[d] = tmn[d] > p[d] ? p[d] : tmn[d]; tmx[d] = tmx[d] < p[d] ? p[d] : tmx[d]; }
            }
            int* lh = &lohi[(size_t)(t - mesh.t_start) * 6];
            for (int k = 0; k < 3; ++k) {    // floor(abs(bbox.min - tri.{min,max}) / width) clamped (Scene.cpp:300-315)
                lh[k] = clampi(f2iX86(std::floor(std::fabs(mesh.bb_min[k] - tmn[k]) / w[k])), 0, gd[k] - 1);
                lh[3 + k] = clampi(f2iX86(std::floor(std::fabs(mesh.bb_min[k] - tmx[k]) / w[k])), 0, gd[k] - 1);
            }
            total += (long long)(lh[3] - lh[0] + 1) * (lh[4] - lh[1] + 1) * (lh[5] - lh[2] + 1);
        }
        widths.push_back(w);
        lohis.push_back(std::move(lohi));
    }
    const long long cells = (long long)grid_model.size() * (long long)ncell;
    if (cells > INT32_MAX) { s->err = "build_grids: " + std::to_string(grid_model.size()) + " grids x " + std::to_string(ncell) + " cells = " + std::to_string(cells) + " cells exceed 2^31 - 1"; return PTAP_E_INVALID; }
    if (total > INT32_MAX) { s->err = "build_grids: " + std::to_string(total) + " references exceed 2^31 - 1"; return PTAP_E_INVALID; }
    s->grid_dim[0] = gx; s->grid_dim[1] = gy; s->grid_dim[2] = gz;
    s->grids.clear(); s->voxels.clear(); s->refs.clear();
    s->voxels.reserve((size_t)cells); s->refs.reserve((size_t)total);
    for (size_t i = 0; i < s->models.size(); ++i) s->models[i].grid_index = grid_of_mesh[s->models[i].mesh_index];
    for (size_t gi = 0; gi < grid_model.size(); ++gi) {
        const PtapMesh& mesh = s->meshes[s->models[grid_model[gi]].mesh_index];
        PtapGrid g{};
        g.entity_type = 0;                  // EntityType::MODEL
        g.entity_index = grid_model[gi];    // the creating model: the traversal reads the bbox through it (Renderer.cpp:245-249)
        for (int k = 0; k < 3; ++k) g.width[k] = widths[gi][k];
        std::vector<int> offs(ncell + 1, 0), cursor;
        const std::vector<int>& lohi = lohis[gi];
        for (int t = mesh.t_start; t < mesh.t_end; ++t) {
            const int* lh = &lohi[(size_t)(t - mesh.t_start) * 6];
            for (int z = lh[2]; z <= lh[5]; ++z)
                for (int y = lh[1]; y <= lh[4]; ++y)
                    for (int x = lh[0]; x <= lh[3]; ++x) offs[(size_t)x + (size_t)y * gx + (size_t)gx * gy * z + 1]++;
        }
        for (size_t c = 0; c < ncell; ++c) offs[c + 1] += offs[c];
        cursor.assign(offs.begin(), offs.end() - 1);
        const int ref_base = (int)s->refs.size();
        s->refs.resize(s->refs.size() + offs[ncell]);
        for (int t = mesh.t_start; t < mesh.t_end; ++t) {     // ascending t inside every cell, as push_back order gives
            const int* lh = &lohi[(size_t)(t - mesh.t_start) * 6];
            for (int z = lh[2]; z <= lh[5]; ++z)
                for (int y = lh[1]; y <= lh[4]; ++y)
                    for (int x = lh[0]; x <= lh[3]; ++x) s->refs[ref_base + cursor[(size_t)x + (size_t)y * gx + (size_t)gx * gy * z]++] = t;
        }
        g.v_start = (int)s->voxels.size();
        for (size_t c = 0; c < ncell; ++c) {
            PtapVoxel vx; vx.start = ref_base + offs[c]; vx.end = ref_base + offs[c + 1]; vx.entity_type = 2;   // EntityType::TRIANGLE
            s->voxels.push_back(vx);
        }
        g.v_end = (int)s->voxels.size();
        s->grids.push_back(g);
    }
    return PTAP_OK;
}

// ---- the scene hard-coded in Scene::Scene (Scene.cpp:3-224): data, not algorithm ---------------------------------

struct BuiltinModel { int mesh; float scale[3]; float rot_deg; float trans[3]; int type; float color[3]; };

const BuiltinModel kBuiltin[] = {
    {2, {0.08f, 0.08f, 0.08f}, 45.0f, {-50.0f, -25.0f, 150.0f}, PTAP_METAL, {0.001f, 0.99f, 0.2f}},       // Scene.cpp:32-42
    {2, {0.1f, 0.1f, 0.1f}, -40.0f, {75.0f, 100.0f, 0.0f}, PTAP_COAT, {0.99f, 0.99f, 0.001f}},            // :44-54
    {2, {0.1f, 0.1f, 0.1f}, 0.0f, {325.0f, 45.0f, 0.0f}, PTAP_REFLECTIVE, {0.99f, 0.99f, 0.75f}},         // :56-66
    {0, {0.1f, 0.1f, 0.1f}, 180.0f, {25.0f, -120.0f, 0.0f}, PTAP_DIFFUSE, {0.99f, 0.99f, 0.99f}},         // :114-124
    {1, {0.1f, 0.1f, 0.1f}, 45.0f, {325.0f, -120.0f, 0.0f}, PTAP_DIFFUSE, {0.99f, 0.50f, 0.60f}},         // :139-149
    {1, {0.1f, 0.1f, 0.1f}, 45.0f, {-225.0f, 8.0f, 0.0f}, PTAP_COAT, {0.40f, 0.10f, 0.99f}},              // :151-161
    {1, {0.1f, 0.1f, 0.1f}, 30.0f, {75.0f, -90.0f, 0.0f}, PTAP_METAL, {0.99f, 0.05f, 0.10f}},             // :163-173
    {1, {0.2f, 0.1f, 0.2f}, 0.0f, {0.0f, 850.0f, -100.0f}, PTAP_EMISSIVE, {0.99f, 0.99f, 0.99f}},         // :175-185
    {1, {0.2f, 0.2f, 0.1f}, 0.0f, {0.0f, 375.0f, 950.0f}, PTAP_EMISSIVE, {0.99f, 0.99f, 0.99f}},          // :187-197
    {1, {0.1f, 0.2f, 0.2f}, 0.0f, {-520.0f, 375.0f, 0.0f}, PTAP_EMISSIVE, {0.99f, 0.99f, 0.99f}},         // :199-209
    {1, {0.1f, 0.2f, 0.2f}, 0.0f, {550.0f, 375.0f, 0.0f}, PTAP_EMISSIVE, {0.99f, 0.99f, 0.99f}},          // :211-221
};

// ---- Config.txt (Config.txt:1-31; never parsed by the reference) --------------------------------------------------

bool parseVec(const std::string& text, float* out, int n)
{
    size_t a = text.find('['), b = text.find(']');
    if (a == std::string::npos || b == std::string::npos || b < a) return false;
    std::string body = text.substr(a + 1, b - a - 1);
    for (char& c : body) if (c == ',') c = ' ';
    std::istringstream is(body);
    for (int i = 0; i < n; ++i) if (!(is >> out[i])) return false;
    return true;
}

std::string trim(const std::string& s)
{
    size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
    return a == std::string::npos ? std::string() : s.substr(a, b - a + 1);
}

int materialType(const std::string& k)
{
    if (k == "DIFFUSE") return PTAP_DIFFUSE;
    if (k == "SPECULAR") return PTAP_SPECULAR;
    if (k == "REFLECTIVE") return PTAP_REFLECTIVE;
    if (k == "REFRACTIVE" || k == "REFRACRIVE") return PTAP_REFRACTIVE;   // the reference's file spells it REFRACRIVE (Config.txt:29)
    if (k == "EMISSIVE") return PTAP_EMISSIVE;
    if (k == "COAT") return PTAP_COAT;
    if (k == "METAL") return PTAP_METAL;
    return -1;
}

void eulerTrs(const float tr[3], const float rot_deg[3], const float sc[3], float m2w[16], float w2m[16])
{
    const float X[3] = {1, 0, 0}, Y[3] = {0, 1, 0}, Z[3] = {0, 0, 1};
    const float k = 0.01745329251994329576923690768489f;
    M4 R = mul(mul(rotateM(rot_deg[2] * k, Z), rotateM(rot_deg[1] * k, Y)), rotateM(rot_deg[0] * k, X));
    M4 M = mul(mul(translateM(tr), R), scaleM(sc));
    M4 I = inverseM(M);
    memcpy(m2w, M.v, sizeof M.v); memcpy(w2m, I.v, sizeof I.v);
}

int addBox(ptap_scene* s, const float mx[3], const float mn[3], int32_t* mesh_index)
{
    // 12 triangles, outward normals, coordinates in OBJ units (scaled by BASE_MODEL_SCALE like an import)
    const int f[6][4] = {{0, 1, 3, 2}, {4, 6, 7, 5}, {0, 4, 5, 1}, {2, 3, 7, 6}, {0, 2, 6, 4}, {1, 5, 7, 3}};
    const float nrm[6][3] = {{-1, 0, 0}, {1, 0, 0}, {0, -1, 0}, {0, 1, 0}, {0, 0, -1}, {0, 0, 1}};
    std::vector<PtapVertex> verts; std::vector<int32_t> idx;
    auto corner = [&](int c, float* p) { p[0] = (c & 4) ? mx[0] : mn[0]; p[1] = (c & 2) ? mx[1] : mn[1]; p[2] = (c & 1) ? mx[2] : mn[2]; };
    for (int face = 0; face < 6; ++face) {
        const int q[6] = {f[face][0], f[face][1], f[face][2], f[face][0], f[face][2], f[face][3]};
        for (int j = 0; j < 6; ++j) {
            PtapVertex pv{}; float p[3]; corner(q[j], p);
            for (int k = 0; k < 3; ++k) { pv.position[k] = p[k] * kBaseModelScale; pv.normal[k] = nrm[face][k] * kBaseModelScale; }
            idx.push_back((int32_t)verts.size()); verts.push_back(pv);
        }
    }
    const int mi = appendMesh(s, verts.data(), (int)verts.size(), idx.data(), 12);
    if (mesh_index) *mesh_index = mi;
    return PTAP_OK;
}

int parseConfig(ptap_scene* s, const std::string& path)
{
    std::ifstream in(path);
    if (!in) { s->err = "cannot open " + path; return PTAP_E_IO; }
    std::string dir = path;
    { size_t k = dir.find_last_of("/\\"); dir = k == std::string::npos ? std::string(".") : dir.substr(0, k); }
    std::vector<std::vector<std::string>> blocks(1);
    std::string line;
    while (std::getline(in, line)) {
        std::string t = trim(line);
        if (t.empty()) { if (!blocks.back().empty()) blocks.emplace_back(); continue; }
        if (t.rfind("//", 0) == 0 || t[0] == '#') continue;
        blocks.back().push_back(t);
    }
    struct Mat { int type; float color[3]; };
    std::map<std::string, Mat> mats;
    struct Obj { int mesh; float tr[3], rot[3], sc[3]; std::string material; };
    std::vector<Obj> objs;
    for (auto& b : blocks) {
        if (b.empty()) continue;
        size_t i = 0;
        while (i < b.size()) {
            const std::string kind = b[i];
            std::string up = kind; for (char& c : up) c = (char)toupper(c);
            const int mt = materialType(up);
            if (mt >= 0) {
                // "DIFFUSE\nname\n[r,g,b]" or a bare keyword (Config.txt:23-30)
                Mat m{mt, {0.99f, 0.99f, 0.99f}};
                std::string name = up;
                if (i + 1 < b.size() && materialType(b[i + 1]) < 0 && b[i + 1].find('[') == std::string::npos) { name = b[i + 1]; ++i; }
                if (i + 1 < b.size() && b[i + 1].find('[') != std::string::npos && b[i + 1].find(':') == std::string::npos) { if (!parseVec(b[i + 1], m.color, 3)) { s->err = path + ": bad colour for material " + name; return PTAP_E_PARSE; } ++i; }
                mats[name] = m; ++i;
                continue;
            }
            if (up == "CAMERA_ORIGIN" || up == "CAMERA_PLANE" || up == "CAMERA_SPAN" || up == "JITTER") {
                if (i + 1 >= b.size()) { s->err = path + ": " + up + " needs a value"; return PTAP_E_PARSE; }
                bool ok = true;
                if (up == "CAMERA_ORIGIN") ok = parseVec(b[i + 1], s->cfg_camera.origin, 3);
                else if (up == "CAMERA_PLANE") ok = parseVec(b[i + 1], s->cfg_camera.plane_min, 3);
                else if (up == "CAMERA_SPAN") ok = parseVec(b[i + 1], s->cfg_camera.span, 2);
                else { s->cfg_camera.jitter = 1; s->cfg_camera.jitter_seed = (uint32_t)strtoul(b[i + 1].c_str(), nullptr, 10); }
                if (!ok) { s->err = path + ": bad " + up; return PTAP_E_PARSE; }
                s->cfg_has_camera = true;
                i += 2; continue;
            }
            if (up == "RESOLUTION" || up == "ITER" || up == "DEPTH" || up == "GRID") {
                if (i + 1 >= b.size()) { s->err = path + ": " + up + " needs a value"; return PTAP_E_PARSE; }
                float v[3] = {0, 0, 0};
                if (up == "RESOLUTION") { if (!parseVec(b[i + 1], v, 2)) { s->err = path + ": bad RESOLUTION"; return PTAP_E_PARSE; } s->cfg_width = (int)v[0]; s->cfg_height = (int)v[1]; }
                else if (up == "GRID") {
                    // each dimension in [1, 2^27] as a float before the conversion ((int) of an out-of-range float is undefined), then the
                    // limits of ptap_scene_build_grids
                    bool ok = parseVec(b[i + 1], v, 3);
                    for (int k = 0; k < 3; ++k) ok = ok && v[k] >= 1.0f && v[k] <= (float)ptap::kMaxGridCells;
                    if (!ok || !ptap::gridDimsOk((int)v[0], (int)v[1], (int)v[2])) { s->err = path + ": bad GRID"; return PTAP_E_PARSE; }
                    for (int k = 0; k < 3; ++k) s->grid_dim[k] = (int)v[k];
                }
                else if (up == "ITER") s->cfg_iter = atoi(b[i + 1].c_str());
                else s->cfg_depth = atoi(b[i + 1].c_str());
                i += 2; continue;
            }
            if (up != "SPHERE" && up != "BOX" && up != "MESH") { s->err = path + ": unknown block '" + kind + "'"; return PTAP_E_PARSE; }
            Obj o{-1, {0, 0, 0}, {0, 0, 0}, {1, 1, 1}, ""};
            size_t j = i + 2;      // b[i+1] = name
            if (i + 1 >= b.size()) { s->err = path + ": " + up + " needs a name"; return PTAP_E_PARSE; }
            if (up == "SPHERE") {
                if (j + 1 >= b.size()) { s->err = path + ": SPHERE needs radius and centre"; return PTAP_E_PARSE; }
                const float radius = (float)atof(b[j].c_str()); float c[3];
                if (!parseVec(b[j + 1], c, 3)) { s->err = path + ": bad SPHERE centre"; return PTAP_E_PARSE; }
                int rc = addIcosphere(s, 4, radius * kBaseModelScale, 0.0f, 0u, &o.mesh); if (rc) return rc;
                // the centre is folded into the vertices so that `translate` stays the model transform
                PtapMesh& mesh = s->meshes[o.mesh];
                const PtapMesh range = mesh;
                mesh = emptyMesh();
                mesh.v_start = range.v_start; mesh.v_end = range.v_end; mesh.t_start = range.t_start; mesh.t_end = range.t_end;
                for (int vi = range.v_start; vi < range.v_end; ++vi) {
                    for (int k = 0; k < 3; ++k) s->vertices[vi].position[k] += c[k] * kBaseModelScale;
                    bbUpdate(mesh, s->vertices[vi].position);
                }
                j += 2;
            } else if (up == "BOX") {
                if (j + 1 >= b.size()) { s->err = path + ": BOX needs max and min"; return PTAP_E_PARSE; }
                float mx[3], mn[3];
                if (!parseVec(b[j], mx, 3) || !parseVec(b[j + 1], mn, 3)) { s->err = path + ": bad BOX corners"; return PTAP_E_PARSE; }
                addBox(s, mx, mn, &o.mesh); j += 2;
            } else {
                if (j >= b.size()) { s->err = path + ": MESH needs a path"; return PTAP_E_PARSE; }
                std::string p = b[j]; for (char& c : p) if (c == '\\') c = '/';
                if (p[0] != '/') p = dir + "/" + p;
                int rc = loadObj(s, p, &o.mesh); if (rc) return rc;
                j += 1;
            }
            for (; j < b.size(); ++j) {
                const std::string& l = b[j];
                const size_t colon = l.find(':');
                if (colon == std::string::npos) break;
                std::string key = trim(l.substr(0, colon)); for (char& c : key) c = (char)tolower(c);
                if (key == "translate") { if (!parseVec(l, o.tr, 3)) { s->err = path + ": bad translate"; return PTAP_E_PARSE; } }
                else if (key == "rotatex" || key == "rotate") { if (!parseVec(l, o.rot, 3)) { s->err = path + ": bad rotate"; return PTAP_E_PARSE; } }
                else if (key == "scale") { if (!parseVec(l, o.sc, 3)) { s->err = path + ": bad scale"; return PTAP_E_PARSE; } }
                else if (key == "material") o.material = trim(l.substr(colon + 1));
                else { s->err = path + ": unknown key '" + key + "'"; return PTAP_E_PARSE; }
            }
            objs.push_back(o);
            i = j;
        }
    }
    for (const Obj& o : objs) {
        PtapModel m{};
        m.mesh_index = o.mesh;
        eulerTrs(o.tr, o.rot, o.sc, m.model_to_world, m.world_to_model);
        Mat mat{PTAP_DIFFUSE, {0.99f, 0.99f, 0.99f}};
        if (!o.material.empty()) {
            auto it = mats.find(o.material);
            if (it == mats.end()) { s->err = path + ": unknown material '" + o.material + "'"; return PTAP_E_PARSE; }
            mat = it->second;
        } else if (mats.size() == 1) mat = mats.begin()->second;
        m.mat.type = mat.type; memcpy(m.mat.color, mat.color, 12);
        s->models.push_back(m);
    }
    if (s->models.empty()) { s->err = path + ": no objects"; return PTAP_E_PARSE; }
    return buildGrids(s, s->grid_dim[0], s->grid_dim[1], s->grid_dim[2]);
}

}  // namespace

extern "C" {

int ptap_scene_create_empty(ptap_scene** out)
{
    if (!out) return PTAP_E_INVALID;
    *out = new ptap_scene();
    return PTAP_OK;
}

void ptap_scene_destroy(ptap_scene* s) { delete s; }
const char* ptap_scene_last_error(const ptap_scene* s) { return s ? s->err.c_str() : "no scene"; }

void ptap_compose_trs(const float translate[3], float rotate_y_degrees, const float scale[3], float model_to_world[16], float world_to_model[16])
{
    // translation_matrix * rotate_matrix * scale_matrix, then glm::inverse (e.g. Scene.cpp:34-39)
    const float Y[3] = {0.0f, 1.0f, 0.0f};
    const float radians = rotate_y_degrees * 0.01745329251994329576923690768489f;      // glm::radians, func_trigonometric.inl:41-46
    const M4 M = mul(mul(translateM(translate), rotateM(radians, Y)), scaleM(scale));
    const M4 I = inverseM(M);
    memcpy(model_to_world, M.v, sizeof M.v);
    memcpy(world_to_model, I.v, sizeof I.v);
}

int ptap_scene_add_obj(ptap_scene* s, const char* path, int32_t* mesh_index)
{
    if (!s || !path) return PTAP_E_INVALID;
    return loadObj(s, path, mesh_index);
}

int ptap_scene_add_mesh(ptap_scene* s, const PtapVertex* vertices, int32_t nvertices, const int32_t* indices, int32_t ntriangles, int32_t* mesh_index)
{
    if (!s || !vertices || !indices || nvertices <= 0 || ntriangles <= 0) return PTAP_E_INVALID;
    for (int i = 0; i < 3 * ntriangles; ++i) if (indices[i] < 0 || indices[i] >= nvertices) { s->err = "add_mesh: index out of range"; return PTAP_E_INVALID; }
    const int mi = appendMesh(s, vertices, nvertices, indices, ntriangles);
    if (mesh_index) *mesh_index = mi;
    return PTAP_OK;
}

int ptap_scene_add_icosphere(ptap_scene* s, int32_t level, float radius, float displacement, uint32_t seed, int32_t* mesh_index)
{
    if (!s) return PTAP_E_INVALID;
    return addIcosphere(s, level, radius, displacement, seed, mesh_index);
}

int ptap_scene_add_model(ptap_scene* s, int32_t mesh_index, const float model_to_world[16], const float* world_to_model, const PtapMaterial* mat, int32_t* model_index)
{
    if (!s || !model_to_world || !mat || mesh_index < 0 || mesh_index >= (int)s->meshes.size()) return PTAP_E_INVALID;
    PtapModel m{};
    m.mesh_index = mesh_index;
    memcpy(m.model_to_world, model_to_world, 64);
    if (world_to_model) memcpy(m.world_to_model, world_to_model, 64);
    else { M4 M; memcpy(M.v, model_to_world, 64); const M4 I = inverseM(M); memcpy(m.world_to_model, I.v, 64); }
    m.mat = *mat;
    s->models.push_back(m);
    if (model_index) *model_index = (int)s->models.size() - 1;
    return PTAP_OK;
}

int ptap_scene_build_grids(ptap_scene* s, int32_t gx, int32_t gy, int32_t gz)
{
    if (!s) return PTAP_E_INVALID;
    if (!ptap::gridDimsOk(gx, gy, gz)) { s->err = "build_grids: bad grid dimensions"; return PTAP_E_INVALID; }
    return buildGrids(s, gx, gy, gz);
}

int ptap_scene_create_builtin(const char* root, ptap_scene** out)
{
    if (!root || !out) return PTAP_E_INVALID;
    ptap_scene* s = new ptap_scene();
    const std::string base = std::string(root) + "/";
    // mesh order of Scene.cpp:6-16; the three Stanford files of Scene.cpp:18-28 are loaded there but never pushed
    const char* files[3] = {"Input data\\enclosing_box.obj", "Input data\\ceiling_light.obj", "Input data\\blender_monkey.obj"};
    for (const char* f : files) {
        int rc = loadObj(s, base + f, nullptr);
        if (rc != PTAP_OK) { fprintf(stderr, "Error loading mesh: %s\n", s->err.c_str()); s->meshes.push_back(emptyMesh()); }   // Scene.cpp:231-235 then push_back
    }
    for (const BuiltinModel& b : kBuiltin) {
        PtapModel m{};
        m.mesh_index = b.mesh;
        ptap_compose_trs(b.trans, b.rot_deg, b.scale, m.model_to_world, m.world_to_model);
        m.mat.type = b.type; memcpy(m.mat.color, b.color, 12);
        s->models.push_back(m);
    }
    if (const int rc = buildGrids(s, 25, 25, 25)) { delete s; return rc; }      // Config.h:8-10, Scene.cpp:223
    *out = s;
    return PTAP_OK;
}

int ptap_scene_create_from_config(const char* config_path, ptap_scene** out)
{
    if (!config_path || !out) return PTAP_E_INVALID;
    ptap_scene* s = new ptap_scene();
    const int rc = parseConfig(s, config_path);
    if (rc != PTAP_OK) { fprintf(stderr, "ptap: %s\n", s->err.c_str()); delete s; *out = nullptr; return rc; }
    *out = s;
    return PTAP_OK;
}

int ptap_scene_create_from_view(const PtapSceneView* v, ptap_scene** out)
{
    if (!v || !out) return PTAP_E_INVALID;
    ptap_scene* s = new ptap_scene();
    s->models.assign(v->models, v->models + v->nmodels);
    s->meshes.assign(v->meshes, v->meshes + v->nmeshes);
    s->vertices.assign(v->vertices, v->vertices + v->nvertices);
    s->triangles.assign(v->triangles, v->triangles + v->ntriangles);
    if (v->grids && v->ngrids > 0) {
        s->grids.assign(v->grids, v->grids + v->ngrids);
        s->voxels.assign(v->voxels, v->voxels + v->nvoxels);
        s->refs.assign(v->refs, v->refs + v->nrefs);
    }
    for (int k = 0; k < 3; ++k) s->grid_dim[k] = v->grid_dim[k] > 0 ? v->grid_dim[k] : 25;
    *out = s;
    return PTAP_OK;
}

int ptap_scene_build_bvh(ptap_scene* s)
{
    if (!s || s->triangles.empty()) return PTAP_E_INVALID;
    std::vector<ptap::TriRec> recs(s->triangles.size());
    ptap::makeTriRecs(s->vertices.data(), s->triangles.data(), (int)s->triangles.size(), recs.data());
    ptap::buildSceneBvh(recs.data(), (int)recs.size(), s->meshes.data(), (int)s->meshes.size(), s->bvh);
    if (!s->st_nodes.fill(s->bvh.nodes.data(), s->bvh.nodes.size() * sizeof(ptap::BvhNode)) ||
        !s->st_tri_id.fill(s->bvh.tri_id.data(), s->bvh.tri_id.size() * sizeof(int)) ||
        !s->st_recs.fill(recs.data(), recs.size() * sizeof(ptap::TriRec))) { s->err = "build_bvh: out of host memory"; return PTAP_E_NOMEM; }
    s->bvh.nodes.clear(); s->bvh.nodes.shrink_to_fit();          // the staging copies are the ones handed out by ptap_scene_view
    s->bvh_nnodes = (int)(s->st_nodes.bytes / sizeof(ptap::BvhNode));
    s->have_bvh = true; s->have_recs = true;
    return PTAP_OK;
}

// The upload-bound triangle records (v0, e1, e2, flat normal: the reference's own arithmetic) without a host BVH: for callers that let the
// GPU build the tree (PTAP_ACCEL_BVH_DEVICE) or walk / emulate the grids, so that ptap_upload_scene is a copy from page-locked memory
// instead of a repack of every triangle on every call.
int ptap_scene_pack_triangles(ptap_scene* s)
{
    if (!s || s->triangles.empty()) return PTAP_E_INVALID;
    if (s->have_recs) return PTAP_OK;
    for (const PtapTriangle& t : s->triangles)
        for (int k = 0; k < 3; ++k)
            if (t.v[k] < 0 || t.v[k] >= (int)s->vertices.size()) { s->err = "pack_triangles: vertex index out of range"; return PTAP_E_INVALID; }
    std::vector<ptap::TriRec> recs(s->triangles.size());
    ptap::makeTriRecs(s->vertices.data(), s->triangles.data(), (int)s->triangles.size(), recs.data());
    if (!s->st_recs.fill(recs.data(), recs.size() * sizeof(ptap::TriRec))) { s->err = "pack_triangles: out of host memory"; return PTAP_E_NOMEM; }
    s->have_recs = true;
    return PTAP_OK;
}

// Structural check of the BVH made by ptap_scene_build_bvh, on the host: every triangle's tolerance band - the set of points the reference's
// predicate can accept, corners at (u, v) = (-e, -e), (1 + 2e, -e), (-e, 1 + 2e), e = 0.0056 > EPSILON - must lie inside EVERY decoded
// (half-precision, outward-rounded) child box on its path from the root; leaf counts, link ranges and the forest property are checked on
// the way.  *violations = 0 for a correct tree.
int ptap_scene_validate_bvh(const ptap_scene* s, int64_t* violations, int32_t* depth)
{
    if (!s || !violations || !s->have_bvh) return PTAP_E_STATE;
    const ptap::BvhNode* nodes = static_cast<const ptap::BvhNode*>(s->st_nodes.p);
    const ptap::TriRec* recs = static_cast<const ptap::TriRec*>(s->st_recs.p);
    const int* tri_id = static_cast<const int*>(s->st_tri_id.p);
    const int nt = (int)s->bvh.tri_id.size();
    auto band = [&](int pos) {
        const ptap::TriRec& r = recs[tri_id[pos]];
        const double e = 0.0056, uv[3][2] = {{-e, -e}, {1 + 2 * e, -e}, {-e, 1 + 2 * e}};
        ptap::ChildBox b;
        for (int k = 0; k < 3; ++k) { b.lo[k] = 3e38f; b.hi[k] = -3e38f; }
        const double v0[3] = {r.v0.x, r.v0.y, r.v0.z}, e1[3] = {r.e1.x, r.e1.y, r.e1.z}, e2[3] = {r.e2.x, r.e2.y, r.e2.z};
        for (auto& c : uv)
            for (int k = 0; k < 3; ++k) {
                const double x = v0[k] + c[0] * e1[k] + c[1] * e2[k];
                b.lo[k] = std::min(b.lo[k], (float)x); b.hi[k] = std::max(b.hi[k], (float)x);
            }
        return b;
    };
    long long bad = 0;
    int maxd = 0;
    std::vector<char> covered(nt, 0);
    for (size_t m = 0; m < s->bvh.mesh_root.size(); ++m) {
        if (s->bvh.mesh_root[m] < 0) continue;
        int d = 0;
        bad += ptap::validateBvh(nodes, s->bvh_nnodes, s->bvh.mesh_root[m], nt, [&](int pos) { covered[pos]++; return band(pos); }, &d);
        maxd = std::max(maxd, d);
    }
    for (int k = 0; k < nt; ++k) if (covered[k] != 1) ++bad;          // every leaf-order position belongs to exactly one leaf
    *violations = bad;
    if (depth) *depth = maxd;
    return PTAP_OK;
}

int ptap_scene_view(const ptap_scene* s, PtapSceneView* out)
{
    if (!s || !out) return PTAP_E_INVALID;
    static_assert(sizeof(PtapBvhNode) == sizeof(ptap::BvhNode), "public and device BVH node layouts must agree");
    out->bvh_nodes = nullptr; out->n_bvh_nodes = 0; out->bvh_tri_id = nullptr; out->n_bvh_tris = 0; out->bvh_mesh_root = nullptr; out->n_bvh_roots = 0;
    out->bvh_depth = 0; out->tri_recs = nullptr; out->n_tri_recs = 0;
    if (s->have_bvh) {
        out->bvh_nodes = static_cast<const PtapBvhNode*>(s->st_nodes.p); out->n_bvh_nodes = s->bvh_nnodes;
        out->bvh_tri_id = static_cast<const int32_t*>(s->st_tri_id.p); out->n_bvh_tris = (int)s->bvh.tri_id.size();
        out->bvh_mesh_root = s->bvh.mesh_root.data(); out->n_bvh_roots = (int)s->bvh.mesh_root.size();
        out->bvh_depth = s->bvh.max_depth + 1;
    }
    if (s->have_recs) { out->tri_recs = s->st_recs.p; out->n_tri_recs = (int)(s->st_recs.bytes / sizeof(ptap::TriRec)); }
    out->models = s->models.data(); out->nmodels = (int)s->models.size();
    out->meshes = s->meshes.data(); out->nmeshes = (int)s->meshes.size();
    out->vertices = s->vertices.data(); out->nvertices = (int)s->vertices.size();
    out->triangles = s->triangles.data(); out->ntriangles = (int)s->triangles.size();
    out->grids = s->grids.empty() ? nullptr : s->grids.data(); out->ngrids = (int)s->grids.size();
    out->voxels = s->voxels.empty() ? nullptr : s->voxels.data(); out->nvoxels = (int)s->voxels.size();
    out->refs = s->refs.empty() ? nullptr : s->refs.data(); out->nrefs = (int)s->refs.size();
    for (int k = 0; k < 3; ++k) out->grid_dim[k] = s->grid_dim[k];
    return PTAP_OK;
}

PtapModel* ptap_scene_models(ptap_scene* s) { return s ? s->models.data() : nullptr; }

int ptap_scene_config_camera(const ptap_scene* s, PtapCamera* out)
{
    if (!s || !out) return 0;
    *out = s->cfg_camera;
    return s->cfg_has_camera ? 1 : 0;
}

int ptap_scene_config_params(const ptap_scene* s, int32_t out4[4])
{
    if (!s || !out4) return PTAP_E_INVALID;
    out4[0] = s->cfg_width; out4[1] = s->cfg_height; out4[2] = s->cfg_iter; out4[3] = s->cfg_depth;
    return PTAP_OK;
}

}  // extern "C"
