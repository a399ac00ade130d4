// Fragment export of the CPU oracle's tet renderer, for the fp64 camera-gradient reference
// (tests/test_gpu_tet_camera_grads.py).  Compiled together with oracle/oracle.cpp: the march of its tet_render is walked
// again with per-pixel ray coordinates given by the caller (pixel centres, or the GPU's jittered coordinates), and the
// reverse march of its tet_backward after it.  Per pixel, in compositing order, the faces the forward composites, each
// with a flag: does the backward walk reach this step?  Test infrastructure only.
#include "../oracle/oracle.cpp"

namespace {

struct PixelMarch {
    std::vector<int32_t> faces;
    int ff = -1, lf = -1;
    bool active = false;
    uint32_t walked = 0;     // steps the reverse march reaches, counted from the last
    bool mismatch = false;   // the reverse march left the forward's faces
    float color[3] = { 0, 0, 0 }, depth = 1.0f;
};

// tet_render's per-pixel body (oracle.cpp) with the ray through (fx, fy)
PixelMarch march_pixel(const Tet& t, int b, int x, int y, float fx, float fy)
{
    const Common& c = t.c;
    PixelMarch r;
    const int tile = (b * c.gy + y / TILE) * c.gx + x / TILE;
    const uint32_t r0 = c.ranges[2 * (size_t)tile], r1 = c.ranges[2 * (size_t)tile + 1];
    V3 ro, rd;
    pixel_ray(&t.imv[16 * b], &t.ipj[16 * b], fx, fy, c.W, c.H, true, ro, rd);
    float min_T = -1.0f, min_T_maxd = -1.0f;
    int ff = -1, ft = -1;
    for (uint32_t i = r0; i < r1; i++) {
        int f = (int)c.vals_sorted[i];
        size_t bf = (size_t)b * c.F + f;
        if (min_T >= 0.0f && c.min_depth[bf] > min_T_maxd) break;
        float tuv[3];
        if (!ray_tri(ro, rd, vert(t.verts, t.faces[3 * f]), vert(t.verts, t.faces[3 * f + 1]), vert(t.verts, t.faces[3 * f + 2]), tuv, true)) continue;
        if (min_T < 0.0f || tuv[0] < min_T) { min_T = tuv[0]; min_T_maxd = c.max_depth[bf]; ff = f; }
    }
    if (ff >= 0)
        for (int i = 0; i < 2; i++) {
            int tet = t.face_tets[2 * ff + i];
            if (tet < 0) continue;
            if (dot(outward_normal(t, ff, tet), rd) < 0.0f) ft = tet;
        }
    r.ff = ff;
    bool done = false, active = false;
    float rt = 0, iu = 0, iv = 0;
    if (ff == -1 || ft == -1) done = true;
    else {
        float tuv[3] = { 0, 0, 0 };
        ray_tri(ro, rd, vert(t.verts, t.faces[3 * ff]), vert(t.verts, t.faces[3 * ff + 1]), vert(t.verts, t.faces[3 * ff + 2]), tuv, true);
        rt = tuv[0]; iu = tuv[1]; iv = tuv[2];
    }
    V3 C = { 0, 0, 0 };
    float D = 0, log_T = 0;
    int lf = -1, lt = -1, cf = ff, ct = ft;
    while (!done) {
        r.faces.push_back(cf);
        V3 c0 = vert(t.vcolor, t.faces[3 * cf]), c1 = vert(t.vcolor, t.faces[3 * cf + 1]), c2 = vert(t.vcolor, t.faces[3 * cf + 2]);
        V3 col = madd(madd(c0, c1 - c0, iu), c2 - c0, iv);
        float op = t.fopacity[cf], in = t.fintense[(size_t)b * c.F + cf];
        col = col * in;
        float tmpT = std::exp(log_T);
        C = madd(C, col, tmpT * op);
        D = fmaf(tmpT * op, point_depth(t, b, ro, rd, rt), D);
        if (op < 1.0f) log_T += std::log(1.0f - op); else log_T = std::log(T_EPS * 0.1f);
        if (std::exp(log_T) < T_EPS) { done = true; active = true; }
        lf = cf; lt = ct;
        if (ct == -1) { active = true; done = true; }
        if (!done) {
            int nf, nt; float tuv[3] = { 0, 0, 0 };
            if (!tet_step(t, ct, cf, ro, rd, true, nf, nt, tuv)) done = true;
            cf = nf; ct = nt; rt = tuv[0]; iu = tuv[1]; iv = tuv[2];
        }
    }
    r.lf = lf;
    r.active = active;
    if (active) {
        float fT = std::exp(log_T);
        r.color[0] = fmaf(fT, t.bg[0], C.x); r.color[1] = fmaf(fT, t.bg[1], C.y); r.color[2] = fmaf(fT, t.bg[2], C.z);
        r.depth = fmaf(fT, 1.0f, D);
    } else {
        for (int ch = 0; ch < 3; ch++) r.color[ch] = t.bg[ch];
    }
    // tet_backward's walk (oracle.cpp): from the last face back towards the first, until the reverse march gives up
    if (!active || lf == -1) return r;
    cf = lf; ct = lt;
    for (int i = 0; i < 2; i++) { int cand = t.face_tets[2 * cf + i]; if (cand == ct) continue; ct = cand; break; }
    const size_t n = r.faces.size();
    while (true) {
        if (r.walked >= n || r.faces[n - 1 - r.walked] != cf) { r.mismatch = true; break; }
        r.walked++;
        if (cf == ff) break;
        if (ct == -1) break;
        int nf, nt; float tv[3] = { 0, 0, 0 };
        if (!tet_step(t, ct, cf, ro, rd, false, nf, nt, tv)) break;
        cf = nf; ct = nt;
    }
    return r;
}

}  // namespace

extern "C" {

// coords[2 * bp] (x, y) pixel coordinates of pixel bp = (b * H + y) * W + x, or null for the pixel centres.
// counts[B*H*W], first_face, last_face, active (0/1), color[B,3,H,W], depth[B,H,W] are always written; face / reach (may
// be null) receive the concatenation in pixel order, at most `cap` entries.  Returns the total count; *mismatch = number
// of pixels whose reverse march left the forward's faces.
size_t oracle_tet_fragments(void* h, const float* coords, uint32_t* counts, int32_t* first_face, int32_t* last_face,
                            uint8_t* active, float* color, float* depth, int32_t* face, uint8_t* reach, size_t cap,
                            uint32_t* mismatch)
{
    const Tet& t = *static_cast<Tet*>(h);
    const Common& c = t.c;
    const size_t HW = (size_t)c.W * c.H, BI = (size_t)c.B * HW;
    std::vector<PixelMarch> px(BI);
#pragma omp parallel for schedule(dynamic, 64)
    for (long long bp = 0; bp < (long long)BI; bp++) {
        const int b = (int)(bp / HW), pix = (int)(bp % HW), y = pix / c.W, x = pix % c.W;
        const float fx = coords ? coords[2 * bp] : x + 0.5f, fy = coords ? coords[2 * bp + 1] : y + 0.5f;
        px[bp] = march_pixel(t, b, x, y, fx, fy);
    }
    size_t n = 0;
    uint32_t bad = 0;
    for (size_t bp = 0; bp < BI; bp++) {
        const PixelMarch& r = px[bp];
        const size_t b = bp / HW, pix = bp % HW, m = r.faces.size();
        counts[bp] = (uint32_t)m;
        first_face[bp] = r.ff; last_face[bp] = r.lf; active[bp] = r.active ? 1 : 0;
        for (int ch = 0; ch < 3; ch++) color[(b * 3 + ch) * HW + pix] = r.color[ch];
        depth[bp] = r.depth;
        bad += r.mismatch ? 1u : 0u;
        for (size_t k = 0; k < m; k++, n++) {
            if (n < cap && face) face[n] = r.faces[k];
            if (n < cap && reach) reach[n] = (r.active && k + r.walked >= m) ? 1 : 0;
        }
    }
    if (mismatch) *mismatch = bad;
    return n;
}

// last_face[B*H*W] of the oracle's own tet_render
void oracle_tet_last_face(void* h, int32_t* last_face)
{
    const Tet& t = *static_cast<Tet*>(h);
    std::copy(t.last_face.begin(), t.last_face.end(), last_face);
}

}  // extern "C"
