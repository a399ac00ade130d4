// Fragment export of the CPU oracle's tri renderer, for the fp64 camera-gradient reference
// (tests/test_gpu_tri_camera_grads.py).  Compiled together with oracle/oracle.cpp, whose tri_render it walks again:
// per pixel, in compositing order, the faces that pass in_tri and shade().ok, up to n_contrib, each with its
// clamp_bary region code.  Test infrastructure only.
#include "../oracle/oracle.cpp"

extern "C" {

// counts[B*H*W] is always written; face / code (may be null) receive the concatenation in pixel order, at most `cap`
// entries.  Returns the total count.
size_t oracle_tri_fragments(void* h, uint32_t* counts, int32_t* face, int32_t* code, size_t cap)
{
    const Tri& t = *static_cast<Tri*>(h);
    const Common& c = t.c;
    const size_t HW = (size_t)c.W * c.H, BI = (size_t)c.B * HW;
    std::vector<std::vector<int32_t>> frag(BI);
#pragma omp parallel for schedule(dynamic, 64)
    for (long long bp = 0; bp < (long long)BI; bp++) {
        int b = (int)(bp / HW), pix = (int)(bp % HW), y = pix / c.W, x = pix % c.W;
        int tile = (b * c.gy + y / TILE) * c.gx + x / TILE;
        uint32_t r0 = c.ranges[2 * (size_t)tile], last = t.n_contrib[bp];
        V3 ro, rd;
        pixel_ray(&t.imv[16 * b], &t.ipj[16 * b], x + 0.5f, y + 0.5f, c.W, c.H, false, ro, rd);
        for (uint32_t k = 0; k < last; k++) {
            int f = (int)c.vals_sorted[r0 + k];
            const int* fv = &t.faces[3 * f];
            const float* im = &c.verts_image[0];
            size_t o = (size_t)b * c.P;
            if (!in_tri(x + 0.5f, y + 0.5f, im + 2 * (o + fv[0]), im + 2 * (o + fv[1]), im + 2 * (o + fv[2]))) continue;
            Hit hh = shade(t, b, f, ro, rd);
            if (!hh.ok) continue;
            frag[bp].push_back(f);
            frag[bp].push_back(hh.code);
        }
    }
    size_t n = 0;
    for (size_t bp = 0; bp < BI; bp++) {
        if (counts) counts[bp] = (uint32_t)(frag[bp].size() / 2);
        for (size_t k = 0; k < frag[bp].size(); k += 2, n++) {
            if (n < cap && face) face[n] = frag[bp][k];
            if (n < cap && code) code[n] = frag[bp][k + 1];
        }
    }
    return n;
}

}  // extern "C"
