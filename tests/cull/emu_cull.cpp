// emu_cull.cpp -- TEST HELPER: the host build of tests/emu (scene upload, traversal steps) plus diagnostics of the exact
// culling that use the production leaf test itself (leaf_margin / leaf_box_culled, csrc/sqt_core.cuh), for
// tests/test_cull_margin.py.  Not linked or loaded by the product library.
#include "../emu/emu.cpp"

extern "C" {

// The leaf culling on one-triangle leaves, pair i = (triangle record i, ray i), tri = 12 floats per record (the device layout:
// v0.xyz e1.x | e1.yz e2.xy | e2.z - - -).  accept[i] = moller_trumbore accepts, t[i] = its t; margin[i] = leaf_margin of the leaf
// holding only that triangle, culled[i] = leaf_box_culled rejects that leaf.
void cull_pairs(const float *tri, const float *org, const float *dir, long long n, int *accept, float *t, float *margin, int *culled) {
    for (long long i = 0; i < n; ++i) {
        const float *q = tri + 12 * i;
        const float4 a[3] = {mk4(q[0], q[1], q[2], q[3]), mk4(q[4], q[5], q[6], q[7]), mk4(q[8], q[9], q[10], q[11])};
        const Ray r{org[3 * i], org[3 * i + 1], org[3 * i + 2], dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]};
        float tt = 0.0f, dist; int stage;
        accept[i] = moller_trumbore(a[0], a[1], a[2], r, tt, dist, stage) ? 1 : 0;
        t[i] = tt;
        float4 b0, b1;
        make_leaf_record(a, 0, 1, b0, b1);
        margin[i] = leaf_margin(b0, b1, r);
        culled[i] = leaf_box_culled(b0, b1, r, XRCP(r.dx), XRCP(r.dy), XRCP(r.dz)) ? 1 : 0;
    }
}

// With the culling off (every leaf the reference visits is entered), the production leaf test applied to the leaf's record and
// to consecutive groups of `group` triangles of it (each with its own record, a finer culling level).
// out = { leaf visits, triangle tests, visits the leaf test rejects, triangle tests in those, visits with an accepted triangle,
//         of those rejected by the leaf test (must be 0), groups, groups rejected, groups with an accepted triangle rejected (must be 0) }
void cull_leaf_stats(emu_scene *s, const float *org, const float *dir, long long n, int group, unsigned long long *out) {
    for (int k = 0; k < 9; ++k) out[k] = 0;
    const uint32_t saved_cull = s->view.leaf_cull;
    s->view.leaf_cull = 0;
    Counters cn = {};
    float4 stack[kStackEntries];
    for (long long i = 0; i < n; ++i) {
        TravLane L; L.stack = stack;
        const LaneRay ra(L);
        L.r = Ray{org[3 * i], org[3 * i + 1], org[3 * i + 2], dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]};
        start_ray<false>(s->view, L, &cn);
        while (L.state != ST_DONE) {
            if (L.state == ST_RET) ret_step(s->view, L, ra);
            if (L.state == ST_DESC) desc_step<false>(s->view, L, ra, &cn);
            if (L.state == ST_SPH) sphere_step(s->view, L, ra);
            if (L.state == ST_ENTER) enter_step<false>(s->view, L, ra, &cn);
            if (L.state == ST_LEAF) {
                const uint32_t first = L.child, count = (uint32_t)L.i + 1;
                const bool safe = !(L.rf & kRfUnsafe);
                float4 b0, b1;
                make_leaf_record(s->tris.data(), first, count, b0, b1);
                const bool leaf_cut = safe && leaf_box_culled(b0, b1, L.r, L.dfx, L.dfy, L.dfz);
                for (uint32_t g0 = 0; g0 < count; g0 += (uint32_t)group) {
                    const uint32_t gc = std::min<uint32_t>((uint32_t)group, count - g0);
                    make_leaf_record(s->tris.data(), first + g0, gc, b0, b1);
                    const bool cut = safe && leaf_box_culled(b0, b1, L.r, L.dfx, L.dfy, L.dfz);
                    bool acc = false;
                    for (uint32_t t = 0; t < gc; ++t) {
                        const TriData d = tri_load(s->view, first + g0 + t);
                        float tt, dd; int st;
                        acc = moller_trumbore(d.a0, d.a1, d.a2, L.r, tt, dd, st) || acc;
                    }
                    out[6] += 1; out[7] += cut; out[8] += cut && acc;
                }
                while (L.state == ST_LEAF) tri_step<false>(s->view, L, &cn);
                out[0] += 1; out[1] += count;
                if (leaf_cut) { out[2] += 1; out[3] += count; }
                if (L.cur.tri >= 0) { out[4] += 1; if (leaf_cut) out[5] += 1; }
            }
        }
    }
    s->view.leaf_cull = saved_cull;
}

}  // extern "C"
