// TEST INFRASTRUCTURE ONLY: Scene::intersect's Hit { t, si, shape } for ray batches on the CPU oracle, the reference
// tests/test_query_surface.py compares yk_query_intersect's surface fields with. The test compiles this file with the oracle's
// flags (oracle/Makefile) into a library of its own: it includes the oracle's C entry points, so its scenes are built by the
// very code liboracle.so runs, and adds one entry point next to them.
#include "yk_oracle.cpp"

extern "C" {

// t (inf on a miss), original shape id and material of the hit shape (-1 on a miss), and the SurfaceInteraction's area_light
// (-1), p, n, uv, shading.n and shading.dpdu (0 on a miss). Every output may be NULL.
void yko_intersect_surface(const yko_scene* sc, const float* o, const float* d, const float* tmax, uint32_t n, float* t_out,
                           int32_t* id_out, int32_t* mat_out, int32_t* al_out, float* p_out, float* n_out, float* uv_out,
                           float* shn_out, float* shdpdu_out) {
    const Scene& s = sc->s;
    auto st3 = [](float* dst, uint32_t i, V3 v) { if (dst) { dst[3 * i] = v.x; dst[3 * i + 1] = v.y; dst[3 * i + 2] = v.z; } };
    for (uint32_t i = 0; i < n; ++i) {
        Ray ray{ld3(o + 3 * i), ld3(d + 3 * i), tmax ? tmax[i] : INFINITY};
        IntersectionResult r = s.intersect(ray, nullptr);
        SurfaceInteraction si{};
        if (r.has_hit) si = r.hit.si;
        else si.area_light = -1;
        const Triangle* shape = r.has_hit ? &s.shapes[r.hit.shape] : nullptr;
        if (t_out) t_out[i] = r.has_hit ? r.hit.t : INFINITY;
        if (id_out) id_out[i] = shape ? (int32_t)shape->orig_id : -1;
        if (mat_out) mat_out[i] = shape ? shape->material : -1;
        if (al_out) al_out[i] = si.area_light;
        st3(p_out, i, si.p);
        st3(n_out, i, si.n);
        if (uv_out) { uv_out[2 * i] = si.uv.x; uv_out[2 * i + 1] = si.uv.y; }
        st3(shn_out, i, si.sh_n);
        st3(shdpdu_out, i, si.sh_dpdu);
    }
}

}  // extern "C"
