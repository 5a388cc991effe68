import os, sys
TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(TESTS)); sys.path.insert(0, TESTS)
import numpy as np
from yuki_b200 import api, desc as D, scenes, transforms as xf
from oracle import oracle as O
from test_sphere import sphere_scene, sphere_field
ctx = api.Context(0)
for name,(scene,cam) in (("cornell+sphere", sphere_scene(xf)), ("field", sphere_field(xf,40))):
    for integ in (D.IntegratorType.path(6), D.IntegratorType.whitted(3)):
        film = D.FilmSettings((128,96),16); smp = D.SamplerType.stratified(3,3)
        dev = api.Scene(ctx, scene)
        r = api.Renderer(ctx).render(dev, cam, film, smp, integ)
        o,_,st = O.OracleScene(scene).render(cam, film, smp, integ)
        d = np.abs(r.film - o)
        rr = np.sqrt(np.mean((r.film-o)**2))/np.mean(o)
        print(name, integ.kind, "rmse", rr, "max", d.max(), "frac>1e-4", np.mean(d.max(axis=2) > 1e-4*(1+o.max(axis=2))), "frac>1e-6", np.mean(d.max(axis=2) > 1e-6*(1+o.max(axis=2))), "rays", r.stats.ray_count, st.ray_count)
