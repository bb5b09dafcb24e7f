"""Ray sets for the occlusion queries, shared by tests/test_gpu_occlusion.py and tools/occlusion_probe.py."""
import numpy as np


def shadow_rays(yart, ctx, preset, width, height, spp=1, seed=5, t_shorten=1e-6):
    """Shadow rays of a preset: from the hit points of its camera rays (yart_closest_hit on the GPU) toward the nearest
    surface point q of each spherical light, as the unnormalised direction q - p; a query with t_max = 1 - t_shorten
    stops just short of the light.  Returns (rays, t_max)."""
    cam = preset.camera(width, height)
    rays, _, _ = ctx.camera_rays(cam, width, height, 0, spp, seed)
    hits, _ = ctx.closest_hit(rays, yart.TARGET_WORLD, 0.001, float("inf"), yart.ORDER_NEAR)
    hit = hits["prim_id"] != yart.MISS
    p = rays["origin"][hit] + hits["t"][hit, None] * rays["direction"][hit]
    sd = preset.desc.contents
    lights = [sd.lights[i] for i in range(sd.n_lights) if sd.lights[i].kind == yart.abi.OBJ_SPHERE]
    assert lights, "the preset has no spherical light"
    o, d = [], []
    for lt in lights:
        c, r = np.array(lt.p[0:3], dtype=np.float64), float(lt.p[3])
        v = p - c
        q = c + r * v / np.linalg.norm(v, axis=1, keepdims=True)
        o.append(p)
        d.append(q - p)
    return yart.make_rays(np.concatenate(o), np.concatenate(d)), 1.0 - t_shorten
