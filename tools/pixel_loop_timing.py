"""K2 time of the Render-API modes that run the shared renderNext pixel loop and that bench.py does not time: ragged slices of the
default scene (k_trace_small_any, 1 and 2x2 samples, 1920x1080, depth 20) and 2x2 SSAA of the config-4 scene (k_trace_blob<MULTI>,
3840x2160, depth 8).  One JSON line; RFX_LIB picks the library (A/B against another build)."""
import json
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from reflaxman_b200 import capi, scenes as S


def k2_ms(c, cam, refl, samples, chunk, reps=5):
    c.render(cam, refl, samples, False, chunk); c.synchronize()   # warm-up: modules, tile order, grids
    c.enable_profiling(True); c.stats_reset()
    for _ in range(reps):
        c.render(cam, refl, samples, False, chunk)
    c.synchronize()
    st = c.stats(); c.enable_profiling(False)
    return {"k2_ms_per_frame": st["trace_kernel_ms"] / reps, "trace_kernels": st["trace_kernels"],
            **{k: st[k] for k in ("launches_small_fast", "launches_small_any", "launches_blob_fast", "launches_blob_any")}}


res = {}
cam = S.default_camera()
c = capi.Context(0)
c.load_scene(S.default_scene()); c.set_seeds(12345, 12345); c.set_image_size(1920, 1080)
for samples in (1, 2):
    # slices of 1920 * 1080 / 7 + 3 pixels start and end inside rows: every launch takes the general kernel
    res["small_any_ragged_samples_%d" % samples] = k2_ms(c, cam, 20, samples, 1920 * 1080 // 7 + 3)
c.close()
c = capi.Context(0)
c.load_scene(S.synthetic_scene(32, floor=S.synthetic_texture(1024, 1024, 11), skybox=S.synthetic_texture(2048, 1536, 7)))
c.set_seeds(12345, 12345); c.set_image_size(3840, 2160)
res["blob_multi_ssaa2_depth8"] = k2_ms(c, cam, 8, 2, None)
c.close()
print(json.dumps(res))
