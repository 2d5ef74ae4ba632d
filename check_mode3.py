import hashlib, os, sys, ctypes as C, numpy as np
sys.path.insert(0, "software-raytracing_b200"); sys.path.insert(0, ".")
import pyraylib as rl
p = rl.Product(); p.lib.Raylib_Initialize()
for cfg, size in ((5, 40), (6, 0), (2, 0)):
    d = np.load("tests/golden/recorded/test_gpu_parity.test_microsurface_normal_and_reflectance_views_vs_compiled_reference_%d-%d.npz" % (cfg, size))
    info = p.create_demo(cfg, size); p.set_viewport(info, 240, 136)
    m3 = p.render(info.settings.copy(renderMode=3), info.scene, info.camera)
    a, n = p.lib.Raylib_CreateImage(240, 136), p.lib.Raylib_CreateImage(240, 136)
    assert p.lib.RaylibB200_RenderAux(C.byref(info.settings), info.scene, info.camera, a, n)
    aux = p.dump_image(n, 240, 136)
    h = lambda x: hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()
    print("config%d: stored mode3 == mode-3 render: %s, == aux normal: %s, render == aux: %s" % (cfg, h(m3) == str(d["mode3/sha256"]), h(aux) == str(d["mode3/sha256"]), h(m3) == h(aux)))
    p.destroy_demo(info)
