"""Generates tests/golden/ref_kernels_golden.npz: what the REFERENCE'S OWN CUDA kernels (oracle/_ref/libmf_ref.so, built by
`make -C oracle -f Makefile.ref` from the reference sources) return on the inputs tests/test_gpu_ref.py builds from the CPU oracle.
Needs a CUDA device.  Images are kept at the test's fixed pixel samples, NaN patterns and binary masks in full; the full-image
statistics the test's tolerances were set on are printed.
Run:  python tests/golden/make_ref_kernels_golden.py [output.npz]"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import oracle_lib as ol                                                          # noqa: E402
from tests.test_gpu_ref import (H, KEEP_IMAGE, KEEP_MAP, W, DataTerm, SOBEL_SCALE, icp_pose, intensity, model_map_textures,  # noqa: E402
                                oracle_state, rgb_level_inputs, shrink, so3_inputs, u8_source)

f32p = C.POINTER(C.c_float)
ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libmf_ref.so"))
sc, orc, pose_before = oracle_state()
fa, od = orc.frame_arrays(), orc.odom(0)
out = {}


def planar(key, a):
    out[key] = shrink(a, KEEP_MAP)
    out[key + "_nan"] = np.packbits(np.isnan(a[0]))


def stat(what, a, b):
    ok = ~np.isnan(b)
    print(f"{what}: max |ref - oracle| {float(np.abs(a[ok] - b[ok]).max()):.3e}, differing {float((a != b)[ok].mean()):.2e}")


# vertex / normal maps of the frame pyramid
for l in range(3):
    w, h = W >> l, H >> l
    v = np.zeros((3, h, w), np.float32); n = np.zeros((3, h, w), np.float32)
    assert ref.ref_vmap_nmap(ol.ptr(np.ascontiguousarray(fa[f"depth{l}"])), w, h, C.c_float(528 / (1 << l)), C.c_float(528 / (1 << l)),
                             C.c_float(320 / (1 << l)), C.c_float(240 / (1 << l)), C.c_float(4.0), ol.ptr(v), ol.ptr(n)) == 0
    planar(f"vmap{l}", v); planar(f"nmap{l}", n)
    stat(f"vmap{l}", v, fa[f"vmap{l}"]); stat(f"nmap{l}", n, fa[f"nmap{l}"])
# depth and 8-bit pyramids
for l in range(2):
    w, h = W >> l, H >> l
    d = np.zeros((h // 2, w // 2), np.float32)
    assert ref.ref_pyrdown_f(ol.ptr(np.ascontiguousarray(fa[f"depth{l}"])), w, h, ol.ptr(d)) == 0
    out[f"pyrdown{l}"] = shrink(d, KEEP_MAP)
    stat(f"pyrdown{l}", d, fa[f"depth{l+1}"])
o1 = np.zeros((H // 2, W // 2), np.uint8); o2 = np.zeros_like(o1)
src = u8_source()
assert ref.ref_pyrdown_u8(ol.ptr(src), W, H, ol.ptr(o1)) == 0
out["pyrdown_u8"] = shrink(o1, KEEP_IMAGE)
orc.L.orc_pyrdown_gauss_u8(ol.ptr(src), W, H, ol.ptr(o2))
stat("pyrdown_u8", o1.astype(float), o2.astype(float))
# model maps at the pose before tracking
vt, nt = model_map_textures(orc)
vs = [np.zeros((3, H >> l, W >> l), np.float32) for l in range(3)]
ns = [np.zeros((3, H >> l, W >> l), np.float32) for l in range(3)]
Rpi, Rc, tc = icp_pose(pose_before)
assert ref.ref_model_maps(ol.ptr(vt), ol.ptr(nt), W, H, ol.ptr(Rc), ol.ptr(tc), (f32p * 3)(*[a.ctypes.data_as(f32p) for a in vs]),
                          (f32p * 3)(*[a.ctypes.data_as(f32p) for a in ns])) == 0
for l in range(3):
    planar(f"model_vmap{l}", vs[l]); planar(f"model_nmap{l}", ns[l])
    stat(f"model_vmap{l}", vs[l], ol.arr(od.vmap_g[l], (3, H >> l, W >> l), np.float32))
# icpStep with the reference's fallback launch config 128x112
for l in range(3):
    w, h = W >> l, H >> l
    A = np.zeros(36, np.float32); b = np.zeros(6, np.float32); res = np.zeros(2, np.float32)
    vg = np.ascontiguousarray(ol.arr(od.vmap_g[l], (3, h, w), np.float32)); ng = np.ascontiguousarray(ol.arr(od.nmap_g[l], (3, h, w), np.float32))
    assert ref.ref_icp_step(ol.ptr(Rc), ol.ptr(tc), ol.ptr(fa[f"vmap{l}"]), ol.ptr(fa[f"nmap{l}"]), ol.ptr(Rpi), ol.ptr(tc),
                            C.c_float(528 / (1 << l)), C.c_float(528 / (1 << l)), C.c_float(320 / (1 << l)), C.c_float(240 / (1 << l)),
                            ol.ptr(vg), ol.ptr(ng), C.c_float(0.1), C.c_float(np.float32(np.sin(20.0 * 3.14159254 / 180.0))), w, h, 128, 112,
                            ol.ptr(A), ol.ptr(b), ol.ptr(res)) == 0
    out[f"icp{l}_A"], out[f"icp{l}_b"], out[f"icp{l}_res"] = A, b, res
# Sobel on frame 3, one SO3 step on level-2 intensities of frames 3 and 4
inten = intensity(orc, sc.render(3)[0])
dx = np.zeros((H, W), np.int16); dy = np.zeros((H, W), np.int16); dxo = np.zeros_like(dx); dyo = np.zeros_like(dy)
assert ref.ref_sobel(ol.ptr(inten), W, H, ol.ptr(dx), ol.ptr(dy)) == 0
out["sobel_dx"], out["sobel_dy"] = shrink(dx, KEEP_IMAGE), shrink(dy, KEEP_IMAGE)
orc.L.orc_sobel(ol.ptr(inten), W, H, ol.ptr(dxo), ol.ptr(dyo))
stat("sobel_dx", dx.astype(float), dxo.astype(float)); stat("sobel_dy", dy.astype(float), dyo.astype(float))
a, b2, basis, kinv, krlr = so3_inputs(sc, orc)
A = np.zeros(9, np.float32); bb = np.zeros(3, np.float32); res = np.zeros(2, np.float32)
assert ref.ref_so3_step(ol.ptr(a), ol.ptr(b2), ol.ptr(basis), ol.ptr(kinv), ol.ptr(krlr), W // 4, H // 4, 160, 64, ol.ptr(A), ol.ptr(bb), ol.ptr(res)) == 0
out["so3_A"], out["so3_b"], out["so3_res"] = A, bb, res
# geometric edges, threshold, invert
e = np.zeros((H, W), np.float32); inv = np.zeros((H, W), np.uint8)
assert ref.ref_geometric_edges(ol.ptr(fa["vmap0"]), ol.ptr(fa["nmap0"]), W, H, C.c_float(150.0), C.c_float(2.8), C.c_float(0.3), ol.ptr(e), ol.ptr(inv)) == 0
assert set(np.unique(inv).tolist()) <= {0, 255}
out["edges"], out["edges_inv"] = shrink(e, KEEP_IMAGE), np.packbits(inv == 255)
eo = np.zeros((H, W), np.float32)
orc.L.orc_geometric_edges(ol.ptr(fa["vmap0"]), ol.ptr(fa["nmap0"]), W, H, C.c_float(150.0), C.c_float(2.8), ol.ptr(eo))
print(f"edges: |ref - oracle| > 1e-3 on {float((np.abs(e - eo) > 1e-3).mean()):.2e} of the pixels (full image), "
      f"{float((np.abs(out['edges'] - shrink(eo, KEEP_IMAGE)) > 1e-3).mean()):.2e} of the sample")
# one photometric Gauss-Newton iteration per level; the weights use the oracle's sigma
for l in range(3):
    q = rgb_level_inputs(od, l)
    w, h = q["w"], q["h"]
    corres = (DataTerm * (w * h))()
    cnt_o, sig_o = C.c_int(0), C.c_int(0)
    orc.L.orc_rgb_residual(C.c_float(q["minScale"]), ol.ptr(q["gx"]), ol.ptr(q["gy"]), ol.ptr(q["ld"]), ol.ptr(q["nd"]), ol.ptr(q["li"]), ol.ptr(q["ni"]),
                           corres, C.c_float(0.07), ol.ptr(q["kt"]), ol.ptr(q["krk"]), w, h, C.byref(cnt_o), C.byref(sig_o))
    cnt_r, sig_r = C.c_int(0), C.c_int(0)
    A = np.zeros(36, np.float32); b = np.zeros(6, np.float32)
    assert ref.ref_rgb_iteration(C.c_float(q["minScale"]), ol.ptr(q["gx"]), ol.ptr(q["gy"]), ol.ptr(q["ld"]), ol.ptr(q["nd"]), ol.ptr(q["li"]),
                                 ol.ptr(q["ni"]), C.c_float(0.07), ol.ptr(q["kt"]), ol.ptr(q["krk"]), C.c_float(float(cnt_o.value)),
                                 C.c_float(q["fx"]), C.c_float(q["fy"]), C.c_float(q["cx"]), C.c_float(q["cy"]), l, C.c_float(SOBEL_SCALE), w, h,
                                 C.byref(cnt_r), C.byref(sig_r), ol.ptr(A), ol.ptr(b)) == 0
    out[f"rgb{l}_sigma_from"] = np.int64(cnt_o.value)
    out[f"rgb{l}_count"], out[f"rgb{l}_sigma"], out[f"rgb{l}_A"], out[f"rgb{l}_b"] = np.int64(cnt_r.value), np.int64(sig_r.value), A, b
    print(f"rgb{l}: count ref {cnt_r.value} oracle {cnt_o.value}, sigma ref {sig_r.value} oracle {sig_o.value}")

path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "ref_kernels_golden.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes")
