"""Image-directory loader (mf_dir_*, the reference's ImageLogReader / "-dir" mode) on the CPU: file discovery, start index,
default prefixes, depth scale, mask description files, last-frame behaviour, error messages -- and the PNG decoder itself against
OpenCV (the library the reference decodes with) when cv2 is importable."""
from __future__ import annotations

import os
import struct
import zlib

import numpy as np
import pytest


def _chunk(t, d):
    return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xffffffff)


def write_png(path, a, filt=0):
    """minimal PNG writer (numpy + zlib): uint8 HxW / HxWx3 / HxWx4 or uint16 HxW; one filter type for all rows"""
    a = np.ascontiguousarray(a)
    h, w = a.shape[:2]
    ch = 1 if a.ndim == 2 else a.shape[2]
    bits = 16 if a.dtype == np.uint16 else 8
    ctype = {1: 0, 3: 2, 4: 6, 2: 4}[ch]
    raw = a.astype(">u2").tobytes() if bits == 16 else a.tobytes()
    row = w * ch * bits // 8
    bpp = max(1, ch * bits // 8)
    rows = np.frombuffer(raw, np.uint8).reshape(h, row).astype(np.int32)
    out = bytearray()
    prev = np.zeros(row, np.int32)
    for y in range(h):
        cur = rows[y]
        left = np.concatenate([np.zeros(bpp, np.int32), cur[:-bpp]])
        ul = np.concatenate([np.zeros(bpp, np.int32), prev[:-bpp]])
        if filt == 0:
            f = cur
        elif filt == 1:
            f = cur - left
        elif filt == 2:
            f = cur - prev
        elif filt == 3:
            f = cur - ((left + prev) >> 1)
        else:
            p = left + prev - ul
            pa, pb, pc = np.abs(p - left), np.abs(p - prev), np.abs(p - ul)
            pred = np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, prev, ul))
            f = cur - pred
        out += bytes([filt]) + (f & 255).astype(np.uint8).tobytes()
        prev = cur
    with open(path, "wb") as fp:
        fp.write(b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, bits, ctype, 0, 0, 0)))
        z = zlib.compress(bytes(out), 6)
        fp.write(_chunk(b"IDAT", z[: len(z) // 2]) + _chunk(b"IDAT", z[len(z) // 2:]) + _chunk(b"IEND", b""))


def make_dataset(root, n=5, start=1, W=64, H=48, masks=True, same_dir=False, seed=0):
    rng = np.random.default_rng(seed)
    cdir = os.path.join(root, "all" if same_dir else "rgb"); ddir = cdir if same_dir else os.path.join(root, "depth")
    mdir = cdir if same_dir else os.path.join(root, "mask")
    for d in {cdir, ddir, mdir}:
        os.makedirs(d, exist_ok=True)
    pre = ("Color", "Depth", "Mask") if same_dir else ("", "", "")
    frames = []
    for i in range(n):
        rgb = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        d16 = rng.integers(0, 6000, (H, W), dtype=np.uint16); d16[rng.random((H, W)) < 0.1] = 0
        m = rng.integers(0, 3, (H, W), dtype=np.uint8)
        idx = f"{i + start:04d}"
        write_png(os.path.join(cdir, pre[0] + idx + ".png"), rgb, filt=i % 5)
        write_png(os.path.join(ddir, pre[1] + idx + ".png"), d16, filt=(i + 2) % 5)
        if masks:
            with open(os.path.join(mdir, pre[2] + idx + ".pgm"), "wb") as fp:
                fp.write(b"P5\n# made by the test\n%d %d\n255\n" % (W, H) + m.tobytes())
            with open(os.path.join(mdir, pre[2] + idx + ".txt"), "w") as fp:
                fp.write("41 77\n1 2 30 40\n5 6 20 25\n")
        frames.append((rgb, d16, m))
    return cdir, ddir, (mdir if masks else None), frames


def test_dir_reader_roundtrip(product_lib, tmp_path):
    import maskfusion_b200 as mfb
    cdir, ddir, mdir, frames = make_dataset(str(tmp_path), n=5, start=1)
    rd = mfb.ImageLogReader(cdir, ddir, mdir)
    assert (rd.W, rd.H) == (64, 48) and rd.getNumFrames() == 5 and rd.hasMasks()
    got = 0
    while rd.hasMore():                                             # all five frames: no hidden last frame (ImageLogReader.cpp:326)
        rgb, depth, ts, mask, cls, rois = rd.getNext()
        r0, d0, m0 = frames[got]
        assert np.array_equal(rgb, r0)                              # file order RGB (imread BGR + unconditional swap, :247-248)
        assert np.array_equal(depth, np.float32(0.001) * d0.astype(np.float32))      # :262-268
        assert np.array_equal(mask, m0)
        assert cls.tolist() == [0, 41, 77]                          # leading background id (:306)
        assert rois.tolist() == [[2, 1, 38, 29], [6, 5, 19, 15]]    # cv::Rect(b, a, d-b, c-a) (:317)
        assert ts == int(np.float32(got) * np.float32(1000.0) / np.float32(24.0))    # :283
        got += 1
    assert got == 5
    with pytest.raises(mfb.MFError):
        rd.getNext()
    rd.close()


def test_dir_reader_default_prefixes_and_max_masks(product_lib, tmp_path):
    import maskfusion_b200 as mfb
    cdir, ddir, mdir, frames = make_dataset(str(tmp_path), n=4, start=0, same_dir=True)
    rd = mfb.ImageLogReader(cdir, ddir, mdir)                       # one directory, no prefixes given => Color/Depth/Mask (:79-84)
    assert rd.getNumFrames() == 4
    rd.setMaxMasks(2)                                               # "-nm 2": masks only for the first two frames (:271)
    seen = []
    while rd.hasMore():
        rgb, depth, ts, mask, cls, rois = rd.getNext()
        seen.append(mask is not None)
        assert np.array_equal(rgb, frames[len(seen) - 1][0])
    assert seen == [True, True, False, False]
    rd.close()


def test_dir_reader_errors(product_lib, tmp_path):
    import maskfusion_b200 as mfb
    cdir, ddir, mdir, frames = make_dataset(str(tmp_path), n=3, start=1, masks=False)
    os.remove(os.path.join(ddir, "0003.png"))
    with pytest.raises(mfb.MFError, match="RGB-frames != Depth-frames"):
        mfb.ImageLogReader(cdir, ddir)
    write_png(os.path.join(ddir, "0003.png"), np.zeros((48, 64), np.uint8))          # 8-bit depth: "Unsupported depth-files: 8UC1"
    rd = mfb.ImageLogReader(cdir, ddir)
    rd.getNext(); rd.getNext()
    with pytest.raises(mfb.MFError, match="Unsupported depth-files: 8UC1"):
        rd.getNext()
    rd.close()
    os.rename(os.path.join(cdir, "0002.png"), os.path.join(cdir, "0002.jpg"))
    with pytest.raises(mfb.MFError, match="same extension"):
        mfb.ImageLogReader(cdir, ddir)
    other = tmp_path / "x"; os.makedirs(other / "rgb"); os.makedirs(other / "depth")
    write_png(str(other / "rgb" / "0005.png"), np.zeros((4, 4, 3), np.uint8)); write_png(str(other / "depth" / "0005.png"), np.zeros((4, 4), np.uint16))
    with pytest.raises(mfb.MFError, match="start index"):
        mfb.ImageLogReader(str(other / "rgb"), str(other / "depth"))


def test_png_decoder_matches_opencv(product_lib, tmp_path):
    """pin the decoder against OpenCV -- the reference's decoder (cv::imread) -- on files OpenCV itself wrote (its own filter choice and
    compression): colour, 16-bit depth, gray mask, RGBA and gray colour inputs"""
    cv2 = pytest.importorskip("cv2")
    import maskfusion_b200 as mfb
    rng = np.random.default_rng(3)
    W, H = 80, 60
    root = str(tmp_path)
    for sub in ("rgb", "depth", "mask"):
        os.makedirs(os.path.join(root, sub))
    yy, xx = np.mgrid[0:H, 0:W]
    for i in range(3):
        bgr = np.stack([(xx * 3 + i * 20) % 256, (yy * 4 + xx) % 256, rng.integers(0, 256, (H, W))], -1).astype(np.uint8)
        if i == 1:
            bgr = np.concatenate([bgr, rng.integers(0, 256, (H, W, 1), dtype=np.uint8)], -1)       # BGRA file: imread drops alpha
        if i == 2:
            bgr = ((xx + yy) % 256).astype(np.uint8)                                             # gray file: imread replicates
        d16 = ((xx * 37 + yy * 91 + i * 1000) % 65536).astype(np.uint16)
        m = ((xx // 20 + yy // 20) % 4).astype(np.uint8)
        assert cv2.imwrite(os.path.join(root, "rgb", f"{i:04d}.png"), bgr)
        assert cv2.imwrite(os.path.join(root, "depth", f"{i:04d}.png"), d16)
        assert cv2.imwrite(os.path.join(root, "mask", f"{i:04d}.png"), m)
    rd = mfb.ImageLogReader(os.path.join(root, "rgb"), os.path.join(root, "depth"), os.path.join(root, "mask"))
    for i in range(3):
        rgb, depth, ts, mask, cls, rois = rd.getNext()
        ref_rgb = cv2.imread(os.path.join(root, "rgb", f"{i:04d}.png"))[:, :, ::-1]              # imread + flipColors()
        ref_d = cv2.imread(os.path.join(root, "depth", f"{i:04d}.png"), cv2.IMREAD_UNCHANGED)
        ref_m = cv2.imread(os.path.join(root, "mask", f"{i:04d}.png"), cv2.IMREAD_GRAYSCALE)
        assert np.array_equal(rgb, ref_rgb), i
        assert np.array_equal(depth, np.float32(0.001) * ref_d.astype(np.float32)), i
        assert np.array_equal(mask, ref_m), i
        assert cls is None
    rd.close()


def test_jpeg_decoder_matches_libjpeg(product_lib):
    """the in-tree baseline JPEG decoder restates libjpeg's default path (islow IDCT, fancy upsampling, fixed-point colour
    conversion): bit-identical to OpenCV's decoder (libjpeg-turbo) over sampling modes, qualities, restart intervals, odd sizes"""
    cv2 = pytest.importorskip("cv2")
    from maskfusion_b200.api import decode_jpeg
    import maskfusion_b200 as mfb
    rng = np.random.default_rng(0)
    n = 0
    for (W, H) in [(64, 48), (67, 45), (17, 9), (1, 1), (320, 240)]:
        yy, xx = np.mgrid[0:H, 0:W]
        for a in (rng.integers(0, 256, (H, W, 3), dtype=np.uint8),
                  np.stack([128 + 100 * np.sin(xx / 7.0) * np.cos(yy / 5.0), 128 + 120 * np.sin((xx + yy) / 11.0), (xx * yy) % 256], -1).clip(0, 255).astype(np.uint8)):
            for q in (30, 90, 100):
                for sf in (cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420):
                    for rst in (0, 3):
                        ok, buf = cv2.imencode(".jpg", a, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, sf, cv2.IMWRITE_JPEG_RST_INTERVAL, rst])
                        assert ok
                        ref = cv2.imdecode(buf, cv2.IMREAD_COLOR)[:, :, ::-1]
                        assert np.array_equal(decode_jpeg(buf.tobytes()), ref), (W, H, q, sf, rst)
                        n += 1
    ok, buf = cv2.imencode(".jpg", rng.integers(0, 256, (30, 41), dtype=np.uint8), [cv2.IMWRITE_JPEG_QUALITY, 80])       # single component
    assert np.array_equal(decode_jpeg(buf.tobytes()), cv2.imdecode(buf, cv2.IMREAD_COLOR)[:, :, ::-1])
    ok, buf = cv2.imencode(".jpg", rng.integers(0, 256, (32, 32, 3), dtype=np.uint8), [cv2.IMWRITE_JPEG_PROGRESSIVE, 1])
    with pytest.raises(mfb.MFError, match="progressive"):
        decode_jpeg(buf.tobytes())
    assert n == 180


def test_klg_with_jpeg_colour_and_zlib_depth(product_lib, tmp_path):
    """the compressed .klg layout Logger2 writes (KlgLogReader.cpp:53-89): zlib depth, JPEG colour decoded as JPEGLoader.h does
    (libjpeg RGB rows with R and B exchanged, :72-81), then the optional -f flip"""
    cv2 = pytest.importorskip("cv2")
    import maskfusion_b200 as mfb
    W, H, n = 64, 48, 3
    rng = np.random.default_rng(1)
    yy, xx = np.mgrid[0:H, 0:W]
    path = str(tmp_path / "c.klg")
    frames = []
    with open(path, "wb") as fp:
        fp.write(struct.pack("<i", n + 1))
        for i in range(n + 1):
            d16 = rng.integers(0, 5000, (H, W), dtype=np.uint16)
            img = np.stack([(xx * 3 + i * 9) % 256, (yy * 5) % 256, (xx + yy) % 256], -1).astype(np.uint8)
            ok, jpg = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, 90])
            z = zlib.compress(d16.tobytes())
            fp.write(struct.pack("<qii", 1000 * i, len(z), len(jpg)) + z + jpg.tobytes())
            frames.append((d16, cv2.imdecode(jpg, cv2.IMREAD_COLOR)))       # BGR == libjpeg RGB with R/B exchanged
    for flip in (False, True):
        rd = mfb.KlgLogReader(path, W, H, flipColors=flip)
        k = 0
        while rd.hasMore():
            rgb, depth, ts = rd.getNext()
            d16, bgr = frames[k]
            assert ts == 1000 * k
            assert np.array_equal(depth, (d16.astype(np.float64) * 0.001).astype(np.float32))
            assert np.array_equal(rgb, bgr[:, :, ::-1] if flip else bgr)
            k += 1
        assert k == n                                                       # the last frame of a .klg is never delivered (N11)
        rd.close()


def test_dir_reader_jpeg_colour(product_lib, tmp_path):
    cv2 = pytest.importorskip("cv2")
    import maskfusion_b200 as mfb
    root = str(tmp_path)
    os.makedirs(os.path.join(root, "rgb")); os.makedirs(os.path.join(root, "depth"))
    rng = np.random.default_rng(2)
    for i in range(2):
        cv2.imwrite(os.path.join(root, "rgb", f"{i:04d}.jpg"), rng.integers(0, 256, (50, 70, 3), dtype=np.uint8))
        cv2.imwrite(os.path.join(root, "depth", f"{i:04d}.png"), rng.integers(0, 4000, (50, 70), dtype=np.uint16))
    rd = mfb.ImageLogReader(os.path.join(root, "rgb"), os.path.join(root, "depth"))
    for i in range(2):
        rgb, depth, ts, mask, cls, rois = rd.getNext()
        assert np.array_equal(rgb, cv2.imread(os.path.join(root, "rgb", f"{i:04d}.jpg"))[:, :, ::-1])
        assert mask is None
    rd.close()


def test_decoders_match_committed_opencv_vectors(product_lib, tmp_path):
    """the same pin without cv2: byte streams encoded AND decoded by OpenCV, committed by tests/golden/make_loader_golden.py"""
    import maskfusion_b200 as mfb
    from maskfusion_b200.api import decode_jpeg
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loader_golden.npz"))
    for k in range(int(g["njpg"])):
        assert np.array_equal(decode_jpeg(g[f"jpg{k}"].tobytes()), g[f"jpg{k}_rgb"]), k
    # the PNG decoder is reached through the directory reader: colour / BGRA colour + 16-bit depth + 8-bit mask
    for ci, cname in enumerate(("png_rgb", "png_rgba")):
        root = tmp_path / f"set{ci}"
        for sub, name in (("rgb", cname), ("depth", "png_d16"), ("mask", "png_m8")):
            os.makedirs(root / sub, exist_ok=True)
            (root / sub / "0000.png").write_bytes(g[name].tobytes())
        rd = mfb.ImageLogReader(str(root / "rgb"), str(root / "depth"), str(root / "mask"))
        rgb, depth, ts, mask, cls, rois = rd.getNext()
        assert np.array_equal(rgb, g[cname + "_dec"])
        assert np.array_equal(depth, np.float32(0.001) * g["png_d16_dec"].astype(np.float32))
        assert np.array_equal(mask, g["png_m8_dec"])
        rd.close()


def test_generate_id_image_matches_reference_python(product_lib):
    """Mask R-CNN post-processing (MaskRCNN/helpers.py:70-98) against vectors produced by importing the reference's own function
    (tests/golden/make_idimage_golden.py): score threshold, class filter,
    special assignments, overwrite order, nothing exported; five hand-made cases and twenty seeded random ones"""
    from maskfusion_b200.api import generate_id_image
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "idimage_golden.npz"))
    for k in range(int(g["ncases"])):
        r = {"masks": g[f"c{k}_masks"], "scores": g[f"c{k}_scores"], "class_ids": g[f"c{k}_class_ids"], "rois": g[f"c{k}_rois"]}
        img, cls, rois = generate_id_image(r, float(g[f"c{k}_min_score"]), g[f"c{k}_filter"].tolist(), g[f"c{k}_special"].tolist())
        assert np.array_equal(img, g[f"c{k}_img"]), k
        assert cls == g[f"c{k}_out_cls"].tolist(), k
        assert np.array_equal(np.array(rois, np.int32).reshape(-1, 4), g[f"c{k}_out_rois"]), k
    assert int(g["ncases"]) == 25


def test_dir_reader_reads_what_the_reference_writes(product_lib, tmp_path):
    """the mask image + description file written by the reference's save_id_image (MaskRCNN/helpers.py:101-113, the -maskdir
    data produced by offline_runner.py) come back through the directory reader as the same id image, class ids and boxes"""
    import maskfusion_b200 as mfb
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "idimage_golden.npz"))
    H, W = g["saved_img"].shape
    for sub in ("rgb", "depth", "mask"):
        os.makedirs(tmp_path / sub)
    write_png(str(tmp_path / "rgb" / "0000.png"), np.zeros((H, W, 3), np.uint8))
    write_png(str(tmp_path / "depth" / "0000.png"), np.zeros((H, W), np.uint16))
    (tmp_path / "mask" / "0000.png").write_bytes(g["saved_png"].tobytes())
    (tmp_path / "mask" / "0000.txt").write_bytes(g["saved_txt"].tobytes())
    rd = mfb.ImageLogReader(str(tmp_path / "rgb"), str(tmp_path / "depth"), str(tmp_path / "mask"))
    rgb, depth, ts, mask, cls, rois = rd.getNext()
    assert np.array_equal(mask, g["saved_img"])
    assert cls.tolist() == [0] + g["saved_cls"].tolist()
    # the file holds y1 x1 y2 x2 (helpers.py:111-113); the reader builds cv::Rect(x1, y1, x2 - x1, y2 - y1) (ImageLogReader.cpp:314-317)
    y1, x1, y2, x2 = g["saved_rois"].T
    assert np.array_equal(rois, np.stack([x1, y1, x2 - x1, y2 - y1], 1))
    rd.close()


def test_write_ply_layout(product_lib, tmp_path):
    """MaskFusion::savePly (MaskFusion.cpp:733-848): header, confidence gate, packed colour -> r g b, negated normals, radius"""
    from maskfusion_b200.api import write_ply
    rng = np.random.default_rng(5)
    n = 50
    s = rng.normal(size=(n, 12)).astype(np.float32)
    s[:, 3] = rng.uniform(0, 20, n)                                   # confidence
    col = rng.integers(0, 256, (n, 3))
    s[:, 4] = ((col[:, 0] << 16) + (col[:, 1] << 8) + col[:, 2]).astype(np.float32)
    s[:, 11] = rng.uniform(0.001, 0.02, n)
    path = str(tmp_path / "cloud-0.ply")
    kept = s[:, 3] > 10.0
    assert write_ply(path, s, 10.0) == int(kept.sum())
    raw = open(path, "rb").read()
    head, body = raw.split(b"end_header\n", 1)
    assert head.decode().split("\n")[:3] == ["ply", "format binary_little_endian 1.0", f"element vertex {int(kept.sum())}"]
    assert [l for l in head.decode().split("\n") if l.startswith("property")] == [
        "property float x", "property float y", "property float z", "property uchar red", "property uchar green", "property uchar blue",
        "property float nx", "property float ny", "property float nz", "property float radius"]
    rec = np.dtype([("p", "<f4", 3), ("c", "u1", 3), ("n", "<f4", 3), ("r", "<f4")])
    v = np.frombuffer(body, rec)
    assert len(v) == int(kept.sum())
    assert np.array_equal(v["p"], s[kept, 0:3]) and np.array_equal(v["c"], col[kept].astype(np.uint8))
    assert np.array_equal(v["n"], -s[kept, 8:11]) and np.array_equal(v["r"], s[kept, 11])


def test_corrupt_streams_are_rejected_not_crashed(product_lib, tmp_path):
    """malformed JPEG / PNG / PNM headers (ADVICE r1): table selectors above 3 in the scan header, a frame component the scan
    never names, duplicate component ids, an empty SOS, implausible image sizes -- every case returns an error (or, for random
    bit flips, any result) through the C ABI; nothing reads out of bounds, throws across the boundary or terminates"""
    import maskfusion_b200 as mfb
    from maskfusion_b200.api import decode_jpeg
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loader_golden.npz"))
    good = bytearray(g["jpg0"].tobytes())
    sos = good.find(b"\xff\xda")
    sof = good.find(b"\xff\xc0")
    assert sos > 0 and sof > 0 and good[sos + 4] == 3
    bad = bytearray(good); bad[sos + 6] = 0xF0                      # td = 15 for the first component
    with pytest.raises(mfb.MFError, match="Huffman table outside"):
        decode_jpeg(bytes(bad))
    bad = bytearray(good); bad[sos + 6] = 0x0F                      # ta = 15
    with pytest.raises(mfb.MFError, match="Huffman table outside"):
        decode_jpeg(bytes(bad))
    bad = bytearray(good); bad[sos + 7] = bad[sos + 5]              # the scan names component 1 twice, component 2 never
    with pytest.raises(mfb.MFError, match="unknown component|missing from the scan"):
        decode_jpeg(bytes(bad))
    bad = bytearray(good); bad[sof + 13] = bad[sof + 10]            # duplicate component ids in the frame header: the scan's id-2 entry finds no taker
    with pytest.raises(mfb.MFError, match="unknown component|missing from the scan"):
        decode_jpeg(bytes(bad))
    bad = bytearray(good[:sos]) + b"\xff\xda\x00\x02" + good[sos + 4:]     # SOS with an empty body
    with pytest.raises(mfb.MFError):
        decode_jpeg(bytes(bad))
    bad = bytearray(good); bad[sof + 5:sof + 9] = b"\xff\xff\xff\xff"      # 65535 x 65535
    with pytest.raises(mfb.MFError, match="16384"):
        decode_jpeg(bytes(bad))
    rng = np.random.default_rng(7)
    for _ in range(300):                                                     # random byte damage after the SOI marker
        b = bytearray(good)
        for p in rng.integers(2, len(b), rng.integers(1, 6)):
            b[p] = int(rng.integers(0, 256))
        try:
            decode_jpeg(bytes(b))
        except mfb.MFError:
            pass
    # PNG with a 2^31-1 IHDR and a PGM with a huge header reach the directory reader
    for name, payload in (("0000.png", b"\x89PNG\r\n\x1a\n" + _chunk(b"IHDR", struct.pack(">IIBBBBB", 0x7fffffff, 0x7fffffff, 8, 2, 0, 0, 0)) + _chunk(b"IDAT", zlib.compress(b"\0")) + _chunk(b"IEND", b"")),
                          ("0000.ppm", b"P6\n99999999999 99999999999\n255\n" + b"\0" * 64)):
        root = tmp_path / name.replace(".", "_")
        os.makedirs(root / "rgb"); os.makedirs(root / "depth")
        (root / "rgb" / name).write_bytes(payload)
        write_png(str(root / "depth" / "0000.png"), np.zeros((4, 4), np.uint16))
        with pytest.raises(mfb.MFError, match="16384"):
            mfb.ImageLogReader(str(root / "rgb"), str(root / "depth"), None)
    L = mfb.load_library()
    assert not L.mf_klg_open(None, 640, 480, 0)
    assert not L.mf_klg_open(b"/nonexistent.klg", -1, 480, 0)


def test_exr_depth_decoder_matches_opencv_golden(tmp_path):
    """in-tree OpenEXR scan-line decoder (HALF/FLOAT, NONE/RLE/ZIPS/ZIP, gray and R,G,B files) against OpenCV's decode of the same
    streams (tests/golden/make_exr_golden.py), bit for bit; through the -dir reader as well (ImageLogReader.cpp:251-258)"""
    import maskfusion_b200 as mfb
    from maskfusion_b200.api import decode_exr_depth, MFError
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "exr_golden.npz"))
    n = int(g["nexr"])
    assert n >= 40
    for k in range(n):
        d = decode_exr_depth(g[f"exr{k}"].tobytes())
        ref = g[f"exr{k}_depth"]
        assert d.shape == ref.shape and np.array_equal(d.view(np.uint32), ref.view(np.uint32)), k
    with pytest.raises(MFError, match="PIZ"):
        decode_exr_depth(g["exr_piz"].tobytes())
    for bad in (b"", b"abcd" * 8, g["exr0"].tobytes()[:60], g["exr3"].tobytes()[:-9]):
        with pytest.raises(MFError):
            decode_exr_depth(bad)
    # corrupted streams either decode to something or are refused with a message -- never a crash (the entry point is behind the C ABI)
    rng = np.random.default_rng(0)
    for k in range(0, n, 3):
        b = bytearray(g[f"exr{k}"].tobytes())
        for _ in range(25):
            c = bytearray(b)
            for _ in range(int(rng.integers(1, 6))):
                c[int(rng.integers(0, len(c)))] = int(rng.integers(0, 256))
            if rng.random() < 0.2:
                c = c[: int(rng.integers(1, len(c)))]
            try:
                decode_exr_depth(bytes(c))
            except MFError:
                pass
    # a two-frame image directory with EXR depth
    ref = g["exr0_depth"]
    H, W = ref.shape
    rgb = (np.arange(H * W * 3) % 251).astype(np.uint8).reshape(H, W, 3)
    for i in range(2):
        with open(tmp_path / f"Color{i:04d}.ppm", "wb") as f:
            f.write(b"P6\n%d %d\n255\n" % (W, H)); f.write(rgb.tobytes())
        with open(tmp_path / f"Depth{i:04d}.exr", "wb") as f:
            f.write(g["exr0"].tobytes())
    rd = mfb.ImageLogReader(str(tmp_path), indexWidth=4)
    assert rd.getNumFrames() == 2
    fr = rd.getNext()
    assert np.array_equal(np.asarray(fr[1]).view(np.uint32), ref.view(np.uint32))
    rd.close()


def _preseg_python(mask, depth, model_ids, next_id, allow_new, mapping):
    """literal restatement of PreSegmentation::performSegmentation (Core/Segmentation/PreSegmentation.cpp:28-90) with float32 running sums"""
    H, W = mask.shape
    m, d = mask.reshape(-1), depth.reshape(-1).astype(np.float32)
    seg = np.zeros(H * W, np.uint8)
    idx = {int(v): i for i, v in enumerate(model_ids)}
    idx[int(next_id)] = len(model_ids)
    out_ids = [0] * 256
    has_new = False
    for i in range(H * W):
        v = int(m[i])
        if v:
            if mapping[v] != 0:
                seg[i] = mapping[v]; out_ids[seg[i]] += 1
            elif allow_new and not has_new:
                seg[i] = next_id; mapping[v] = next_id; has_new = True; out_ids[next_id] += 1
        else:
            out_ids[0] += 1
    n = len(model_ids) + (1 if has_new else 0)
    spc = [out_ids[int(v)] // 256 for v in model_ids]
    if has_new:
        spc.append(int(max(np.float32(out_ids[next_id] // 256), np.float32(1.0))))
    mean = [np.float32(0)] * n; std = [np.float32(0)] * n; cnt = [0] * n
    for i in range(H * W):
        k = idx.get(int(seg[i]), 0)
        if k < n:
            mean[k] = np.float32(mean[k] + d[i]); cnt[k] += 1
    mean = [np.float32(mean[k] / np.float32(cnt[k] if cnt[k] else 1)) for k in range(n)]
    for i in range(H * W):
        k = idx.get(int(seg[i]), 0)
        if k < n:
            std[k] = np.float32(std[k] + np.float32(abs(np.float32(mean[k] - d[i]))))
    std = [np.float32(std[k] / np.float32(cnt[k] if cnt[k] else 1)) for k in range(n)]
    return seg.reshape(H, W), has_new, np.array(spc, np.uint32), np.array(mean, np.float32), np.array(std, np.float32)


def test_pre_segmentation_matches_restatement():
    """mf_pre_segmentation (the reference's precomputed-masks performer, host code) against a literal Python restatement over a short replay: the
    persistent mapping table, one new label per frame in raster order, superpixel counts, float32 running depth statistics -- bit for bit"""
    from maskfusion_b200.api import pre_segmentation
    rng = np.random.default_rng(9)
    H, W = 48, 64
    map_c = np.zeros(256, np.uint8); map_p = np.zeros(256, np.uint8)
    model_ids = [0]
    next_id = 1
    labels = [17, 40, 3, 200]
    for t in range(7):
        mask = np.zeros((H, W), np.uint8)
        for j, lab in enumerate(labels[: 1 + t // 2 + 1]):
            y0, x0 = 4 + 9 * j + t, 6 + 13 * j
            mask[y0:y0 + 12, x0:x0 + 14] = lab
        depth = (1.0 + rng.random((H, W)) * 2).astype(np.float32)
        depth[rng.random((H, W)) < 0.05] = 0.0
        allow = t != 3                                        # one frame in which new models are not allowed
        seg_c, new_c, spc_c, mean_c, std_c = pre_segmentation(mask, depth, model_ids, next_id, allow, map_c)
        seg_p, new_p, spc_p, mean_p, std_p = _preseg_python(mask, depth, model_ids, next_id, allow, map_p)
        assert np.array_equal(seg_c, seg_p) and new_c == new_p, t
        assert np.array_equal(map_c, map_p)
        assert np.array_equal(spc_c, spc_p), (t, spc_c, spc_p)
        assert np.array_equal(mean_c.view(np.uint32), mean_p.view(np.uint32)) and np.array_equal(std_c.view(np.uint32), std_p.view(np.uint32)), t
        if new_c:
            model_ids.append(next_id); next_id += 1
    assert len(model_ids) >= 4 and map_c[17] == 1 and map_c[40] == 2
