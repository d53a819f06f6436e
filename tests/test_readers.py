"""Format readers (VDB-224 + Blosc/LZ4, Radiance HDR, BMP, EXR) against the committed fixtures and the
files' own metadata -- the only pins these formats offer (SURVEY 8(c), Appendix A)."""
import os

import numpy as np
import pytest

import vpt_b200 as V
from vpt_b200.scene import load_vdb_grid, load_bmp_rbg, load_exr_rgb, load_hdr, find_asset


def test_dragon_vdb_matches_file_metadata_and_survey_numbers():
    dens, meta = load_vdb_grid(find_asset("dragon.vdb"), "density")
    assert dens.shape == (31, 49, 70) and meta["dim"] == (70, 49, 31)
    assert meta["bbox_min"] == (16, 1, 35) and meta["bbox_max"] == (85, 49, 65)
    assert meta["active_voxels"] == 19660 and meta["leaf_count"] == 131           # file_voxel_count metadata, checked inside the reader too
    assert meta["max_value"] == 1.0 and meta["min_density"] == np.float32(np.finfo(np.float32).eps)   # quirk Q10
    assert abs(float(dens.mean()) - 0.0958042) < 1e-6 and abs(float((dens != 0).mean()) - 0.185) < 1e-3
    assert abs(meta["voxel_size"] - 0.1) < 1e-7
    X = meta["xform"]
    assert np.allclose(np.diag(X), [0.1, 0.1, 0.1, 1.0]) and np.count_nonzero(X) == 4


def test_vdb_missing_grid_and_bad_file(tmp_path):
    assert load_vdb_grid(find_asset("dragon.vdb"), "no_such_grid") is None
    bad = tmp_path / "bad.vdb"; bad.write_bytes(b"not a vdb file at all, definitely")
    with pytest.raises(V.VptError):
        load_vdb_grid(str(bad), "density")
    trunc = tmp_path / "trunc.vdb"; trunc.write_bytes(open(find_asset("dragon.vdb"), "rb").read()[:5000])
    with pytest.raises(V.VptError):
        load_vdb_grid(str(trunc), "density")


_LARGE_VDBS = ("fireball.vdb", "colored_smoke.vdb", "dragon_with_xform.vdb")


@pytest.mark.skipif(any(find_asset(n) is None for n in _LARGE_VDBS), reason="large reference assets not staged (oracle/_ref/assets)")
def test_large_reference_vdbs_decode_to_their_metadata():
    dens, m = load_vdb_grid(find_asset("fireball.vdb"), "density")
    assert m["dim"] == (239, 257, 234) and m["active_voxels"] == 4901516 and abs(m["max_value"] - 12.4696) < 1e-3
    heat, mh = load_vdb_grid(find_asset("fireball.vdb"), "heat")
    assert mh["dim"] == (270, 288, 268) and mh["active_voxels"] == 20839680 and abs(mh["background"] + 0.01) < 1e-6
    cd, mc = load_vdb_grid(find_asset("colored_smoke.vdb"), "Cd")
    assert mc["channels"] == 3 and cd.shape[-1] == 3 and mc["active_voxels"] == 1676306
    d2, m2 = load_vdb_grid(find_asset("dragon_with_xform.vdb"), "density")
    assert m2["active_voxels"] == 156161 and m2["dim"] == (141, 99, 63)


def test_blue_noise_bmp_channel_swap():
    bn = load_bmp_rbg(find_asset("BN0.bmp"))
    assert bn.shape == (256, 256, 3)
    # first pixel of BN0.bmp is R=26 G=70 B=108: x = R/255, y = B/255, z = G/255 (quirk Q16)
    assert np.allclose(bn[0, 0], [26 / 255.0, 108 / 255.0, 70 / 255.0])
    assert 0.45 < bn.mean() < 0.55


def test_exr_luts():
    bb = load_exr_rgb(find_asset("blackbody_texture.exr"))
    assert bb.shape == (1, 256, 3)
    assert np.allclose(bb[0, 0], [5.9604645e-06, 1.0430813e-05, 2.6345253e-05], rtol=1e-6)
    assert np.allclose(bb[0, -1], [0.9711914, 0.8720703, 0.72265625])
    dc = load_exr_rgb(find_asset("density_color_texture2.exr"))
    assert dc.shape == (1, 256, 3) and np.all(dc == 1.0)


def test_hdr_rgbe_rule(tmp_path):
    # two scanlines: one flat (non-RLE because width < 8), values follow (m + 0.5) * 2^(e - 136)
    p = tmp_path / "t.hdr"
    px = bytes([128, 64, 32, 129,  0, 0, 0, 0,  255, 255, 255, 128,  1, 2, 3, 120])
    p.write_bytes(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y 2 +X 2\n" + px)
    img = load_hdr(str(p))
    assert img.shape == (2, 2, 4)
    assert np.allclose(img[0, 0, :3], [(128 + 0.5) * 2.0 ** -7, (64 + 0.5) * 2.0 ** -7, (32 + 0.5) * 2.0 ** -7])
    assert np.all(img[0, 1, :3] == 0) and np.all(img[..., 3] == 0)
    assert np.allclose(img[1, 0, :3], [(255.5) * 2.0 ** -8] * 3)
    hdr = find_asset("Barce_Rooftop_C_3k.hdr")
    if hdr:
        big = load_hdr(hdr)
        assert big.shape == (1500, 3000, 4) and abs(float(big[..., :3].mean()) - 0.245057) < 1e-4


def test_ins_scene_file_reader(tmp_path):
    """`.ins` grammar of the reference's read_instance_file (main.cpp:980-1040): volumes form."""
    from vpt_b200.scene import load_ins
    p = tmp_path / "two.ins"
    p.write_text("2\n./assets/dragon.vdb\n3\n0 0 0 0 0 0 1 1\n1.5 -2 3e0 0.0 0.7071068 0 0.7071068 0.5\n-4 5 6 1 0 0 0 2\r\n"
                 "clouds/cumulus 01.vdb\n1\n10 20 30 0 0 0 1 0.25\n")
    d = load_ins(str(p))
    assert d["kind"] == "volumes" and [f["path"] for f in d["files"]] == ["./assets/dragon.vdb", "clouds/cumulus 01.vdb"]
    assert [len(f["instances"]) for f in d["files"]] == [3, 1]
    pos, quat, scale = d["files"][0]["instances"][1]
    assert pos == (1.5, -2.0, 3.0) and quat == (0.0, 0.7071068, 0.0, 0.7071068) and scale == 0.5
    assert d["files"][1]["instances"][0] == ((10.0, 20.0, 30.0), (0.0, 0.0, 0.0, 1.0), 0.25)


def test_ins_light_file_reader_and_errors(tmp_path):
    from vpt_b200.scene import load_ins
    p = tmp_path / "lights.ins"
    p.write_text("light\n2\n9 6 2 1 0.8 0.6 40\n-2 3 8 0.5 0.7 1 25\n")
    d = load_ins(str(p))
    assert d == {"kind": "lights", "lights": [((9.0, 6.0, 2.0), (1.0, 0.8, 0.6), 40.0), ((-2.0, 3.0, 8.0), (0.5, 0.7, 1.0), 25.0)]}
    bad = tmp_path / "short.ins"
    bad.write_text("1\nfoo.vdb\n2\n0 0 0 0 0 0 1 1\n1 2 3\n")                 # second record has too few numbers
    with pytest.raises(V.VptError, match="8 numbers"):
        load_ins(str(bad))
    with pytest.raises(V.VptError, match="cannot open"):
        load_ins(str(tmp_path / "missing.ins"))
    empty = tmp_path / "empty.ins"; empty.write_text("")
    with pytest.raises(V.VptError, match="empty file"):
        load_ins(str(empty))


def _analytic_sky_numpy(azimuth, elevation, res):
    """Independent float64 restatement of the reference's host-side sky (source/main.cpp:242-301) and of the direction grid of
    create_cdf (:683-693), vectorised over the res x res directions."""
    pi = np.pi
    az = np.clip(azimuth, 0, 360) * pi / 180; el = (90 - np.clip(elevation, 0, 90)) * pi / 180
    sun = np.array([np.sin(el) * np.cos(az), np.cos(el), np.sin(el) * np.sin(az)]); sun /= np.linalg.norm(sun)
    e = (np.arange(res) / (res - 1) * pi)[:, None]; a = (np.arange(res) / (res - 1) * 2 * pi)[None, :]
    d = np.stack([np.sin(e) * np.cos(a), np.cos(e) + 0 * a, np.sin(e) * np.sin(a)], axis=-1).reshape(-1, 3)
    Re, Ra, Hr, Hm = 6360e3, 6420e3, 7994.0, 1200.0
    bR = np.array([3.8e-6, 13.5e-6, 33.1e-6]); bM = np.array([21e-6] * 3)
    pos = np.array([0.0, 1000 + 6360e3, 0.0])

    def hit(o, dd, r):                                       # smaller / larger root of |o + t dd| = r (nan where none)
        A = (dd * dd).sum(-1); B = 2 * (dd * o).sum(-1); Cc = (o * o).sum(-1) - r * r
        disc = B * B - 4 * A * Cc
        ok = disc >= 0
        sq = np.sqrt(np.where(ok, disc, 0))
        q = np.where(B < 0, -0.5 * (B - sq), -0.5 * (B + sq))
        with np.errstate(divide="ignore", invalid="ignore"):
            x1 = q / A; x2 = Cc / q
        return ok, np.minimum(x1, x2), np.maximum(x1, x2)

    n = d.shape[0]
    oke, t0e, t1e = hit(pos[None, :], d, Re)
    tmax = np.where(oke & (t1e > 0), np.maximum(0, t0e), np.inf)
    oka, t0a, t1a = hit(pos[None, :], d, Ra)
    red = ~oka | (t1a < 0)
    tmin = np.where((t0a > 0), t0a, 0.0)
    tmax = np.minimum(tmax, t1a)
    seg = (tmax - tmin) / 16
    mu = d @ sun
    phR = 3 / (16 * pi) * (1 + mu * mu); g = 0.76
    phM = 3 / (8 * pi) * ((1 - g * g) * (1 + mu * mu)) / ((2 + g * g) * (1 + g * g - 2 * g * mu) ** 1.5)
    sumR = np.zeros((n, 3)); sumM = np.zeros((n, 3)); dR = np.zeros(n); dM = np.zeros(n); t = tmin.copy()
    for _ in range(16):
        p = pos[None, :] + (t + seg * 0.5)[:, None] * d
        h = np.linalg.norm(p, axis=1) - Re
        hr = np.exp(-h / Hr) * seg; hm = np.exp(-h / Hm) * seg
        dR += hr; dM += hm
        _, _, t1l = hit(p, sun[None, :], Ra)
        sl = t1l / 8; tl = np.zeros(n); lr = np.zeros(n); lm = np.zeros(n); alive = np.ones(n, bool)
        for _ in range(8):
            pl = p + (tl + sl * 0.5)[:, None] * sun[None, :]
            hl = np.linalg.norm(pl, axis=1) - Re
            alive &= hl >= 0
            lr += np.where(alive, np.exp(-hl / Hr) * sl, 0); lm += np.where(alive, np.exp(-hl / Hm) * sl, 0)
            tl += sl
        tau = bR[None, :] * (dR + lr)[:, None] + bM[None, :] * 1.1 * (dM + lm)[:, None]
        att = np.exp(-tau)
        sumR += np.where(alive[:, None], att * hr[:, None], 0); sumM += np.where(alive[:, None], att * hm[:, None], 0)
        t += seg
    rgb = sumR * bR[None, :] * phR[:, None] + sumM * bM[None, :] * phM[:, None]
    rgb[red] = [1.0, 0.0, 0.0]
    return np.linalg.norm(rgb, axis=1).reshape(res, res)


@pytest.mark.parametrize("az,el", [(120.0, 30.0), (300.0, 75.0), (10.0, 2.0)])
def test_env_sky_tabulation_matches_independent_restatement(az, el):
    """vpt_env_sky_tabulate (host fp32) against a float64 numpy restatement of main.cpp:242-301 / :683-693."""
    from vpt_b200.scene import sky_power_table
    res = 48
    got = sky_power_table(az, el, (1.0, 1.0, 1.0), res).astype(np.float64)
    want = _analytic_sky_numpy(az, el, res)
    assert got.shape == (res, res) and np.isfinite(got).all() and got.min() > 0
    # fp32 marching vs fp64: agree to a few 1e-3 except where the view ray grazes the planet (t0 of a near-tangent quadratic)
    rel = np.abs(got - want) / np.maximum(want, 1e-12)
    assert np.quantile(rel, 0.98) < 5e-3 and np.median(rel) < 5e-4, (np.quantile(rel, 0.98), np.median(rel))
    # colour scaling is linear (intensity multiplies the radiance, main.cpp:300)
    half = sky_power_table(az, el, (0.5, 0.5, 0.5), res).astype(np.float64)
    assert np.allclose(half, 0.5 * got, rtol=1e-5)


def _mutations(blob, seed, n, header_bias=400):
    """Deterministic single-field corruptions: truncations, 1/4/8-byte overwrites with extreme values, mostly in the header
    region where the offsets / counts / sizes live."""
    rng = np.random.RandomState(seed)
    out = []
    for i in range(n):
        b = bytearray(blob)
        kind = i % 4
        if kind == 0:
            out.append(bytes(b[:int(rng.randint(1, len(b)))])); continue
        pos = int(rng.randint(0, min(len(b) - 8, header_bias))) if rng.rand() < 0.7 else int(rng.randint(0, len(b) - 8))
        pick = lambda vals: vals[int(rng.randint(0, len(vals)))]
        if kind == 1: b[pos] = pick([0, 1, 0x7f, 0x80, 0xff])
        elif kind == 2: b[pos:pos + 4] = pick([0, 0x7fffffff, 0x80000000, 0xffffffff, 0xfffffff0]).to_bytes(4, "little")
        else: b[pos:pos + 8] = pick([0, 0x7fffffffffffffff, 0x8000000000000000, 0xffffffffffffffff, len(b) + 1, 0xfffffffffffffff0]).to_bytes(8, "little")
        out.append(bytes(b))
    return out


def test_corrupt_vdb_files_fail_cleanly(tmp_path):
    """ADVICE r1: sizes and offsets taken from the file (grid/block/end positions, Blosc block starts, typesize, bbox) must be
    validated: a malformed .vdb either decodes or raises VptError -- it never reads out of bounds (this test would crash)."""
    blob = open(find_asset("dragon.vdb"), "rb").read()
    # the descriptor offsets live right after the grid name/type strings: make sure those bytes are hit, too
    at = blob.index(b"Tree_float_5_4_3")
    p = tmp_path / "m.vdb"
    ok = bad = 0
    for m in _mutations(blob, 5, 160) + _mutations(blob[:at + 200] + blob[at + 200:], 6, 80, header_bias=at + 120):
        p.write_bytes(m)
        try:
            got = load_vdb_grid(str(p), "density")
            ok += 1
            if got is not None: assert got[0].size <= 1 << 28
        except V.VptError:
            bad += 1
    assert bad > 40 and ok + bad == 240


def test_corrupt_image_files_fail_cleanly(tmp_path):
    for name, loader in (("blackbody_texture.exr", load_exr_rgb), ("BN0.bmp", load_bmp_rbg)):
        blob = open(find_asset(name), "rb").read()
        p = tmp_path / ("m" + os.path.splitext(name)[1])
        bad = 0
        for m in _mutations(blob, 9, 200, header_bias=min(len(blob) - 8, 700)):
            p.write_bytes(m)
            try:
                img = loader(str(p))
                assert img.size <= 1 << 28
            except V.VptError:
                bad += 1
        assert bad > 20, name


_CDF_REF = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libcreate_cdf_ref.so")


@pytest.mark.parametrize("kind", ["sky", "random", "zero_first_row", "all_zero", "spiky"])
def test_env_tables_equal_the_reference_create_cdf_bit_for_bit(request, kind):
    """VERDICT r1 item 6 / ADVICE: the env sampling tables against the reference's OWN create_cdf arithmetic (main.cpp:681-751,
    compiled from the original project into oracle/_ref, or its outputs recorded under tests/golden/reference; its two out-of-array
    reads see 0).  Bit-exact, including the carry-over of the previous row's last element into every row y > 0 and the
    marginal_func[0] == 0 fallback rule."""
    import reference_outputs
    import ctypes as C
    from vpt_b200.scene import sky_power_table
    res = 180
    rng = np.random.RandomState(4)
    if kind == "sky": func = sky_power_table(120.0, 30.0, (1.0, 0.9, 0.8), res)
    elif kind == "random": func = rng.rand(res, res).astype(np.float32) * 3.0
    elif kind == "zero_first_row": func = rng.rand(res, res).astype(np.float32); func[0, :] = 0.0
    elif kind == "all_zero": func = np.zeros((res, res), dtype=np.float32)
    else: func = np.maximum((rng.rand(res, res) ** 8).astype(np.float32) * 100.0, np.float32(1e-12)); func[50, :] = 0.0   # (no underflow in the stand-in's sqrt(v*v))
    func = np.ascontiguousarray(func, dtype=np.float32)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))

    def reference():
        ref = C.CDLL(_CDF_REF)
        ref.vptref_create_cdf.argtypes = [C.POINTER(C.c_float)] * 5 + [C.POINTER(C.c_float), C.c_float]
        r_func = np.empty((res, res), np.float32); r_cdf = np.empty((res, res), np.float32)
        r_mf = np.empty(res, np.float32); r_mc = np.empty(res, np.float32); r_int = C.c_float(0)
        assert ref.vptref_create_cdf(fp(func), fp(r_func), fp(r_cdf), fp(r_mf), fp(r_mc), C.byref(r_int), 0.0) == 0
        return dict(func=r_func, cdf=r_cdf, marginal_func=r_mf, marginal_cdf=r_mc, integral=np.float32(r_int.value))
    R = reference_outputs.load(request, reference, live=os.path.exists(_CDF_REF), exact=("func", "cdf", "marginal_func", "marginal_cdf"))
    assert R.same("func", func)                                             # the stand-in sky reproduced the table exactly
    cdf = np.empty((res, res), np.float32); mf = np.empty(res, np.float32); mc = np.empty(res, np.float32); mint = C.c_float(0)
    assert V.lib.vpt_env_tables_compute(fp(func), res, fp(cdf), fp(mf), fp(mc), C.byref(mint)) == 0
    assert R.same("marginal_func", mf), "marginal_func"
    assert R.same("cdf", cdf), "conditional cdf"
    assert R.same("marginal_cdf", mc), "marginal cdf"
    r_int = R.want("integral")
    assert np.float32(mint.value) == r_int or (np.isnan(mint.value) and np.isnan(r_int))
    if kind in ("sky", "random"):
        assert np.all(cdf[:, -1] == 1.0) and np.all(np.diff(mc) >= 0) and abs(mc[-1] - 1.0) < 1e-5
        assert np.allclose(cdf[1:, 0] * mf[1:], func[:-1, -1] / res, rtol=1e-5)   # the carry-over is really there
