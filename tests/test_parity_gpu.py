"""GPU parity tests: the sm_100a wavefront path (through the C ABI) against
  (1) the committed golden fixtures -- outputs of the reference's own kernel (tests/golden/make_golden.py), and
  (2) the reference kernel on the same parameter block: executed live where oracle/_ref was built, else its outputs as
      recorded under tests/golden/reference (tests/reference_outputs.py).

Tolerance (stated once, used everywhere): per channel |d| <= 1e-5 + 1e-4*|ref| on >= 99.9 % of the pixels; the rest
are counted as decision-flipped pixels (chaotic estimator, SURVEY 8(c)).  In practice 0 pixels differ.
Integer outputs: display words may differ by at most 1 LSB per channel on <= 0.1 % of pixels; blue-noise state,
cost buffer and (in the octree tests) every node field are compared bit-exactly.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

import vpt_b200 as V
from vpt_b200.scene import synthetic_env
import oracle_ref
import reference_outputs

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL, ATOL, MAX_FLIPPED = 1e-4, 1e-5, 1e-3


def flipped_fraction(got, want):
    """Fraction of the pixels (rows) with a channel outside the tolerance.  A non-finite value matches only the same value:
    NaN against NaN, +Inf against +Inf, -Inf against -Inf; finite against non-finite is a flip."""
    got = np.asarray(got, dtype=np.float64); want = np.asarray(want, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        bad = np.abs(got - want) > ATOL + RTOL * np.abs(want)
    fin_g, fin_w = np.isfinite(got), np.isfinite(want)
    both = ~fin_g & ~fin_w
    bad |= (fin_g != fin_w) | (both & ~((np.isnan(got) & np.isnan(want)) | (got == want)))
    if bad.ndim > 1:
        bad = bad.reshape(bad.shape[0] * bad.shape[1] if bad.ndim == 3 else bad.shape[0], -1).any(axis=1)
    return float(bad.mean())


@pytest.fixture(scope="module")
def dragon():
    return V.Volume.load_vdb(V.find_asset("dragon.vdb"))


def make_scene(dragon, lights=None, env=None, instances=None):
    return V.Scene(instances or [dragon.instance()], env=synthetic_env(512, 256) if env is None else env, lights=lights)


def make_kp(**over):
    kp = V.default_kernel_params(); kp.environment_type = 1; kp.max_interactions = 1000
    for k, v in over.items(): setattr(kp, k, v)
    return kp


@pytest.mark.parametrize("name", ["dragon_single", "dragon_multi"])
def test_against_reference_golden(dragon, name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    meta = json.loads(str(g["meta"]))
    lights = [tuple(map(tuple, l[:2])) + (l[2],) for l in meta["lights"]] if meta["lights"] else None
    scene = make_scene(dragon, lights=lights)
    r = V.Renderer(scene, meta["W"], meta["H"], kp=make_kp(**meta["kp"]))
    assert bytes(r.cam) == g["camera"].tobytes(), "camera set-up drifted from the fixture"
    r.render(meta["passes"]); torch.cuda.synchronize()
    H, W = meta["H"], meta["W"]
    assert flipped_fraction(r.buffers.accum.cpu().numpy().reshape(H, W, 3), g["accum"]) <= MAX_FLIPPED
    assert flipped_fraction(r.buffers.depth.cpu().numpy().reshape(H, W, 1), g["depth"][..., None]) <= MAX_FLIPPED
    raw = r.buffers.raw.cpu().numpy().reshape(H, W, 4)
    assert flipped_fraction(raw[..., :3], g["raw"][..., :3]) <= MAX_FLIPPED
    assert np.mean(np.abs(raw[..., 3] - g["raw"][..., 3]) > 1e-5) <= MAX_FLIPPED          # tr: replayed depth-walk sum, see DESIGN.md
    dm = r.buffers.display.cpu().numpy().view(np.uint8).reshape(-1, 4).astype(int)
    dg = g["display"].astype(np.int32).view(np.uint8).reshape(-1, 4).astype(int)
    assert np.abs(dm - dg).max() <= 1 and np.mean(np.abs(dm - dg).max(axis=1) > 0) <= MAX_FLIPPED
    assert np.array_equal(scene.d_blue_noise.cpu().numpy(), g["blue_noise"]), "blue-noise state must be bit-exact"
    assert float(r.buffers.cost.abs().max()) == 0.0


needs_ref = pytest.mark.skipif(not oracle_ref.available(), reason="oracle/_ref (reference kernel build) not in this snapshot")


@pytest.mark.parametrize("cfg", [
    dict(W=256, H=256, passes=1, kp=dict(ray_depth=1)),                                   # BASELINE config 1 shape (HDRI env)
    dict(W=512, H=512, passes=1, kp=dict(ray_depth=1)),                                   # BASELINE config 1 resolution
    dict(W=320, H=200, passes=3, kp=dict(ray_depth=100)),                                 # config 2 parameters, ragged size
    dict(W=256, H=96, passes=2, kp=dict(ray_depth=4, volume_depth=5, phase_g1=-0.4)),     # multiple scattering via volume_depth
    dict(W=200, H=120, passes=2, kp=dict(ray_depth=2, density_mult=6.0, tr_depth=0.5, sun_mult=3.0)),
    dict(W=33, H=17, passes=2, kp=dict(ray_depth=2)),                                     # tiny / not a multiple of any tile
])
def test_live_against_reference_kernel(request, dragon, cfg):
    scene = make_scene(dragon)
    mine = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**cfg["kp"]))

    def reference():
        ref = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**cfg["kp"]), cam=mine.cam)
        orc = oracle_ref.RefOracle()
        ref.params.p_oct.value = orc.build_octree(scene.h_volumes, 1)
        scene.reset_blue_noise(); orc.render(ref, cfg["passes"])
        return dict(accum=ref.buffers.accum, depth=ref.buffers.depth, blue_noise=scene.d_blue_noise, iteration=ref.kp.iteration)
    R = reference_outputs.load(request, reference, exact=("blue_noise",))
    scene.reset_blue_noise(); mine.render(cfg["passes"]); torch.cuda.synchronize()
    assert flipped_fraction(R.pick("accum", mine.buffers.accum), R.want("accum")) <= MAX_FLIPPED
    assert flipped_fraction(R.pick("depth", mine.buffers.depth)[:, None], R.want("depth")[:, None]) <= MAX_FLIPPED
    assert R.same("blue_noise", scene.d_blue_noise)
    assert mine.kp.iteration == int(R.want("iteration")) == cfg["passes"]


def test_point_lights_and_sphere_against_reference(request, dragon):
    lights = [((9.0, 6.0, 2.0), (1.0, 0.8, 0.6), 40.0), ((-2.0, 3.0, 8.0), (0.5, 0.7, 1.0), 25.0), ((4.0, 9.0, 3.0), (1.0, 1.0, 1.0), 10.0)]
    scene = make_scene(dragon, lights=lights)
    # put the reference sphere where rays actually hit it: next to the dragon
    sp = scene.h_sphere; sp.center = V.f3(4.0, 6.5, 3.0); sp.radius = 1.2; sp.roughness = 0.7; sp.color = V.f3(0.8, 0.6, 0.3)
    scene.d_sphere.copy_(torch.frombuffer(bytearray(bytes(sp)), dtype=torch.uint8))
    kw = dict(ray_depth=3, volume_depth=2)
    mine = V.Renderer(scene, 256, 160, kp=make_kp(**kw))

    def reference():
        ref = V.Renderer(scene, 256, 160, kp=make_kp(**kw), cam=mine.cam)
        scene.reset_blue_noise(); oracle_ref.RefOracle().render(ref, 2)
        return dict(accum=ref.buffers.accum, mean=float(ref.buffers.accum.mean()))
    R = reference_outputs.load(request, reference)
    scene.reset_blue_noise(); mine.render(2); torch.cuda.synchronize()
    assert float(R.want("mean")) > 0
    assert flipped_fraction(R.pick("accum", mine.buffers.accum), R.want("accum")) <= MAX_FLIPPED


def octree_arrays(tree):
    """An octree read with vpt_octree_read (node number -> OCTNode) as flat arrays; the host-built root (node 0) carries
    no voxel size, depth or child flag."""
    paths = sorted(tree)
    n = [tree[p].num_volumes for p in paths]
    return dict(paths=np.array(paths, dtype=np.int32), num_volumes=np.array(n, dtype=np.int32),
                vol_indices=np.array([v for p in paths for v in tree[p].vol_indices[:tree[p].num_volumes]], dtype=np.int32),
                bbox=np.array([np.frombuffer(bytes(tree[p].bbox), dtype=np.float32) for p in paths], dtype=np.float32),
                extinction=np.array([(tree[p].max_extinction, tree[p].min_extinction) for p in paths], dtype=np.float32),
                node=np.array([(tree[p].voxel_size, tree[p].depth, tree[p].has_children) if p else (0, 0, 0) for p in paths], dtype=np.float32))


OCTREE_ARRAYS = ("paths", "num_volumes", "vol_indices", "bbox", "extinction", "node")


def assert_octree_equals_reference(R, tree):
    for k, a in octree_arrays(tree).items():
        assert R.same(k, a), k


def test_instanced_scene_and_octree_bit_exact(request, dragon):
    """8 rotated / scaled instances: my parallel octree build vs the reference's device-heap recursion, node by
    node (bbox, volume lists, extinctions bit-exact), then the render on both octrees."""
    rng = np.random.RandomState(7)
    inst = []
    for i in range(8):
        q = rng.randn(4); q /= np.linalg.norm(q)
        inst.append(dragon.instance(pos=tuple(rng.uniform(-6, 6, 3)), quat=tuple(q), scale=float(rng.uniform(0.6, 1.4))))
    scene = make_scene(dragon, instances=inst)
    kw = dict(ray_depth=2)
    mine = V.Renderer(scene, 256, 128, kp=make_kp(**kw))

    def reference():
        orc = oracle_ref.RefOracle()
        ref_root = orc.build_octree(scene.h_volumes, len(inst))
        ref = V.Renderer(scene, 256, 128, kp=make_kp(**kw), cam=mine.cam)
        ref.params.p_oct.value = ref_root
        scene.reset_blue_noise(); orc.render(ref, 2)
        return dict(octree_arrays(read_tree(ref_root)), accum=ref.buffers.accum)
    R = reference_outputs.load(request, reference, exact=OCTREE_ARRAYS)
    mine_t = read_tree(scene.d_oct_root)
    assert len(mine_t) > 9
    assert_octree_equals_reference(R, mine_t)
    scene.reset_blue_noise(); mine.render(2); torch.cuda.synchronize()
    assert flipped_fraction(R.pick("accum", mine.buffers.accum), R.want("accum")) <= MAX_FLIPPED


def read_tree(root):
    nodes = (V.OCTNode * 585)(); ex = (C.c_int * 585)()
    V._native.check(V.lib.vpt_octree_read(root, nodes, ex), None, "vpt_octree_read")
    return {j: nodes[j] for j in range(585) if ex[j]}


def test_instance_transform_matches_reference_mat4_algebra(request, dragon):
    from vpt_b200.scene import instance_xform
    rng = np.random.RandomState(3)
    base = np.array([[dragon.rec.xform[a][b] for b in range(4)] for a in range(4)], dtype=np.float32)
    base[0][3], base[1][3], base[2][3] = 0.3, -0.2, 0.1
    args = []
    for _ in range(20):
        q = rng.randn(4).astype(np.float32); pos = rng.uniform(-50, 50, 3).astype(np.float32); s = np.float32(rng.uniform(0.2, 3))
        args.append((pos, q, s))

    def reference():
        orc = oracle_ref.RefOracle()
        xf = []
        for pos, q, s in args:
            out = (C.c_float * 16)()
            orc.lib.vptref_instance_xform(V._native.fvec(base.reshape(-1)), V._native.fvec(pos), V._native.fvec(q), float(s), out)
            xf.append(np.array(list(out), dtype=np.float32).reshape(4, 4))
        return dict(xforms=np.stack(xf))
    R = reference_outputs.load(request, reference)
    assert R.same("xforms", np.stack([instance_xform(base, pos, q, s) for pos, q, s in args]).astype(np.float32))


def _big_asset(name):
    return V.find_asset(name)


@needs_ref
@pytest.mark.skipif(_big_asset("fireball.vdb") is None, reason="fireball.vdb not staged (oracle/_ref/assets)")
def test_fireball_emission_against_reference():
    """BASELINE config 3 parameters at reduced size: emission walk + blackbody LUT, heat grid addressed with the
    density grid's bounds (quirk Q8), sigma_max = 12.47, multiple scattering through volume_depth."""
    vol = V.Volume.load_vdb(_big_asset("fireball.vdb"))
    assert vol.rec.vdb_info.has_emission == 1 and abs(vol.rec.vdb_info.max_density - 12.4696) < 1e-3
    scene = V.Scene([vol.instance()], env=synthetic_env(512, 256))
    kw = dict(ray_depth=2, volume_depth=6, emission_scale=1.0, emission_pivot=1.0)
    mine = V.Renderer(scene, 320, 180, kp=make_kp(**kw)); ref = V.Renderer(scene, 320, 180, kp=make_kp(**kw), cam=mine.cam)
    orc = oracle_ref.RefOracle()
    ref.params.p_oct.value = orc.build_octree(scene.h_volumes, 1)
    scene.reset_blue_noise(); orc.render(ref, 2)
    scene.reset_blue_noise(); mine.render(2); torch.cuda.synchronize()
    assert float(ref.buffers.accum.mean()) > 1e-3
    assert flipped_fraction(mine.buffers.accum.cpu().numpy(), ref.buffers.accum.cpu().numpy()) <= MAX_FLIPPED
    assert flipped_fraction(mine.buffers.depth.cpu().numpy()[:, None], ref.buffers.depth.cpu().numpy()[:, None]) <= MAX_FLIPPED


@needs_ref
@pytest.mark.skipif(_big_asset("colored_smoke.vdb") is None, reason="colored_smoke.vdb not staged (oracle/_ref/assets)")
def test_colored_smoke_against_reference():
    vol = V.Volume.load_vdb(_big_asset("colored_smoke.vdb"))
    assert vol.rec.vdb_info.has_color == 1
    scene = V.Scene([vol.instance()], env=synthetic_env(512, 256))
    kw = dict(ray_depth=2, volume_depth=4, density_mult=4.0)
    mine = V.Renderer(scene, 320, 180, kp=make_kp(**kw)); ref = V.Renderer(scene, 320, 180, kp=make_kp(**kw), cam=mine.cam)
    orc = oracle_ref.RefOracle()
    scene.reset_blue_noise(); orc.render(ref, 2)
    scene.reset_blue_noise(); mine.render(2); torch.cuda.synchronize()
    a = ref.buffers.accum.cpu().numpy()
    assert np.abs(a[:, 0] - a[:, 2]).max() > 1e-3, "the colour grid should tint the radiance"
    assert flipped_fraction(mine.buffers.accum.cpu().numpy(), a) <= MAX_FLIPPED


def test_many_instances_against_reference(request, dragon):
    """BASELINE config 5 shape (instanced dragon through the octree's leaf lists) at the size the oracle finishes quickly."""
    rng = np.random.RandomState(11)
    inst = []
    for i in range(120):
        q = rng.randn(4); q /= np.linalg.norm(q)
        inst.append(dragon.instance(pos=tuple(rng.uniform(-25, 25, 3)), quat=tuple(q), scale=float(rng.uniform(0.7, 1.3))))
    scene = make_scene(dragon, instances=inst)
    kw = dict(ray_depth=2)
    mine = V.Renderer(scene, 256, 144, kp=make_kp(**kw))

    def reference():
        ref = V.Renderer(scene, 256, 144, kp=make_kp(**kw), cam=mine.cam)
        scene.reset_blue_noise(); oracle_ref.RefOracle().render(ref, 1)
        return dict(accum=ref.buffers.accum, mean=float(ref.buffers.accum.mean()))
    R = reference_outputs.load(request, reference)
    scene.reset_blue_noise(); mine.render(1); torch.cuda.synchronize()
    assert float(R.want("mean")) > 1e-4
    assert flipped_fraction(R.pick("accum", mine.buffers.accum), R.want("accum")) <= MAX_FLIPPED


# ---- the sky look-up tables: the reference's own precompute (live only) and this library's ----------------------------
SKY_TABLES = ("reference", "own")
_OWN_SKY = {}


def sky_tables(scene, source, luminance=0):
    """Hand `scene` the four sky look-up textures of one precompute, default options otherwise: "reference" (the reference's
    own atmosphere::init, oracle/_ref) or "own" (this library's).  Both kernels then read the same textures."""
    if source == "reference":
        oracle_ref.RefOracle().atmosphere_init(scene.atmos, luminance=luminance)
    else:
        if luminance not in _OWN_SKY:
            _OWN_SKY[luminance] = V.Atmosphere(luminance=luminance)
        _OWN_SKY[luminance].apply(scene.atmos)


def sky_sources(R):
    """The table sources a test compares on: both where the reference runs live; its recorded frames on this library's tables otherwise."""
    return SKY_TABLES if R.live else ("own",)


def live_only_keys(*names):
    return tuple(f"reference.{n}" for n in names)


has_ref_atmo = os.path.exists(os.path.join(oracle_ref.REF_DIR, "atmo", "atmosphere_kernels.ptx"))


@pytest.mark.parametrize("cfg", [
    dict(W=512, H=512, passes=1, elevation=30.0, kp=dict(ray_depth=1)),                          # BASELINE config 1 literally (env type 0)
    dict(W=320, H=200, passes=3, elevation=4.0, kp=dict(ray_depth=20, sky_mult=2.0)),            # low sun, multi-pass, deeper paths
    dict(W=256, H=128, passes=2, elevation=60.0, aperture=0.2, kp=dict(ray_depth=3)),            # thin lens (env_pos != cam origin)
    dict(W=256, H=128, passes=1, elevation=45.0, luminance=1, kp=dict(ray_depth=2)),             # APPROXIMATE luminance mode
    dict(W=256, H=128, passes=1, elevation=45.0, luminance=2, kp=dict(ray_depth=2)),             # PRECOMPUTED luminance mode
])
def test_precomputed_sky_environment_against_reference(request, dragon, cfg):
    """environment_type == 0: both kernels read the SAME look-up textures, produced by the reference's own precompute and by
    this library's."""
    scene = make_scene(dragon)
    kw = dict(environment_type=0, elevation=cfg["elevation"], **cfg["kp"])
    cam = scene.frame_camera(cfg["W"], cfg["H"], aperture=cfg.get("aperture", 0.0))
    lum = cfg.get("luminance", 0)

    def reference():
        out = {}
        for src in SKY_TABLES:
            sky_tables(scene, src, lum)
            ref = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**kw), cam=cam)
            scene.reset_blue_noise(); oracle_ref.RefOracle().render(ref, cfg["passes"])
            a = ref.buffers.accum.cpu().numpy()
            out.update({f"{src}.accum": a, f"{src}.depth": ref.buffers.depth,
                        f"{src}.stats": np.array([np.isfinite(a).all(), a.mean(), a.std()], dtype=np.float64)})
        return out
    R = reference_outputs.load(request, reference, live=oracle_ref.available() and has_ref_atmo, live_only=live_only_keys("accum", "depth", "stats"))
    for src in sky_sources(R):
        sky_tables(scene, src, lum)
        mine = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**kw), cam=cam)
        scene.reset_blue_noise(); mine.render(cfg["passes"]); torch.cuda.synchronize()
        want = R.want(f"{src}.accum"); got = R.pick(f"{src}.accum", mine.buffers.accum)
        finite, mean, std = R.want(f"{src}.stats")
        print(f"sky cfg {cfg}, {src} tables: reference mean {mean:.6g}, ours {float(mine.buffers.accum.mean()):.6g}")
        assert finite
        if not lum:
            assert mean > 1e-3 and std > 0, "the sky must actually light the frame"
        assert flipped_fraction(got, want) <= MAX_FLIPPED
        assert flipped_fraction(R.pick(f"{src}.depth", mine.buffers.depth)[:, None], R.want(f"{src}.depth")[:, None]) <= MAX_FLIPPED


def _sky_power_table(res=180, sun_az=2.0, sun_el=1.0):
    """A smooth, strictly positive stand-in for the sky's luminous power over (azimuth, elevation): what the reference's
    create_cdf tabulates from its host-side sky model.  Both kernels sample from the same tables."""
    el = (np.arange(res, dtype=np.float32) / (res - 1) * np.pi)[:, None]
    az = (np.arange(res, dtype=np.float32) / (res - 1) * 2 * np.pi)[None, :]
    return (0.05 + np.sin(el) * (1.2 + np.cos(az - sun_az)) * (0.3 + np.exp(-4.0 * (el - sun_el) ** 2))).astype(np.float32)


@pytest.mark.parametrize("cfg", [
    dict(W=256, H=160, passes=2, env=1, kp=dict(ray_depth=8)),                                    # HDRI sky estimator (uniform sphere + HG MIS)
    dict(W=256, H=160, passes=2, env=1, kp=dict(ray_depth=100, phase_g1=0.6, density_mult=3.0)),  # cfg 2's "true multiple scattering" variant
    dict(W=200, H=120, passes=2, env=0, kp=dict(ray_depth=6)),                                    # tabulated sky sampling (env-CDF MIS)
    dict(W=200, H=120, passes=1, env=1, lights=True, kp=dict(ray_depth=5, sky_mult=0.0)),         # point lights, sky class switched off
    dict(W=160, H=100, passes=1, env=1, sphere=True, aperture=0.15, kp=dict(ray_depth=4)),        # sphere in the way + thin lens
])
def test_volumetric_path_integrator_against_reference(request, dragon, cfg):
    """Kernel_params.integrator = 1 (reference vol_integrator): light-class selection, NEE per scatter, sky MIS, sky tail."""
    lights = [((9.0, 6.0, 2.0), (1.0, 0.8, 0.6), 40.0), ((-2.0, 3.0, 8.0), (0.5, 0.7, 1.0), 25.0)] if cfg.get("lights") else None
    scene = make_scene(dragon, lights=lights)
    if cfg.get("sphere"):
        sp = scene.h_sphere; sp.center = V.f3(6.0, 6.0, 5.0); sp.radius = 1.0
        scene.d_sphere.copy_(torch.frombuffer(bytearray(bytes(sp)), dtype=torch.uint8))
    tables = V.EnvTables(_sky_power_table())
    kw = dict(integrator=1, environment_type=cfg["env"], **cfg["kp"])
    cam = scene.frame_camera(cfg["W"], cfg["H"], aperture=cfg.get("aperture", 0.0))

    def reference():
        out = {}
        for src in SKY_TABLES:
            sky_tables(scene, src)
            ref = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**kw), cam=cam)
            tables.apply(ref.kp)
            scene.reset_blue_noise(); oracle_ref.RefOracle().render(ref, cfg["passes"])
            a = ref.buffers.accum.cpu().numpy()
            out.update({f"{src}.accum": a, f"{src}.depth": ref.buffers.depth, f"{src}.tr": ref.buffers.raw.reshape(-1, 4)[:, 3],
                        f"{src}.stats": np.array([np.isfinite(a).all(), a.mean()], dtype=np.float64)})
        return out
    R = reference_outputs.load(request, reference, live=oracle_ref.available() and has_ref_atmo, live_only=live_only_keys("accum", "depth", "tr", "stats"))
    for src in sky_sources(R):
        sky_tables(scene, src)
        mine = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**kw), cam=cam)
        tables.apply(mine.kp)
        scene.reset_blue_noise(); mine.render(cfg["passes"]); torch.cuda.synchronize()
        want = R.want(f"{src}.accum"); got = R.pick(f"{src}.accum", mine.buffers.accum)
        frac = flipped_fraction(got, want)
        dfrac = flipped_fraction(R.pick(f"{src}.depth", mine.buffers.depth)[:, None], R.want(f"{src}.depth")[:, None])
        finite, mean = R.want(f"{src}.stats")
        print(f"vol cfg {cfg}, {src} tables: ref mean {mean:.6g} ours {float(mine.buffers.accum.mean()):.6g} flipped {frac:.3g} depth-flipped {dfrac:.3g}")
        assert finite and mean > 1e-3
        # Measured: no pixel outside tolerance in any configuration.  With the tabulated sky (env 0) the sky model is also evaluated
        # INSIDE the path, where the reference build contracts three ill-conditioned sums differently from its end-of-path call sites;
        # vpt_atmosphere.cuh mirrors both orders (kInPath).  Before that 0.25 % of the pixels were off by up to 1 % (DESIGN.md section 5).
        limit = 1e-4 if cfg["env"] == 0 else 0.0
        assert frac <= limit and dfrac == 0.0
        tr = R.pick(f"{src}.tr", mine.buffers.raw.reshape(-1, 4)[:, 3])
        assert np.mean(np.abs(tr - R.want(f"{src}.tr")) > 1e-5) <= MAX_FLIPPED
    tables.destroy()


def test_fused_passes_equal_single_passes_bitwise_full_hd(dragon):
    scene = make_scene(dragon)
    a = V.Renderer(scene, 1920, 1080, kp=make_kp(ray_depth=100), options=dict(passes_per_chunk=4))
    b = V.Renderer(scene, 1920, 1080, kp=make_kp(ray_depth=100), cam=a.cam)
    scene.reset_blue_noise(); a.render(6)                                   # chunks of 4 + 2
    bn_a = scene.d_blue_noise.clone()
    scene.reset_blue_noise()
    for _ in range(6): b.render_pass()
    torch.cuda.synchronize()
    for name in ("accum", "depth", "cost", "raw", "display"):
        assert torch.equal(getattr(a.buffers, name), getattr(b.buffers, name)), name
    assert torch.equal(bn_a, scene.d_blue_noise)
    assert float(a.buffers.accum.mean()) > 1e-3 and bool(torch.isfinite(a.buffers.accum).all())


def test_lean_and_generic_trace_kernels_agree_bitwise(dragon):
    """The host picks a trace-kernel instantiation without multi-volume / emission / point-light code when none is in play."""
    scene = make_scene(dragon)
    a = V.Renderer(scene, 640, 360, kp=make_kp(ray_depth=100))
    b = V.Renderer(scene, 640, 360, kp=make_kp(ray_depth=100), options={"generic_kernel": 1})
    scene.reset_blue_noise(); a.render(4); torch.cuda.synchronize()
    scene.reset_blue_noise(); b.render(4); torch.cuda.synchronize()
    for name in ("accum", "depth", "raw", "display"):
        assert torch.equal(getattr(a.buffers, name), getattr(b.buffers, name)), name


def test_partition_invariance_and_determinism(dragon):
    """Rendering the frame as 4 interleaved-stripe shards and un-permuting reproduces the single-rank frame
    bit for bit (global pixel index keys the RNG), whatever the scheduling options."""
    W, H = 640, 360
    scene = make_scene(dragon)
    one = V.Renderer(scene, W, H, kp=make_kp(ray_depth=2))
    scene.reset_blue_noise(); one.render(3); torch.cuda.synchronize()
    parts = []
    for rank in range(4):
        r = V.Renderer(scene, W, H, kp=make_kp(ray_depth=2), cam=one.cam, rank=rank, n_ranks=4, stripe_rows=8,
                       options=dict(sched_min_lanes=(1, 8, 16, 32)[rank], passes_per_chunk=rank + 1))
        scene.reset_blue_noise(); r.render(3); parts.append(r)
    torch.cuda.synchronize()
    gathered = torch.cat([p.buffers.accum for p in parts], dim=0)
    full = parts[0].unpermute(gathered, 3)
    assert torch.equal(full, one.buffers.accum)


def test_iteration_limit_and_render_flag_semantics(dragon):
    scene = make_scene(dragon)
    r = V.Renderer(scene, 128, 64, kp=make_kp(ray_depth=1, max_interactions=2))
    r.render(2); torch.cuda.synchronize(); acc2 = r.buffers.accum.clone()
    r.render(3); torch.cuda.synchronize()                                    # iteration >= max_interactions: re-tonemap only
    assert torch.equal(acc2, r.buffers.accum)
    r2 = V.Renderer(scene, 128, 64, kp=make_kp(ray_depth=1, render=0))
    r2.render_pass(); torch.cuda.synchronize()
    assert torch.equal(r2.buffers.accum, torch.ones_like(r2.buffers.accum))  # WHITE when render == false (:2248, :2278)


def test_unsupported_configurations_fail_loudly(dragon):
    scene = make_scene(dragon)
    r = V.Renderer(scene, 64, 64, kp=make_kp(integrator=1, environment_type=0))   # no sampling tables in Kernel_params
    with pytest.raises(V.VptError, match="sampling tables"):
        r.render_pass()
    scene.atmos.transmittance_texture = 0                                   # sky environment without its look-up textures
    r = V.Renderer(scene, 64, 64, kp=make_kp(environment_type=0))
    with pytest.raises(V.VptError, match="atmosphere"):
        r.render_pass()


def test_ins_scene_file_end_to_end_against_reference(request, tmp_path):
    """SURVEY 8(f) N4: a `.ins` file is read by the library, instanced with the reference's transform algebra, rendered."""
    from vpt_b200.scene import scene_from_ins
    ins = tmp_path / "three.ins"
    ins.write_text("1\ndragon.vdb\n3\n0 0 0 0 0 0 1 1\n9 1 -2 0 0.3826834 0 0.9238795 0.8\n-6 2 5 0.2588190 0 0 0.9659258 1.3\n")
    scene = scene_from_ins(str(ins), env=synthetic_env(512, 256), resolve=V.find_asset)
    assert len(scene.instances) == 3
    kw = dict(ray_depth=3, volume_depth=2)
    mine = V.Renderer(scene, 320, 200, kp=make_kp(**kw))

    def reference():
        ref = V.Renderer(scene, 320, 200, kp=make_kp(**kw), cam=mine.cam)
        orc = oracle_ref.RefOracle()
        ref.params.p_oct.value = orc.build_octree(scene.h_volumes, 3)
        scene.reset_blue_noise(); orc.render(ref, 2)
        return dict(accum=ref.buffers.accum, mean=float(ref.buffers.accum.mean()))
    R = reference_outputs.load(request, reference)
    scene.reset_blue_noise(); mine.render(2); torch.cuda.synchronize()
    assert float(R.want("mean")) > 0
    assert flipped_fraction(R.pick("accum", mine.buffers.accum), R.want("accum")) <= MAX_FLIPPED
