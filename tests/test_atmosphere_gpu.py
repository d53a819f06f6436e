"""Bruneton sky precompute (SURVEY 8(f) row N2): this library's own tables and parameter block against the reference's
atmosphere::init (compiled unmodified into oracle/_ref), and the sky-lit render paths running on the library's own tables --
no reference code involved in producing their inputs.

Tables: compared texel for texel.  The reference's precompute indexes its scattering buffers one row / slice past the end for
coordinates that reach 1 (atmosphere_kernels.cu:366-372) and reads whatever memory follows (zeros in the oracle harness's padded
slab); this build clamps.  Texels whose look-ups touch that rim therefore differ BY CONSTRUCTION; the test reports how many and
requires the rest (the interior) to agree within 2e-3 relative (fp32 quadratures of 50..500 steps, fast-math on both sides).
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import vpt_b200 as V
from vpt_b200.scene import synthetic_env
import oracle_ref
import reference_outputs
from test_parity_gpu import flipped_fraction, make_kp, make_scene, MAX_FLIPPED, _sky_power_table

pytestmark = pytest.mark.gpu
has_atmo = os.path.exists(os.path.join(oracle_ref.REF_DIR, "atmo", "atmosphere_kernels.ptx"))


@pytest.fixture(scope="module")
def dragon():
    return V.Volume.load_vdb(V.find_asset("dragon.vdb"))


@pytest.fixture(scope="module")
def mine_default():
    return V.Atmosphere()


def rel_err(a, b, floor):
    return np.abs(a - b) / np.maximum(np.abs(b), floor)


@pytest.mark.parametrize("opts", [dict(), dict(use_constant_solar_spectrum=False, use_ozone=False), dict(luminance=1, white_balance=False, exposure=2.5)])
def test_parameter_block_equals_reference(request, opts):
    """Every scalar of AtmosphereParameters the render path reads by value (bytes 0..351), bit for bit."""
    a = V.Atmosphere(**opts)

    def flat(p):
        """every named scalar the render path reads by value, padding excluded (the reference leaves its padding uninitialised)"""
        out = []
        for name, _ in V.AtmosphereParameters._fields_:
            if name.startswith("_") or name in ("scratch_buffers", "transmittance_texture", "scattering_texture", "irradiance_texture", "single_mie_scattering_texture"): continue
            v = getattr(p, name)
            if name.endswith("_density"):
                for li in range(2):
                    l = v.layers[li]
                    out += [(f"{name}.layers[{li}].{k}", np.float32(getattr(l, k))) for k in ("width", "exp_term", "exp_scale", "linear_term", "const_term")]
            elif hasattr(v, "x"): out += [(f"{name}.{k}", np.float32(getattr(v, k))) for k in "xyz"]
            else: out.append((name, v))
        return out

    def reference():
        ref = V.AtmosphereParameters()
        oracle_ref.RefOracle().atmosphere_init(ref, use_constant_solar_spectrum=opts.get("use_constant_solar_spectrum", True), use_ozone=opts.get("use_ozone", True),
                                               luminance=opts.get("luminance", 0), white_balance=opts.get("white_balance", True), exposure=opts.get("exposure", 1.0))
        return dict(values=np.array([v for _, v in flat(ref)], dtype=np.float64))
    R = reference_outputs.load(request, reference, live=has_atmo and oracle_ref.available())
    fa, fr = flat(a.params), R.want("values")
    diff = [(n, x, y) for (n, x), y in zip(fa, fr) if not (x == y)]
    for d in diff: print("differs:", d)
    assert len(fa) > 50 and len(fa) == len(fr) and not diff
    a.destroy()


TABLES = ("transmittance", "single_mie", "irradiance", "scattering")


def test_tables_against_reference_precompute(request, mine_default):
    def reference():
        ref = V.AtmosphereParameters()
        oracle_ref.RefOracle().atmosphere_init(ref)
        T_ref = V.read_atmosphere_tables(ref)
        return dict({name: T_ref[name][..., :3] for name in TABLES}, absmax=np.array([np.abs(T_ref[name][..., :3]).max() for name in TABLES], dtype=np.float64))
    R = reference_outputs.load(request, reference, live=has_atmo and oracle_ref.available())
    T = V.read_atmosphere_tables(mine_default.params)
    report = {}
    for name, bmax in zip(TABLES, R.want("absmax")):
        a, b = R.pick(name, T[name][..., :3]).astype(np.float64), R.want(name).astype(np.float64)
        floor = 1e-6 * max(bmax, 1e-30)
        e = rel_err(a, b, floor)
        bad = e > 2e-3
        report[name] = (float(np.median(e)), float(np.quantile(e, 0.999)), float(bad.mean()), float(np.abs(b).max()))
        print(f"{name:14s}: median rel err {report[name][0]:.3g}, 99.9 % quantile {report[name][1]:.3g}, texels off by > 2e-3: {100 * report[name][2]:.3f} %, max |ref| {report[name][3]:.3g}")
    # first-order tables have no look-up into a scattering table: everything must agree
    assert report["transmittance"][2] == 0.0 and report["single_mie"][2] <= 1e-4
    # later orders: interior agrees, the rim (look-ups the reference takes beyond its buffers) is reported above
    assert report["scattering"][2] <= 0.05 and report["irradiance"][2] <= 0.05
    assert np.isfinite(T["scattering"]).all() and float(np.abs(T["scattering"]).max()) > 0


@pytest.mark.parametrize("cfg", [
    dict(W=512, H=512, passes=1, elevation=30.0, kp=dict(ray_depth=1)),                          # BASELINE configs[0] literally (environment_type 0)
    dict(W=320, H=200, passes=2, elevation=4.0, kp=dict(ray_depth=20, sky_mult=2.0)),
])
def test_sky_environment_on_own_tables_against_reference_kernel(request, dragon, mine_default, cfg):
    """environment_type == 0 with the library's OWN tables handed to both kernels: per-seed parity, no reference precompute anywhere."""
    scene = make_scene(dragon)
    mine_default.apply(scene.atmos)
    kw = dict(environment_type=0, elevation=cfg["elevation"], **cfg["kp"])
    mine = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**kw))

    def reference():
        ref = V.Renderer(scene, cfg["W"], cfg["H"], kp=make_kp(**kw), cam=mine.cam)
        orc = oracle_ref.RefOracle()
        ref.params.p_oct.value = orc.build_octree(scene.h_volumes, 1)
        scene.reset_blue_noise(); orc.render(ref, cfg["passes"])
        return dict(accum=ref.buffers.accum, mean=float(ref.buffers.accum.mean()))
    R = reference_outputs.load(request, reference)
    scene.reset_blue_noise(); mine.render(cfg["passes"]); torch.cuda.synchronize()
    want = R.want("accum"); got = R.pick("accum", mine.buffers.accum)
    print(f"own-table sky {cfg}: ref mean {float(R.want('mean')):.6g}, flipped {flipped_fraction(got, want):.3g}")
    assert float(R.want("mean")) > 1e-3 and flipped_fraction(got, want) <= MAX_FLIPPED


def test_sky_render_own_tables_vs_reference_tables(request, dragon, mine_default):
    """The whole chain: this library's precompute + render against the reference's precompute + its kernel.  The tables differ in the
    last digits (and at the rim), so this is a radiometric comparison: mean radiance within 1 %, 99 % of the pixels within 2 %."""
    scene_a = make_scene(dragon)
    mine_default.apply(scene_a.atmos)
    kw = dict(environment_type=0, elevation=25.0, ray_depth=2)
    a = V.Renderer(scene_a, 320, 200, kp=make_kp(**kw))

    def reference():
        scene_b = make_scene(dragon)
        orc = oracle_ref.RefOracle(); orc.atmosphere_init(scene_b.atmos)
        b = V.Renderer(scene_b, 320, 200, kp=make_kp(**kw), cam=a.cam)
        b.params.p_oct.value = orc.build_octree(scene_b.h_volumes, 1)
        scene_b.reset_blue_noise(); orc.render(b, 2); torch.cuda.synchronize()
        return dict(accum=b.buffers.accum, mean=float(b.buffers.accum.double().mean()))
    R = reference_outputs.load(request, reference, live=has_atmo and oracle_ref.available())
    scene_a.reset_blue_noise(); a.render(2); torch.cuda.synchronize()
    x_mean = float(a.buffers.accum.double().mean()); y_mean = float(R.want("mean"))
    x = R.pick("accum", a.buffers.accum).astype(np.float64); y = R.want("accum").astype(np.float64)
    rel = np.abs(x - y).max(axis=1) / np.maximum(np.abs(y).max(axis=1), 1e-4)
    print(f"own precompute vs reference precompute: mean {x_mean:.6g} vs {y_mean:.6g}, 99 % quantile of per-pixel rel diff {np.quantile(rel, 0.99):.3g}")
    assert abs(x_mean - y_mean) <= 0.01 * y_mean and np.quantile(rel, 0.99) <= 0.02


def test_volumetric_path_integrator_runs_on_own_tables(dragon, mine_default):
    """integrator = 1 with environment_type 0 needs the sky tables inside the path and the env sampling tables: all library-built."""
    scene = make_scene(dragon)
    mine_default.apply(scene.atmos)
    tables = V.EnvTables(V.sky_power_table(120.0, 30.0, (1.0, 1.0, 1.0), 180))
    r = V.Renderer(scene, 200, 120, kp=make_kp(integrator=1, environment_type=0, ray_depth=6))
    tables.apply(r.kp)
    r.render(2); torch.cuda.synchronize()
    acc = r.buffers.accum.cpu().numpy()
    assert np.isfinite(acc).all() and float(acc.mean()) > 1e-3
    tables.destroy()
