"""The per-pixel tail of the render pass (reference render_kernel.cu:2262-2316: NaN / Inf guard, running mean, ACES, display,
raw, cost, the `render` flag, `max_interactions`, viz_dof, exposure_scale) against the reference kernel, on the states the
reference application actually hands it:

  * stale buffers: every edit in the reference UI sets iteration = 0 and leaves accum / depth / cost holding the previous
    frame (main.cpp:1667-1780).  At iteration 0 a non-finite sample is replaced by that stale pixel (:2263), not by zero;
  * non-finite samples: Inf / NaN environment texels, and a zero channel of `extinction` (albedo * Cd * dc / extinction,
    :1674, is then Inf or NaN);
  * progressive hand-off between the two implementations, iteration limits, the curand offset wrap at iteration 2^20, and
    the viz_dof / exposure display path.

Every case compares accum, depth and raw.xyz within the suite's tolerance (test_parity_gpu.py), raw.w like the goldens
test, display within 1 LSB, and cost and the blue-noise state bit for bit, through level (B) (Renderer: fused, single-pass
and a 3-shard partition on one GPU) and level (A) (the volume_rt_kernel cubin).  Frames of 320x200 are recorded as a
384-pixel sample (tests/reference_outputs.py), so full-frame scalars are recorded alongside: the number of pixels whose accum
still equals the stale value bit for bit, the number of non-finite pixels per buffer and the sum of the finite accum entries.

Why these inputs cannot hang a kernel.  Non-finite values enter only through environment texels and through the
throughput (extinction.y / .z; extinction.x, which scales the tracking step length at :1177 and :1331, stays 1).  No loop
exit depends on either:
  * the bounce loops (ray_depth, volume_depth) and the point-light loop count down integer budgets;
  * delta, ratio and emission tracking end on `t` against the box exit distance; `t` grows by -log(1 - xi) / sigma_max *
    tr_depth / extinction.x with finite densities, tr_depth and extinction.x, so it is finite and strictly increasing;
  * octree hops compare positions and directions; directions change only through hg_sample (a finite draw and phase_g1 =
    0, never -1) and the sphere bounce, neither of which reads the throughput;
  * the thin-lens rejection loop reads only the RNG.
The throughput itself only feeds `isBlack(beta)` (Inf or NaN is not black: the path continues until its budget runs out,
in both kernels) and `length(beta) > 0.9999` in the path integrator's env_pos choice (False for NaN, in both kernels).
Environment texels are read at path ends and in the sky estimator's `!isBlack(Li)` branch, never by a loop condition.
"""
import numpy as np
import pytest
import torch

import vpt_b200 as V
from vpt_b200.scene import synthetic_env, texture_env
import oracle_ref
import reference_outputs
from test_parity_gpu import flipped_fraction, make_kp, make_scene, MAX_FLIPPED, _sky_power_table, sky_tables
from test_scale_gpu import level_a_launcher

pytestmark = pytest.mark.gpu
BUFFERS = ("accum", "depth", "cost", "raw", "display")
ELEM = dict(accum=3, depth=1, cost=3, raw=4, display=1)


@pytest.fixture(scope="module")
def dragon():
    return V.Volume.load_vdb(V.find_asset("dragon.vdb"))


# ---- inputs ------------------------------------------------------------------------------------------------------------
def camera_env_coords(cam, W, H):
    """(u, v) environment coordinates of every pixel's pinhole camera ray, as the kernels look the HDRI up (atan2 / acos)."""
    g = lambda f: np.array([f.x, f.y, f.z], dtype=np.float64)
    x = (np.arange(W) + 0.5) / W; y = (np.arange(H) + 0.5) / H
    d = g(cam.lower_left_corner)[None, None] + x[None, :, None] * g(cam.horizontal) + y[:, None, None] * g(cam.vertical) - g(cam.origin)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    return np.arctan2(d[..., 2], d[..., 0]) / (2 * np.pi) + 0.5, np.arccos(np.clip(d[..., 1], -1, 1)) / np.pi


def non_finite_env(cam, W, H, ew=512, eh=256):
    """The synthetic HDRI with +Inf in the red channel over a band of rows that covers the middle 40 % of the elevations the
    frame sees, and a smaller NaN patch in green above it."""
    env = synthetic_env(ew, eh)
    u, v = camera_env_coords(cam, W, H)
    lo, hi = float(v.min()), float(v.max())
    span = hi - lo
    env[int(np.floor((lo + 0.3 * span) * eh)):int(np.ceil((lo + 0.7 * span) * eh)), :, 0] = np.inf
    uc = float(np.median(u))
    r0, r1 = int(np.floor((lo + 0.08 * span) * eh)), int(np.ceil((lo + 0.2 * span) * eh))
    c0, c1 = int(np.floor((uc - 0.02) * ew)), int(np.ceil((uc + 0.02) * ew))
    env[r0:r1, c0:c1, 1] = np.nan
    return env


def stale_frame(n, seed=5):
    """A finite previous frame plus a handful of NaN / +Inf / -Inf pixels in each buffer."""
    rng = np.random.RandomState(seed)
    f = dict(accum=rng.uniform(0.02, 3.0, (n, 3)).astype(np.float32), depth=rng.uniform(0.0, 60.0, n).astype(np.float32),
             cost=rng.uniform(0.0, 1.0, (n, 3)).astype(np.float32))
    for i, p in enumerate(rng.choice(n, 30, replace=False)):
        bad = (np.nan, np.inf, -np.inf)[i % 3]
        f["accum"][p, i % 3] = bad; f["cost"][p, (i + 1) % 3] = bad
        if i % 2: f["depth"][p] = bad
    return f


def zero_frame(n):
    return dict(accum=np.zeros((n, 3), np.float32), depth=np.zeros(n, np.float32), cost=np.zeros((n, 3), np.float32))


def fill(r, frame, rows=None):
    """Pre-fill a renderer's accum / depth / cost with `frame` (full-frame arrays); a shard takes its rows of it (global rows
    `rows`, padding rows >= H left zero)."""
    for k in ("accum", "depth", "cost"):
        a = torch.from_numpy(np.ascontiguousarray(frame[k]))
        buf = getattr(r.buffers, k)
        if rows is None:
            buf.copy_(a.to(buf.device))
        else:
            full = a.reshape(r.height, r.width, -1)
            loc = torch.zeros((len(rows), r.width, full.shape[-1]), dtype=full.dtype)
            ok = rows < r.height
            loc[torch.from_numpy(np.nonzero(ok)[0])] = full[torch.from_numpy(rows[ok])]
            buf.copy_(loc.reshape(buf.shape).to(buf.device))


SCENES = {
    # HDRI with Inf / NaN texels, direct integrator
    "hdri": dict(kp=dict(ray_depth=4), env="non_finite"),
    # zero green extinction: Inf / NaN throughput after the first scatter, direct integrator
    "extinction": dict(kp=dict(ray_depth=4, extinction=V.f3(1.0, 0.0, 1.0))),
    # zero green extinction through the volumetric path integrator (NEE, sky MIS), sky tables as in test_parity_gpu
    "integrator1": dict(kp=dict(ray_depth=4, integrator=1, extinction=V.f3(1.0, 0.0, 1.0)), tables=True),
}


class Case:
    """A scene, a camera and the kernel parameters both kernels run with."""

    def __init__(self, dragon, W, H, kp=None, env=None, tables=False):
        self.W, self.H, self.n = W, H, W * H
        self.scene = make_scene(dragon)
        self.cam = self.scene.frame_camera(W, H)
        if env == "non_finite":
            self.scene.env_tex.destroy(); self.scene.env_tex = texture_env(non_finite_env(self.cam, W, H))
        self.kw = dict(kp or {})
        self.tables = V.EnvTables(_sky_power_table()) if tables else None
        if tables:
            sky_tables(self.scene, "own")

    def renderer(self, **extra):
        r = V.Renderer(self.scene, self.W, self.H, kp=make_kp(**self.kw), cam=self.cam, **extra)
        if self.tables: self.tables.apply(r.kp)
        return r

    def close(self):
        if self.tables: self.tables.destroy()
        self.scene.destroy()


def outputs(r, scene):
    return {k: getattr(r.buffers, k).clone() for k in BUFFERS} | dict(blue_noise=scene.d_blue_noise.clone(), iteration=r.kp.iteration)


def host(t):
    return t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)


def scalars(out, prev):
    """Full-frame scalars: pixels whose accum equals the previous frame's bit for bit, non-finite pixels per buffer, sum of
    the finite accum entries."""
    a = host(out["accum"]).reshape(-1, 3)
    same = (a.view(np.uint32) == np.ascontiguousarray(prev["accum"]).view(np.uint32)).all(axis=1)
    nf = [int((~np.isfinite(host(out[k]).reshape(a.shape[0], -1))).any(axis=1).sum()) for k in ("accum", "depth", "cost", "raw")]
    return dict(n_stale=np.int64(same.sum()), nonfinite=np.array(nf, np.int64), finite_sum=np.float64(a[np.isfinite(a)].astype(np.float64).sum()))


def reference_run(case, frame, start, passes):
    """The reference kernel on `frame` from iteration `start`, `passes` passes (race-free protocol), blue noise from its
    initial state.  Returns the outputs and the full-frame scalars."""
    orc = oracle_ref.RefOracle()
    ref = case.renderer()
    ref.params.p_oct.value = orc.build_octree(case.scene.h_volumes, 1)
    fill(ref, frame); ref.kp.iteration = start
    case.scene.reset_blue_noise()
    orc.render(ref, passes)
    out = outputs(ref, case.scene)
    ref.close()
    return out | scalars(out, frame)


def run_protocol(case, proto, frame, start, passes):
    """This library on `frame` from iteration `start`: "fused" (one render(passes) call), "single" (render_pass() per pass),
    "level_a" (the cubin, one launch per pass) or "shards" (3 interleaved-stripe ranks on this GPU, un-permuted)."""
    sc = case.scene
    if proto == "shards":
        parts = []
        for rank in range(3):
            r = case.renderer(rank=rank, n_ranks=3, stripe_rows=8)
            fill(r, frame, V.stripe_rows_of_rank(case.H, rank, 3, 8)); r.kp.iteration = start
            sc.reset_blue_noise(); r.render(passes); parts.append(r)
        torch.cuda.synchronize()
        out = {k: parts[0].unpermute(torch.cat([getattr(p.buffers, k).reshape(p.n_local, -1) for p in parts]), ELEM[k]) for k in BUFFERS}
        out["depth"] = out["depth"].reshape(-1); out["display"] = out["display"].reshape(-1)
        out |= dict(blue_noise=sc.d_blue_noise.clone(), iteration=parts[-1].kp.iteration)
        for p in parts: p.close()
        return out
    r = case.renderer()
    fill(r, frame); r.kp.iteration = start
    sc.reset_blue_noise()
    if proto == "fused":
        r.render(passes)
    elif proto == "single":
        for _ in range(passes): r.render_pass()
    else:
        level_a_launcher()(r, passes)
    torch.cuda.synchronize()
    out = outputs(r, sc)
    r.close()
    return out


def compare(want, got, same, what):
    """What differs between two frames: want(k) and got(k) give the arrays (the same rows of each), same(k) says whether
    cost and blue_noise are bit-identical."""
    errs = []
    if flipped_fraction(got("accum"), want("accum")) > MAX_FLIPPED: errs.append("accum")
    if flipped_fraction(got("depth")[:, None], want("depth")[:, None]) > MAX_FLIPPED: errs.append("depth")
    raw, rw = got("raw"), want("raw")
    if flipped_fraction(raw[:, :3], rw[:, :3]) > MAX_FLIPPED: errs.append("raw.xyz")
    if np.mean(np.abs(raw[:, 3] - rw[:, 3]) > 1e-5) > MAX_FLIPPED: errs.append("raw.w")
    dm = got("display").view(np.uint8).reshape(-1, 4).astype(int)
    dr = want("display").view(np.uint8).reshape(-1, 4).astype(int)
    if np.abs(dm - dr).max() > 1 or np.mean(np.abs(dm - dr).max(axis=1) > 0) > MAX_FLIPPED: errs.append("display")
    errs += [k for k in EXACT if not same(k)]
    if int(got("iteration")) != int(want("iteration")): errs.append("iteration")
    return [f"{what}: {e}" for e in errs]


def mismatches(R, got, what, prefix="", prev=None):
    """What differs between this library's outputs `got` and the reference's (keys under `prefix`); with the previous frame
    `prev`, the full-frame scalars too."""
    k = lambda name: prefix + name
    errs = compare(lambda n: R.want(k(n)), lambda n: R.pick(k(n), host(got[n])), lambda n: R.same(k(n), host(got[n])), what)
    if prev is not None:
        s = scalars(got, prev)
        if int(s["n_stale"]) != int(R.want(k("n_stale"))): errs.append(f"{what}: n_stale {int(s['n_stale'])} != {int(R.want(k('n_stale')))}")
        if not np.array_equal(s["nonfinite"], R.want(k("nonfinite"))): errs.append(f"{what}: nonfinite {s['nonfinite'].tolist()} != {R.want(k('nonfinite')).tolist()}")
        want_sum = float(R.want(k("finite_sum")))
        if not abs(float(s["finite_sum"]) - want_sum) <= 1e-4 * abs(want_sum): errs.append(f"{what}: finite_sum {float(s['finite_sum']):.9g} != {want_sum:.9g}")
    return errs


def recorded_mismatches(R, a, b, what):
    """What differs between two of the reference's own outputs (prefixes a and b): bit-exact arrays by digest where only the
    digest was recorded."""
    def same(n):
        if R.live or f"{a}{n}" not in R.meta:
            return host(R.want(f"{a}{n}")).tobytes() == host(R.want(f"{b}{n}")).tobytes()
        return R.meta[f"{a}{n}"]["sha256"] == R.meta[f"{b}{n}"]["sha256"]
    return compare(lambda n: R.want(f"{b}{n}"), lambda n: R.want(f"{a}{n}"), same, what)


EXACT = ("cost", "blue_noise")


def check_protocols(request, case, frame, start, passes, protocols):
    R = reference_outputs.load(request, lambda: reference_run(case, frame, start, passes), exact=EXACT)
    errs = []
    for proto in protocols:
        got = run_protocol(case, proto, frame, start, passes)
        errs += mismatches(R, got, proto, prev=frame)
    return R, errs


# ---- (a) stale frame at iteration 0, non-finite samples -----------------------------------------------------------------
@pytest.mark.parametrize("scene", list(SCENES))
def test_stale_frame_at_iteration_zero_with_non_finite_samples(request, dragon, scene):
    """accum / depth / cost hold a previous frame (with a few NaN / Inf pixels) and iteration is 0, as after any edit in the
    reference UI; 3 passes.  Where the first sample is non-finite the reference keeps the stale pixel (:2263)."""
    W, H, P = 320, 200, 3
    case = Case(dragon, W, H, **SCENES[scene])
    frame = stale_frame(W * H)
    R, errs = check_protocols(request, case, frame, 0, P, ("fused", "single", "level_a", "shards"))
    case.close()
    n_stale = int(R.want("n_stale"))
    print(f"{scene}: reference keeps the stale pixel in {n_stale} of {W * H}; non-finite pixels {R.want('nonfinite').tolist()}")
    assert n_stale >= (0.2 * W * H if scene == "hdri" else 1), "too few pixels take the guard at iteration 0"
    assert not errs, "; ".join(errs)


# ---- (b) non-finite samples on zeroed buffers, iterations 0..3 -----------------------------------------------------------
@pytest.mark.parametrize("scene", list(SCENES))
def test_non_finite_samples_on_zeroed_buffers(request, dragon, scene):
    """The running-mean guard (value = accum for iteration > 0) and the tr guard (raw.w = 1) over passes 0..3."""
    W, H, P = 320, 200, 4
    case = Case(dragon, W, H, **SCENES[scene])
    R, errs = check_protocols(request, case, zero_frame(W * H), 0, P, ("fused", "single", "level_a"))
    case.close()
    assert int(R.want("nonfinite")[0]) < W * H and float(R.want("finite_sum")) > 0
    assert not errs, "; ".join(errs)


# ---- (c) progressive hand-off between the two implementations ------------------------------------------------------------
HW = (24, 16)          # small enough that the reference's whole state is recorded (tests/reference_outputs.py WHOLE_BYTES)


def state_of(out, n):
    """What a pass reads from the previous one: accum / depth / cost and the blue-noise entries a frame of n pixels advances."""
    return dict(accum=host(out["accum"]), depth=host(out["depth"]), cost=host(out["cost"]), bn_head=np.ascontiguousarray(host(out["blue_noise"])[:n]))


def load_state(r, scene, st):
    """Hand `r` and the scene a state as state_of() took it."""
    fill(r, st)
    bn = torch.from_numpy(scene.bn_host.copy()); bn[:len(st["bn_head"])] = torch.from_numpy(st["bn_head"])
    scene.d_blue_noise.copy_(bn.to(scene.device))


def library_passes(level, r, passes):
    """`passes` passes of this library on `r`: level (B), one fused call, or level (A), one cubin launch per pass."""
    if level == "A":
        level_a_launcher()(r, passes)
    else:
        r.render(passes)
    torch.cuda.synchronize()


STATE = ("accum", "depth", "cost", "bn_head")


@pytest.mark.parametrize("order", ["reference_first", "library_first"])
def test_progressive_hand_off(request, dragon, order):
    """Passes 0..2 by one implementation, 3..5 by the other on exactly those buffers and that blue-noise state, against six
    reference passes, through level (B) and level (A).  Library first, where the reference is not built: the library's state
    after passes 0..2 must still equal the reference's own, and the reference's continuation recorded from the library's
    state must equal its six passes."""
    W, H = HW
    case = Case(dragon, W, H, kp=dict(ray_depth=4), env="non_finite")
    zero = zero_frame(W * H)
    levels = ("B", "A")

    def reference():
        three = reference_run(case, zero, 0, 3)
        assert np.array_equal(host(three["blue_noise"])[W * H:], case.scene.bn_host[W * H:]), "entries beyond W*H must stay put"
        out = {f"handoff.{k}": v for k, v in state_of(three, W * H).items()} | {f"six.{k}": v for k, v in reference_run(case, zero, 0, 6).items()}
        if order == "library_first":
            orc = oracle_ref.RefOracle()
            for level in levels:
                r = case.renderer(); case.scene.reset_blue_noise(); library_passes(level, r, 3)
                st = state_of(outputs(r, case.scene), W * H); r.close()
                ref = case.renderer(); ref.params.p_oct.value = orc.build_octree(case.scene.h_volumes, 1)
                load_state(ref, case.scene, st); ref.kp.iteration = 3
                orc.render(ref, 3)
                out |= {f"mixed{level}.{k}": v for k, v in outputs(ref, case.scene).items()}
                ref.close()
        return out
    R = reference_outputs.load(request, reference, exact=tuple(f"{p}.{k}" for p in ("six", "mixedA", "mixedB") for k in EXACT))
    handoff = {k: R.want(f"handoff.{k}") for k in STATE}
    errs = []
    for level in levels:
        if order == "reference_first":
            r = case.renderer(); load_state(r, case.scene, handoff); r.kp.iteration = 3
            library_passes(level, r, 3)
            errs += mismatches(R, outputs(r, case.scene), f"level {level} after the reference", prefix="six.")
            r.close()
            continue
        r = case.renderer(); case.scene.reset_blue_noise(); library_passes(level, r, 3)
        st = state_of(outputs(r, case.scene), W * H); r.close()
        if flipped_fraction(st["accum"], handoff["accum"]) > MAX_FLIPPED or \
                flipped_fraction(st["depth"][:, None], handoff["depth"][:, None]) > MAX_FLIPPED or \
                any(not np.array_equal(st[k], handoff[k]) for k in ("cost", "bn_head")):
            errs.append(f"level {level}: state after passes 0..2 differs from the reference's")
        errs += recorded_mismatches(R, f"mixed{level}.", "six.", f"reference after level {level}")
    case.close()
    assert not errs, "; ".join(errs)


# ---- (d) limits and flags ---------------------------------------------------------------------------------------------------
def test_iteration_limit_from_reference_state(request, dragon):
    """max_interactions = 5: the reference renders passes 0..2, then one render(4) call from iteration 3 samples two passes and
    only re-tonemaps two (:2254, :2283)."""
    W, H = HW
    case = Case(dragon, W, H, kp=dict(ray_depth=4, max_interactions=5))
    zero = zero_frame(W * H)

    def reference():
        three = reference_run(case, zero, 0, 3)
        seven = reference_run(case, zero, 0, 7)
        return {f"handoff.{k}": v for k, v in state_of(three, W * H).items()} | {f"seven.{k}": v for k, v in seven.items()}
    R = reference_outputs.load(request, reference, exact=tuple(f"seven.{k}" for k in EXACT))
    handoff = {k: R.want(f"handoff.{k}") for k in STATE}
    assert int(R.want("seven.iteration")) == 7
    errs = []
    for level in ("B", "A"):
        r = case.renderer(); load_state(r, case.scene, handoff); r.kp.iteration = 3
        library_passes(level, r, 4)
        errs += mismatches(R, outputs(r, case.scene), f"level {level}", prefix="seven.")
        r.close()
    case.close()
    assert not errs, "; ".join(errs)


def test_render_flag_off_on_stale_frame(request, dragon):
    """render == false from iteration 2 on a stale frame: WHITE enters the running mean (:2248, :2283), nothing is traced."""
    W, H, P = 160, 100, 2
    case = Case(dragon, W, H, kp=dict(ray_depth=2, render=0))
    frame = stale_frame(W * H, seed=9)
    R, errs = check_protocols(request, case, frame, 2, P, ("fused", "single", "level_a"))
    case.close()
    assert not errs, "; ".join(errs)


def test_curand_offset_wrap(request, dragon):
    """Passes 2^20 - 2 .. 2^20 + 1: the reference's curand offset iteration * 4096 wraps modulo 2^32 at 2^20 (:2235)."""
    W, H, P = 160, 100, 4
    case = Case(dragon, W, H, kp=dict(ray_depth=4, max_interactions=1 << 21))
    frame = stale_frame(W * H, seed=11)
    R, errs = check_protocols(request, case, frame, (1 << 20) - 2, P, ("fused", "single", "level_a"))
    case.close()
    assert not errs, "; ".join(errs)


# ---- (e) display path ---------------------------------------------------------------------------------------------------------
def test_viz_dof_and_exposure_display_path(request, dragon):
    """cam.viz_dof with a thin lens and a focus distance at which all three bands occur (far: red, near: blue, in focus:
    green; :2270-2274), exposure_scale = 2.5 (:2305)."""
    W, H, P = 256, 160, 2
    case = Case(dragon, W, H, kp=dict(ray_depth=3, exposure_scale=2.5))
    lo, hi = case.scene.world_bounds()
    aof = float(np.linalg.norm(hi - lo)) / 6.0                     # 1 / lens_radius
    case.cam = case.scene.frame_camera(W, H, aperture=2.0 / aof)
    case.cam.viz_dof = 1
    case.cam.focus_dist = case.cam.focus_dist - aof                # in focus: depths in (D - 2 aof, D), D the distance to the box centre
    R, errs = check_protocols(request, case, zero_frame(W * H), 0, P, ("fused", "level_a"))
    aof_k = 1.0 / case.cam.lens_radius
    r = case.renderer(); case.scene.reset_blue_noise(); r.render_pass(); torch.cuda.synchronize()
    d = r.buffers.depth.cpu().numpy(); f = case.cam.focus_dist
    bands = [float(np.mean(d > f + aof_k)), float(np.mean(d < f - aof_k)), float(np.mean((d > f - aof_k) & (d < f + aof_k)))]
    r.close(); case.close()
    print(f"viz_dof bands of the first pass (red, blue, green): {bands}")
    assert min(bands) > 0.005, "every band must occur"
    assert not errs, "; ".join(errs)
