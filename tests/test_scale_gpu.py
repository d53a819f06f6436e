"""GPU parity at the MEASURED scale and for the round-2 rows (VERDICT r1 "next" items 1 and 5):
  * the timed configuration itself (BASELINE configs[1]: 1920x1080x64 spp, real HDRI) against the reference kernel;
  * configs[2] with SURVEY's real parameters (volume_depth = 50; integrator = 1, ray_depth = 50);
  * the UNMODIFIED reference kernel at its race-free size (256x256) against the race-free protocol used everywhere else;
  * octrees of 120 and 600 instances node for node against the reference builder, > 600 instances through the flat tables;
  * the LBVH against the reference's BuildBVH (sorted ids, topology, boxes: bit-exact);
  * a 2-rank NCCL job (when the box has 2 GPUs) whose gathered frame must be bit-identical to the single-GPU frame.
Tolerance as in test_parity_gpu.py: |d| <= 1e-5 + 1e-4*|ref| per channel on >= 99.9 % of the pixels.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import vpt_b200 as V
from vpt_b200.scene import synthetic_env
import oracle_ref
import reference_outputs
from test_parity_gpu import (flipped_fraction, make_kp, make_scene, MAX_FLIPPED, needs_ref, _big_asset, _sky_power_table, read_tree, octree_arrays,
                             assert_octree_equals_reference, OCTREE_ARRAYS, SKY_TABLES, sky_tables, sky_sources)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
has_atmo = os.path.exists(os.path.join(oracle_ref.REF_DIR, "atmo", "atmosphere_kernels.ptx"))


@pytest.fixture(scope="module")
def dragon():
    return V.Volume.load_vdb(V.find_asset("dragon.vdb"))


def scattered(dragon, n, seed, spread):
    rng = np.random.RandomState(seed)
    inst = []
    for _ in range(n):
        q = rng.randn(4); q /= np.linalg.norm(q)
        inst.append(dragon.instance(pos=tuple(rng.uniform(-spread, spread, 3)), quat=tuple(q), scale=float(rng.uniform(0.7, 1.3))))
    return inst


# ---- the timed configuration, checked ------------------------------------------------------------------------------
@needs_ref
@pytest.mark.skipif(_big_asset("Barce_Rooftop_C_3k.hdr") is None, reason="HDRI not staged (oracle/_ref/assets)")
def test_baseline_config2_full_frame_against_reference(dragon):
    """BASELINE configs[1] exactly as bench.py times it: 1920x1080, 64 spp, ray_depth 100, sun + real HDRI."""
    scene = V.Scene([dragon.instance()], env="Barce_Rooftop_C_3k.hdr")
    assert not scene.data_notes
    kw = dict(ray_depth=100, volume_depth=1, integrator=0)
    mine = V.Renderer(scene, 1920, 1080, kp=make_kp(**kw)); ref = V.Renderer(scene, 1920, 1080, kp=make_kp(**kw), cam=mine.cam)
    orc = oracle_ref.RefOracle()
    ref.params.p_oct.value = orc.build_octree(scene.h_volumes, 1)
    scene.reset_blue_noise(); orc.render(ref, 64); bn_ref = scene.d_blue_noise.clone()
    scene.reset_blue_noise(); mine.render(64); torch.cuda.synchronize()
    want = ref.buffers.accum.cpu().numpy(); got = mine.buffers.accum.cpu().numpy()
    frac = flipped_fraction(got, want)
    print(f"cfg2 full frame: flipped {frac:.3g}, max |d| {np.abs(got - want).max():.3g}, ref mean {want.mean():.6g}")
    assert frac <= MAX_FLIPPED
    assert flipped_fraction(mine.buffers.depth.cpu().numpy()[:, None], ref.buffers.depth.cpu().numpy()[:, None]) <= MAX_FLIPPED
    assert torch.equal(scene.d_blue_noise, bn_ref)
    dm = mine.buffers.display.cpu().numpy().view(np.uint8).reshape(-1, 4).astype(int)
    dr = ref.buffers.display.cpu().numpy().view(np.uint8).reshape(-1, 4).astype(int)
    assert np.abs(dm - dr).max() <= 1 and np.mean(np.abs(dm - dr).max(axis=1) > 0) <= MAX_FLIPPED


@needs_ref
@pytest.mark.skipif(_big_asset("fireball.vdb") is None, reason="fireball.vdb not staged (oracle/_ref/assets)")
def test_baseline_config3_real_parameters_against_reference():
    """BASELINE configs[2] with SURVEY 8(d)'s parameters: emission + multiple scattering through volume_depth = 50."""
    vol = V.Volume.load_vdb(_big_asset("fireball.vdb"))
    scene = V.Scene([vol.instance()], env=synthetic_env(512, 256))
    kw = dict(ray_depth=2, volume_depth=50, emission_scale=1.0, emission_pivot=1.0)
    mine = V.Renderer(scene, 640, 360, kp=make_kp(**kw)); ref = V.Renderer(scene, 640, 360, kp=make_kp(**kw), cam=mine.cam)
    orc = oracle_ref.RefOracle()
    ref.params.p_oct.value = orc.build_octree(scene.h_volumes, 1)
    scene.reset_blue_noise(); orc.render(ref, 3)
    scene.reset_blue_noise(); mine.render(3); torch.cuda.synchronize()
    want = ref.buffers.accum.cpu().numpy(); got = mine.buffers.accum.cpu().numpy()
    frac = flipped_fraction(got, want)
    print(f"cfg3 volume_depth=50: flipped {frac:.3g}, ref mean {want.mean():.6g}")
    assert float(want.mean()) > 1e-3 and frac <= MAX_FLIPPED
    assert flipped_fraction(mine.buffers.depth.cpu().numpy()[:, None], ref.buffers.depth.cpu().numpy()[:, None]) <= MAX_FLIPPED


@needs_ref
@pytest.mark.skipif(_big_asset("fireball.vdb") is None or not has_atmo, reason="fireball.vdb / oracle/_ref/atmo not staged")
def test_baseline_config3_volumetric_path_integrator_against_reference():
    """configs[2], secondary variant of SURVEY 8(d): integrator = 1, ray_depth = 50, emission, sky environment (type 0)."""
    vol = V.Volume.load_vdb(_big_asset("fireball.vdb"))
    scene = V.Scene([vol.instance()], env=synthetic_env(512, 256))
    orc = oracle_ref.RefOracle()
    orc.atmosphere_init(scene.atmos)
    tables = V.EnvTables(_sky_power_table())
    kw = dict(integrator=1, environment_type=0, ray_depth=50, emission_scale=1.0, emission_pivot=1.0)
    mine = V.Renderer(scene, 640, 360, kp=make_kp(**kw)); ref = V.Renderer(scene, 640, 360, kp=make_kp(**kw), cam=mine.cam)
    tables.apply(mine.kp); tables.apply(ref.kp)
    ref.params.p_oct.value = orc.build_octree(scene.h_volumes, 1)
    scene.reset_blue_noise(); orc.render(ref, 2)
    scene.reset_blue_noise(); mine.render(2); torch.cuda.synchronize()
    want = ref.buffers.accum.cpu().numpy(); got = mine.buffers.accum.cpu().numpy()
    frac = flipped_fraction(got, want)
    print(f"cfg3 integrator=1 ray_depth=50: flipped {frac:.3g}, ref mean {want.mean():.6g}")
    assert np.isfinite(want).all() and float(want.mean()) > 1e-3 and frac <= MAX_FLIPPED
    tables.destroy()


def test_unmodified_reference_kernel_equals_race_free_protocol_at_256(request, dragon):
    """SURVEY 8(c)(i): at 256x256 every thread of the unmodified kernel touches only its own blue-noise entry, so the kernel is
    race-free there.  It must equal the protocol every other test uses (nobn build + the reference's own update statements as a
    separate launch) bit for bit -- and this library."""
    scene = make_scene(dragon)
    kw = dict(ray_depth=3, volume_depth=2)
    mine = V.Renderer(scene, 256, 256, kp=make_kp(**kw))

    def reference():
        a = V.Renderer(scene, 256, 256, kp=make_kp(**kw), cam=mine.cam); b = V.Renderer(scene, 256, 256, kp=make_kp(**kw), cam=mine.cam)
        orc = oracle_ref.RefOracle()
        root = orc.build_octree(scene.h_volumes, 1)
        a.params.p_oct.value = root; b.params.p_oct.value = root
        scene.reset_blue_noise(); orc.render(a, 4, race_free=False); bn_a = scene.d_blue_noise.clone()
        scene.reset_blue_noise(); orc.render(b, 4, race_free=True); bn_b = scene.d_blue_noise.clone()
        for name in ("accum", "depth", "raw", "display", "cost"):
            assert torch.equal(getattr(a.buffers, name), getattr(b.buffers, name)), name
        assert torch.equal(bn_a, bn_b)
        return dict(accum=a.buffers.accum, blue_noise=bn_a)
    R = reference_outputs.load(request, reference, exact=("blue_noise",))
    scene.reset_blue_noise(); mine.render(4); torch.cuda.synchronize()
    assert R.same("blue_noise", scene.d_blue_noise)
    assert flipped_fraction(R.pick("accum", mine.buffers.accum), R.want("accum")) <= MAX_FLIPPED


# ---- instance acceleration build (row N1) --------------------------------------------------------------------------
@pytest.mark.parametrize("n,spread", [(120, 25.0), (600, 40.0)])
def test_octree_node_for_node_and_render_at_many_instances(request, dragon, n, spread):
    inst = scattered(dragon, n, 11 + n, spread)
    scene = make_scene(dragon, instances=inst)
    kw = dict(ray_depth=2)
    W, H = (256, 144) if n <= 120 else (192, 108)
    mine = V.Renderer(scene, W, H, kp=make_kp(**kw))
    foreign = None

    def reference():
        nonlocal foreign
        orc = oracle_ref.RefOracle()
        ref_root = orc.build_octree(scene.h_volumes, n)
        ref = V.Renderer(scene, W, H, kp=make_kp(**kw), cam=mine.cam)
        foreign = V.Renderer(scene, W, H, kp=make_kp(**kw), cam=mine.cam)
        ref.params.p_oct.value = ref_root
        foreign.params.p_oct.value = ref_root        # this library on the REFERENCE's pointer-linked octree (k_prepare_scene path)
        scene.reset_blue_noise(); orc.render(ref, 1)
        scene.reset_blue_noise(); foreign.render(1); torch.cuda.synchronize()
        return dict(octree_arrays(read_tree(ref_root)), accum=ref.buffers.accum, mean=float(ref.buffers.accum.mean()))
    R = reference_outputs.load(request, reference, exact=OCTREE_ARRAYS)
    mine_t = read_tree(scene.d_oct_root)
    assert_octree_equals_reference(R, mine_t)
    # the flat (CSR) tables the render kernels read carry the same leaf lists
    lists = scene.leaf_lists()
    for l in range(512):
        j = 73 + l
        want = list(mine_t[j].vol_indices[:mine_t[j].num_volumes]) if j in mine_t else []
        assert lists[l] == want, l
    info = scene.octree_info()
    assert info["n"] == n and info["reference_layout"] and info["total_leaf_entries"] == sum(len(x) for x in lists)
    scene.reset_blue_noise(); mine.render(1); torch.cuda.synchronize()
    assert float(R.want("mean")) > 1e-4
    assert flipped_fraction(R.pick("accum", mine.buffers.accum), R.want("accum")) <= MAX_FLIPPED
    if foreign is not None:
        for name in ("accum", "depth", "raw", "display"):
            assert torch.equal(getattr(mine.buffers, name), getattr(foreign.buffers, name)), name


def test_more_than_600_instances_through_flat_tables(request, dragon):
    """BASELINE configs[4] shape: 1000 instances, beyond the reference's OCTNode capacity (quirk Q11).  No oracle can run this,
    so: 500 real instances, each followed by a GHOST twin (same transform, all-zero density grid).  A ghost adds exactly +0.0f to
    every density sum and leaves every node's occupancy, the root box and the majorant unchanged, so the 1000-instance frame must
    be bit-identical to the 500-instance frame -- which IS checked against the reference kernel."""
    real = scattered(dragon, 500, 5, 38.0)
    zero = np.zeros((31, 49, 70), dtype=np.float32)
    ghost = V.Volume.from_dense(zero, bbox_min=dragon.meta["bbox_min"], xform=dragon.meta["xform"], voxelsize=dragon.meta["voxel_size"])
    ghost.rec.vdb_info.bmax = dragon.rec.vdb_info.bmax
    ghost.rec.vdb_info.max_density = 0.0
    both = []
    for g in real:
        t = V.GPU_VDB(); C.memmove(C.byref(t), C.byref(g), C.sizeof(V.GPU_VDB))
        t.vdb_info.density_texture = ghost.rec.vdb_info.density_texture
        t.vdb_info.max_density = 0.0
        both += [g, t]
    s500 = make_scene(dragon, instances=real)
    s1000 = make_scene(dragon, instances=both); s1000.keep.append(ghost)
    info = s1000.octree_info()
    assert info["n"] == 1000 and not info["reference_layout"]
    l500, l1000 = s500.leaf_lists(), s1000.leaf_lists()
    for l in range(512):
        assert l1000[l] == [x for i in l500[l] for x in (2 * i, 2 * i + 1)], l
    kw = dict(ray_depth=2, volume_depth=2)
    a = V.Renderer(s500, 256, 144, kp=make_kp(**kw)); b = V.Renderer(s1000, 256, 144, kp=make_kp(**kw), cam=a.cam)

    def reference():
        ref = V.Renderer(s500, 256, 144, kp=make_kp(**kw), cam=a.cam)
        orc = oracle_ref.RefOracle()
        ref.params.p_oct.value = orc.build_octree(s500.h_volumes, 500)
        s500.reset_blue_noise(); orc.render(ref, 2)
        return dict(accum=ref.buffers.accum, mean=float(ref.buffers.accum.mean()))
    R = reference_outputs.load(request, reference)
    s500.reset_blue_noise(); a.render(2)
    s1000.reset_blue_noise(); b.render(2); torch.cuda.synchronize()
    assert float(R.want("mean")) > 1e-4
    assert flipped_fraction(R.pick("accum", a.buffers.accum), R.want("accum")) <= MAX_FLIPPED
    for name in ("accum", "depth", "raw", "display"):
        assert torch.equal(getattr(a.buffers, name), getattr(b.buffers, name)), name
    with pytest.raises(V.VptError):                      # no reference-layout nodes exist for > 600 instances
        read_tree(s1000.d_oct_root)


BVH_ARRAYS = ("scene_bounds", "leaves", "leaf_boxes", "nodes", "node_boxes")


def bvh_arrays(scene_bounds, bvh):
    """A BVH read with read_bvh as flat arrays (the reference never writes the root's parent: stored as 0)."""
    box = lambda b: np.frombuffer(bytes(b), dtype=np.float32)
    return dict(scene_bounds=np.array(scene_bounds, dtype=np.float32),
                leaves=np.array([(l["volIndex"], l["parent"]) for l in bvh["leaves"]], dtype=np.int64).reshape(-1, 2),
                leaf_boxes=np.array([box(l["box"]) for l in bvh["leaves"]], dtype=np.float32).reshape(-1, 6),
                nodes=np.array([(d["left"], d["right"], d["minId"], d["maxId"], d["parent"] if i else 0) for i, d in enumerate(bvh["nodes"])],
                               dtype=np.int64).reshape(-1, 5),
                node_boxes=np.array([box(d["box"]) for d in bvh["nodes"]], dtype=np.float32).reshape(-1, 6))


@pytest.mark.parametrize("n,spread,dups", [(2, 5.0, 0), (3, 5.0, 0), (37, 12.0, 6), (120, 25.0, 0), (600, 40.0, 40)])
def test_lbvh_bit_exact_against_reference_builder(request, dragon, n, spread, dups):
    """Karras LBVH (bvh_kernels.cu:253-453, 460-580): sorted instance ids, child / parent topology, node ranges and boxes.
    `dups` instances repeat an earlier transform exactly, so equal Morton codes exercise the (code, id) tie-break."""
    inst = scattered(dragon, n - dups, 100 + n, spread)
    inst += [inst[i % len(inst)] for i in range(dups)]
    scene = make_scene(dragon, instances=inst)
    mine = scene.build_bvh()

    def reference():
        orc = oracle_ref.RefOracle()
        dn, dl = C.c_void_p(0), C.c_void_p(0); sb = (C.c_float * 6)()
        rc = orc.lib.vptref_build_bvh(C.cast(scene.h_volumes, C.c_void_p), n, C.byref(dn), C.byref(dl), sb)
        assert rc == 0
        return bvh_arrays(list(sb), V.read_bvh(dn.value, dl.value, n))
    R = reference_outputs.load(request, reference, exact=BVH_ARRAYS)
    assert mine["ids"] == [l["volIndex"] for l in mine["leaves"]]
    assert sorted(mine["ids"]) == list(range(n)) and mine["codes"] == sorted(mine["codes"]) and max(mine["codes"]) < (1 << 30)
    for k, a in bvh_arrays(mine["scene_bounds"], mine).items():
        assert R.same(k, a), k
    # the root's box is the scene box, every internal node covers its [minId, maxId] leaf range
    root_box = np.frombuffer(mine["nodes"][0]["box"], dtype=np.float32)
    assert list(root_box) == mine["scene_bounds"]


def test_lbvh_single_instance_and_large_count(dragon):
    one = make_scene(dragon).build_bvh()                 # n == 1: the reference dereferences an unwritten pointer here (Q18)
    assert one["nodes"] == [] and one["leaves"][0]["volIndex"] == 0 and one["leaves"][0]["parent"] == -1
    n = 5000
    scene = make_scene(dragon, instances=scattered(dragon, n, 77, 120.0))
    b = scene.build_bvh()
    assert sorted(b["ids"]) == list(range(n)) and b["codes"] == sorted(b["codes"])
    # structural invariants of a Karras tree: every node but the root has exactly one parent, ranges nest
    seen = [0] * (2 * n - 1)
    for i, nd in enumerate(b["nodes"]):
        for ch in (nd["left"], nd["right"]):
            seen[ch] += 1
            child = b["nodes"][ch] if ch < n - 1 else b["leaves"][ch - (n - 1)]
            assert child["parent"] == i
            lo, hi = (child["minId"], child["maxId"]) if ch < n - 1 else (ch - (n - 1),) * 2
            assert nd["minId"] <= lo <= hi <= nd["maxId"]
            cb = np.frombuffer(child["box"], dtype=np.float32); pb = np.frombuffer(nd["box"], dtype=np.float32)
            assert (pb[:3] <= cb[:3]).all() and (pb[3:] >= cb[3:]).all()
    assert seen[0] == 0 and all(s == 1 for s in seen[1:])
    assert (b["nodes"][0]["minId"], b["nodes"][0]["maxId"]) == (0, n - 1)


def test_scene_cache_survives_address_reuse(dragon):
    """ADVICE r1: the flattened scene tables must not be keyed on device addresses alone -- a freed and rebuilt octree / GPU_VDB
    array often gets the same addresses back.  Render scene A, destroy it, build a different scene B (same sizes), render with the
    SAME context: the frame must equal B rendered by a fresh context."""
    a_inst = scattered(dragon, 8, 1, 6.0); b_inst = scattered(dragon, 8, 2, 6.0)
    sa = make_scene(dragon, instances=a_inst)
    r = V.Renderer(sa, 160, 96, kp=make_kp(ray_depth=2))
    r.render(2); torch.cuda.synchronize()
    addr = (sa.d_volumes.data_ptr(), sa.d_oct_root)
    cam = r.cam
    sa.destroy(); del sa.d_volumes
    sb = make_scene(dragon, instances=b_inst)
    reused = (sb.d_volumes.data_ptr(), sb.d_oct_root) == addr
    fresh = V.Renderer(sb, 160, 96, kp=make_kp(ray_depth=2), cam=cam)
    sb.reset_blue_noise(); fresh.render(2); torch.cuda.synchronize()
    # same context, new scene behind (possibly) the same addresses
    r.scene = sb; r.params = V.LaunchParams(sb, r.cam, r.kp); r.kp.blue_noise_buffer = sb.d_blue_noise.data_ptr()
    r.kp.emission_texture = sb.d_emission_lut.data_ptr(); r.kp.density_color_texture = sb.d_density_color.data_ptr(); r.kp.env_tex = sb.env_tex.tex
    r.kp.iteration = 0; r.buffers.zero_()
    sb.reset_blue_noise(); r.render(2); torch.cuda.synchronize()
    print("addresses reused:", reused)
    assert torch.equal(r.buffers.accum, fresh.buffers.accum)


# ---- multi-GPU: gathered frame == single-GPU frame, bit for bit ---------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs on the box")
def test_two_rank_exchange_is_bitwise_identical():
    """tools/mgpu_check.py under torchrun on 2 GPUs: peer-memory exchange and NCCL gather, accumulators and display words, two consecutive
    frames, side-stream gather -- each equal to the single-GPU frame bit for bit."""
    env = dict(os.environ); env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tools", "mgpu_check.py")]
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    print(out.stdout[-2000:], out.stderr[-2000:])
    assert out.returncode == 0 and "BITWISE_OK" in out.stdout


def test_peer_memory_exchange_with_three_shards_on_one_gpu(dragon):
    """The multi-GPU exchange protocol on ONE device: three contexts render the three shards of a frame on three streams and exchange
    through each other's blocks (same-process peer import).  The last resolve kernel of every shard stores its pixels into all three
    frames between the two flag handshakes; every frame must equal the single-context frame bit for bit, twice in a row (the second
    call exercises the "previous frame consumed" handshake), display words included."""
    W, H, P, R = 640, 360, 3, 3
    one_scene = make_scene(dragon)
    one = V.Renderer(one_scene, W, H, kp=make_kp(ray_depth=3))
    one.render(P); torch.cuda.synchronize()
    want1 = one.buffers.accum.clone(); disp1 = one.buffers.display.clone()
    one.kp.iteration = 0; one.render(P); torch.cuda.synchronize()
    want2 = one.buffers.accum.clone()
    scenes = [make_scene(dragon) for _ in range(R)]                    # one blue-noise state per shard, as one per process
    rs = [V.Renderer(scenes[k], W, H, kp=make_kp(ray_depth=3), cam=one.cam, rank=k, n_ranks=R, stripe_rows=8) for k in range(R)]
    blocks = (C.c_uint64 * R)()
    for k, r in enumerate(rs):
        raw = (C.c_ubyte * 64)()
        V._native.check(V.lib.vpt_comm_p2p_export(r.ctx, k, R, 8, W, H, 1, raw), r.ctx, "vpt_comm_p2p_export")
        b = C.c_uint64(0); V._native.check(V.lib.vpt_comm_p2p_block(r.ctx, C.byref(b)), r.ctx, "vpt_comm_p2p_block"); blocks[k] = b.value
    frames = []
    for r in rs:
        V._native.check(V.lib.vpt_comm_p2p_import_local(r.ctx, blocks), r.ctx, "vpt_comm_p2p_import_local")
        pa, pd = C.c_uint64(0), C.c_uint64(0)
        V._native.check(V.lib.vpt_comm_p2p_frame(r.ctx, C.byref(pa), C.byref(pd)), r.ctx, "vpt_comm_p2p_frame")
        frames.append((torch.as_tensor(V.renderer._DeviceView(pa.value, (W * H, 3), "<f4"), device="cuda"),
                       torch.as_tensor(V.renderer._DeviceView(pd.value, (W * H,), "<i4"), device="cuda")))
    streams = [torch.cuda.Stream() for _ in range(R)]
    torch.cuda.synchronize()
    for want, check_display in ((want1, True), (want2, False)):
        for r, st in zip(rs, streams):
            r.kp.iteration = 0
            r.render(P, stream=st.cuda_stream)                          # asynchronous: the three calls overlap on the device
        torch.cuda.synchronize()
        for k, (fa, fd) in enumerate(frames):
            assert torch.equal(fa, want), f"frame held by shard {k}"
            if check_display: assert torch.equal(fd, disp1.view(torch.int32) if disp1.dtype != torch.int32 else disp1), f"display held by shard {k}"
    for r in rs:
        n = C.c_uint64(0); V._native.check(V.lib.vpt_comm_p2p_status(r.ctx, C.byref(n)), r.ctx, "vpt_comm_p2p_status")
        assert n.value == 0, "a flag wait was abandoned"
    frames.clear()
    for r in rs: r.close()


# ---- level (A): the single-entry module behind the reference's unchanged Driver-API loader ------------------------------------
LEVEL_A = os.path.join(os.path.dirname(V.LIB_PATH), "volume_rt_kernel_b200.cubin")


def level_a_launcher():
    """launch(r, passes): the level (A) cubin loaded and launched with cuModuleLoad + cuModuleGetFunction("volume_rt_kernel") +
    cuLaunchKernel, one synchronised launch per pass with ++iteration (main.cpp:1823-1829).  Where oracle/_ref was built the calls
    are the oracle harness's own, the very ones that drive the reference kernel; elsewhere LevelAModule issues the same three."""
    if oracle_ref.available():
        orc = oracle_ref.RefOracle(); orc.load_kernels(); orc.load_candidate(LEVEL_A)

        def launch(r, passes):
            for _ in range(passes):
                orc.launch(r.params.array, r.width, r.height, orc.CANDIDATE)
                r.kp.iteration += 1
            torch.cuda.synchronize()
        return launch
    mod = V.LevelAModule(LEVEL_A)

    def launch(r, passes):
        for _ in range(passes):
            mod.launch(r, sync=True)
    return launch


@pytest.mark.skipif(not os.path.exists(LEVEL_A), reason="volume_rt_kernel_b200.cubin not built")
@pytest.mark.parametrize("cfg", [
    dict(W=512, H=512, passes=1, kp=dict(ray_depth=1)),                                    # BASELINE configs[0] resolution (plumbing config)
    dict(W=256, H=256, passes=3, kp=dict(ray_depth=100), unmodified=True),                 # vs the UNMODIFIED reference kernel at its race-free size
    dict(W=320, H=200, passes=2, kp=dict(ray_depth=4, volume_depth=5, phase_g1=-0.4)),
    dict(W=33, H=17, passes=2, kp=dict(ray_depth=2)),                                      # fewer pixels than blue-noise entries, ragged grid
    dict(W=256, H=160, passes=2, kp=dict(ray_depth=3, volume_depth=2), lights=True, sphere=True),
    dict(W=256, H=128, passes=2, kp=dict(ray_depth=3), aperture=0.2),                      # thin lens
    dict(W=200, H=120, passes=2, kp=dict(ray_depth=2), instances=8),                       # leaf lists read from the caller's OCTNodes
    dict(W=200, H=120, passes=1, kp=dict(ray_depth=6, integrator=1), atmo=True),           # volumetric path integrator, HDRI sky estimator
    dict(W=200, H=120, passes=1, kp=dict(ray_depth=2, environment_type=0), atmo=True),     # precomputed sky environment
])
def test_level_a_module_through_the_reference_loader(request, dragon, cfg):
    """The cubin is loaded with cuModuleLoad + cuModuleGetFunction("volume_rt_kernel") -- the same two calls and the same
    cuLaunchKernel line that drive the reference kernel -- and must match the oracle.  Live it runs on the REFERENCE's own
    pointer-linked octree; on the recorded outputs, on this library's octree in the same layout (node for node equal to the
    reference's: test_octree_node_for_node_and_render_at_many_instances)."""
    lights = [((9.0, 6.0, 2.0), (1.0, 0.8, 0.6), 40.0), ((-2.0, 3.0, 8.0), (0.5, 0.7, 1.0), 25.0)] if cfg.get("lights") else None
    inst = scattered(dragon, cfg["instances"], 9, 6.0) if cfg.get("instances") else None
    scene = make_scene(dragon, lights=lights, instances=inst)
    if cfg.get("sphere"):
        sp = scene.h_sphere; sp.center = V.f3(4.0, 6.5, 3.0); sp.radius = 1.2; sp.roughness = 0.7; sp.color = V.f3(0.8, 0.6, 0.3)
        scene.d_sphere.copy_(torch.frombuffer(bytearray(bytes(sp)), dtype=torch.uint8))
    W, H, P = cfg["W"], cfg["H"], cfg["passes"]
    cam = scene.frame_camera(W, H, aperture=cfg.get("aperture", 0.0))
    sources = SKY_TABLES if cfg.get("atmo") else ("hdri",)
    ref_root = None

    def reference():
        nonlocal ref_root
        orc = oracle_ref.RefOracle()
        ref_root = orc.build_octree(scene.h_volumes, len(scene.instances))
        out = {}
        for src in sources:
            if cfg.get("atmo"): sky_tables(scene, src)
            ref = V.Renderer(scene, W, H, kp=make_kp(**cfg["kp"]), cam=cam)
            ref.params.p_oct.value = ref_root
            scene.reset_blue_noise(); orc.render(ref, P, race_free=not cfg.get("unmodified"))
            out.update({f"{src}.accum": ref.buffers.accum, f"{src}.depth": ref.buffers.depth, f"{src}.display": ref.buffers.display,
                        f"{src}.blue_noise": scene.d_blue_noise.clone(), f"{src}.mean": float(ref.buffers.accum.mean()), f"{src}.iteration": ref.kp.iteration})
        return out
    live = oracle_ref.available() and (has_atmo or not cfg.get("atmo"))
    R = reference_outputs.load(request, reference, live=live, exact=tuple(f"{s}.blue_noise" for s in sources),
                               live_only=tuple(f"reference.{k}" for k in ("accum", "depth", "display", "blue_noise", "mean", "iteration")))
    launch = level_a_launcher()
    for src in (sky_sources(R) if cfg.get("atmo") else sources):
        if cfg.get("atmo"): sky_tables(scene, src)
        a = V.Renderer(scene, W, H, kp=make_kp(**cfg["kp"]), cam=cam)
        if ref_root is not None: a.params.p_oct.value = ref_root
        scene.reset_blue_noise(); launch(a, P)
        want = R.want(f"{src}.accum"); got = R.pick(f"{src}.accum", a.buffers.accum)
        frac = flipped_fraction(got, want)
        print(f"level A {cfg}, {src}: flipped {frac:.3g}, max |d| {np.abs(got - want).max():.3g}, ref mean {float(R.want(f'{src}.mean')):.6g}")
        assert float(R.want(f"{src}.mean")) > 1e-4 and frac <= MAX_FLIPPED
        assert flipped_fraction(R.pick(f"{src}.depth", a.buffers.depth)[:, None], R.want(f"{src}.depth")[:, None]) <= MAX_FLIPPED
        assert R.same(f"{src}.blue_noise", scene.d_blue_noise), "blue-noise state after the passes"
        assert float(a.buffers.cost.abs().max()) == 0.0
        dm = R.pick(f"{src}.display", a.buffers.display).view(np.uint8).reshape(-1, 4).astype(int)
        dr = R.want(f"{src}.display").view(np.uint8).reshape(-1, 4).astype(int)
        assert np.abs(dm - dr).max() <= 1
        assert a.kp.iteration == int(R.want(f"{src}.iteration")) == P


@pytest.mark.skipif(not os.path.exists(LEVEL_A), reason="volume_rt_kernel_b200.cubin not built")
def test_level_a_non_sampling_passes(dragon):
    """iteration >= max_interactions: buffers are only re-tonemapped; render == false: WHITE into the accumulator (:2248-2287)."""
    scene = make_scene(dragon)
    launch = level_a_launcher()
    a = V.Renderer(scene, 128, 64, kp=make_kp(ray_depth=1, max_interactions=2))
    if oracle_ref.available():
        a.params.p_oct.value = oracle_ref.RefOracle().build_octree(scene.h_volumes, 1)
    launch(a, 2); acc2 = a.buffers.accum.clone()
    launch(a, 2)
    assert torch.equal(acc2, a.buffers.accum)
    b = V.Renderer(scene, 128, 64, kp=make_kp(ray_depth=1, render=0), cam=a.cam)
    b.params.p_oct.value = a.params.p_oct.value
    launch(b, 1)
    assert torch.equal(b.buffers.accum, torch.ones_like(b.buffers.accum))
