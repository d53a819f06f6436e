"""Boundary ABI: the library loads on a CPU-only host, exports every symbol include/vpt_b200.h declares,
and the struct layouts agree between the C header, the ctypes mirror and (when present) the reference."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    import vpt_b200 as V
    from vpt_b200 import _native as N
    hdr = open(os.path.join(ROOT, "include", "vpt_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(vpt_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(N.lib, name), f"libvpt_b200.so does not export {name}"
    assert sorted(N.EXPORTED_SYMBOLS) == declared
    assert b"sm_100a" in N.lib.vpt_version()


def test_struct_sizes_match_between_c_and_ctypes():
    from vpt_b200 import _native as N
    out = (C.c_size_t * 12)()
    n = N.lib.vpt_abi_sizes(out, 12)
    assert n == 12
    assert list(out) == N.ABI_SIZES == [C.sizeof(s) for s in N.ABI_STRUCTS]


def test_kernel_params_offsets():
    from vpt_b200 import _native as N
    kp = N.Kernel_params
    expect = dict(resolution=8, exposure_scale=16, display_buffer=24, raw_buffer=32, blue_noise_buffer=40, emission_texture=48,
                  emission_scale=56, density_color_texture=64, iteration=72, accum_buffer=80, depth_buffer=88, max_interactions=96,
                  ray_depth=100, volume_depth=104, phase_g1=112, albedo=124, extinction=136, tr_depth=160, density_mult=164,
                  environment_type=168, azimuth=172, sun_color=180, sky_color=192, sun_mult=204, sky_mult=208, energy_inject=216,
                  env_tex=224, env_marginal_int=280, cost_buffer=296, integrator=304)
    for k, off in expect.items():
        assert getattr(kp, k).offset == off, k
    assert N.camera.lens_radius.offset == 96 and N.camera.viz_dof.offset == 100
    assert N.OCTNode.bbox.offset == 2496 and N.OCTNode.children.offset == 2424 and N.GPU_VDB.xform.offset == 80


def test_no_gpu_means_loud_failure_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from vpt_b200 import _native as N
    ctx = C.c_void_p(0)
    assert N.lib.vpt_create(C.byref(ctx)) == -2          # VPT_ERR_CUDA
    assert b"no CPU path" in N.lib.vpt_last_error(None)


def test_layouts_against_reference_headers(request):
    """sizeof/offsetof as the reference's own headers declare them: measured by oracle/ref_layouts.cu (`make -C oracle ref`)
    where the reference build exists, else as recorded under tests/golden/reference."""
    import numpy as np
    import reference_outputs
    path = os.path.join(ROOT, "oracle", "_ref", "abi_layouts.txt")
    R = reference_outputs.load(request, lambda: dict(layouts=np.array([int(x) for x in open(path).read().split()], dtype=np.int64)),
                               live=os.path.exists(path))
    out = [int(x) for x in R.want("layouts")]
    from vpt_b200 import _native as N
    assert out[:12] == N.ABI_SIZES
    assert out[12:] == [304, 216, 2496, 424]
