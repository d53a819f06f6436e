// vpt_level_a.cu -- level (A) of the drop-in boundary (SURVEY 8(b)): ONE module entry `volume_rt_kernel` with the reference's
// own name, parameter list and launch contract, for the UNCHANGED Driver-API loader of the reference application
// (cuModuleLoad / cuLinkAddFile -> cuModuleGetFunction(&f, module, "volume_rt_kernel"), source/main.cpp:1221-1236) and its
// unchanged launch (grid (w/16+1, h/16+1), block (16,16), 0 bytes of dynamic shared memory, params[9]; main.cpp:1823-1827).
//
// Replaces source/render_kernel.cu:2216-2326 one launch for one launch.  It is a megakernel -- the host is not ours here, so
// there is no queue / workspace to run the wavefront stages on -- built from the very same device code as the wavefront path
// (walk_step, advance, advance_vol, begin_ratio_walk, closest_object, hg_sample: vpt_frame.cuh), one path per thread, with
// the warp voting between the tracking step and the integrator's bookkeeping like k_trace does.  What it still does better
// than the reference kernel: the octree is flattened once per CTA into shared memory (no 2520-byte pointer chase per step),
// the world->index affine of every volume is computed once per CTA instead of one 4x4 inverse per look-up, the depth pass
// reuses the integrator's first walk, later bounces that cannot change the sample are retired, and the blue-noise update is
// race-free: every CTA reads its jitter first, the LAST CTA to finish advances the 256x256 buffer (quirk Q6 made
// deterministic with the semantics "all reads before the update").
//
// Module hygiene: this translation unit is compiled to its own cubin (volume_rt_kernel_b200.cubin) and exports exactly one
// entry.  Inputs are the caller's own structures: the pointer-linked OCTNode tree is read in place.
#include "vpt_frame.cuh"

namespace vpt {

__device__ unsigned int g_done_ctas = 0;                        // CTAs that have read their blue-noise jitter and finished
__device__ VolumeRec g_vrec[VPT_OCT_MAX_VOLUMES];               // per-volume records of instanced scenes (rewritten by every CTA with identical values)

struct LevelAShared {
    FrameShared fs;
    FrameArgs   fa;
    const void* leaf_nodes[kOctLeaves];
    SphereRec   sph;
    TraceConsts tc;
    int         last_cta;
};

// the tail of the reference kernel for one pixel and one pass (render_kernel.cu:2262-2316), as k_resolve evaluates it
template <int kSky>
VPT_DEV void resolve_pixel(const FrameArgs& fa, const vpt_atmosphere& atmo, uint32_t idx, bool sampled, bool hit,
                           float3 ray_dir, float3 L, float3 beta, float depth, float tr, float3 env_pos)
{
    const vpt_kernel_params& kp = fa.kp;
    const vpt_camera& cam = fa.cam;
    float3* accum_buf = reinterpret_cast<float3*>(kp.accum_buffer);
    float3* cost_buf = reinterpret_cast<float3*>(kp.cost_buffer);
    float*  depth_buf = reinterpret_cast<float*>(kp.depth_buffer);
    float3 accum = f3(0.f), costv = f3(0.f); float depthv = 0.f;
    if (kp.iteration > 0 || !sampled) { accum = accum_buf[idx]; costv = cost_buf[idx]; depthv = depth_buf[idx]; }
    const uint32_t iteration = kp.iteration;
    float3 value = f3(1.0f);
    if (!sampled) { depth = .0f; tr = .0f; }
    else {
        if (!hit) { beta = f3(1.0f); L = f3(0.0f); depth = .0f; tr = .0f; }
        if constexpr (kSky == 1) {
            L += sample_atmosphere(atmo, kp.azimuth, kp.elevation, env_pos, ray_dir) * beta * kp.sky_mult * ld3(kp.sky_color);
        } else if constexpr (kSky == 2) {
            L += beta * sample_atmosphere(atmo, kp.azimuth, kp.elevation, env_pos, ray_dir);
        } else {
            const float4 texval = tex2D<float4>((cudaTextureObject_t)kp.env_tex,
                atan2f(ray_dir.z, ray_dir.x) * (float)(0.5 / 3.14159265358979323846) + 0.5f,
                acosf(fmaxf(fminf(ray_dir.y, 1.0f), -1.0f)) * (float)(1.0 / 3.14159265358979323846));
            L += f3(texval.x, texval.y, texval.z) * ld3(kp.sky_color) * beta * (1.0f / (4.0f * VPT_PI_F));
        }
        tr = fminf(tr, 1.0f);
        value = L;
    }
    // NaN / Inf guard (:2263): the pixel as the buffer holds it -- at iteration 0 the previous frame, which `accum` was not loaded with
    if (any_nan(value) || any_inf(value)) value = iteration == 0 ? accum_buf[idx] : accum;
    if (isnan(tr) || isinf(tr)) tr = 1.0f;

    float aof = 1 / cam.lens_radius;
    aof = clampf(aof, .0f, 3.402823466e+38F);
    if (cam.viz_dof) {
        if (depth > (cam.focus_dist + aof)) value = lerp3(value, f3(1.f, 0.f, 0.f), 0.5f);
        if (depth < (cam.focus_dist - aof)) value = lerp3(value, f3(0.f, 0.f, 1.f), 0.5f);
        if (depth > (cam.focus_dist - aof) && depth < (cam.focus_dist + aof)) value = lerp3(value, f3(0.f, 1.f, 0.f), 0.5f);
    }
    if (iteration == 0) { accum = value; costv = f3(0.f); depthv = depth; }
    else if (iteration < kp.max_interactions) {
        accum = accum + (value - accum) / (float)(iteration + 1);
        costv = costv + (f3(0.f) - costv) / (float)(iteration + 1);
        depthv = depthv + (depth - depthv) / (float)(iteration + 1);
    }
    accum_buf[idx] = accum; cost_buf[idx] = costv; depth_buf[idx] = depthv;

    const float aces_in[9]  = { 0.59719f, 0.35458f, 0.04823f, 0.07600f, 0.90834f, 0.01566f, 0.02840f, 0.13383f, 0.83777f };
    const float aces_out[9] = { 1.60475f, -0.53108f, -0.07367f, -0.10208f, 1.10813f, -0.00605f, -0.00327f, -0.07276f, 1.07602f };
    float3 val = mat3_mul(aces_in, accum);
    val = aces_fit(val);
    val = mat3_mul(aces_out, val) * kp.exposure_scale;
    const unsigned int r = (unsigned int)(255.0f * fminf(powf(fmaxf(val.x, 0.0f), (float)(1.0 / 2.2)), 1.0f));
    const unsigned int gg = (unsigned int)(255.0f * fminf(powf(fmaxf(val.y, 0.0f), (float)(1.0 / 2.2)), 1.0f));
    const unsigned int b = (unsigned int)(255.0f * fminf(powf(fmaxf(val.z, 0.0f), (float)(1.0 / 2.2)), 1.0f));
    reinterpret_cast<unsigned int*>(kp.display_buffer)[idx] = 0xff000000 | (r << 16) | (gg << 8) | b;
    reinterpret_cast<float4*>(kp.raw_buffer)[idx] = make_float4(val.x, val.y, val.z, tr);
}

} // namespace vpt

using namespace vpt;

extern "C" __global__ void __launch_bounds__(256, 2)
volume_rt_kernel(const vpt_camera cam, const vpt_light_list lights, const vpt_gpu_vdb* gpu_vdb, const vpt_sphere& sphere,
                 const vpt_geometry_list& geo_list, vpt_bvhnode* root_node, vpt_octnode* oct_root,
                 const vpt_atmosphere atmosphere, const vpt_kernel_params kernel_params)
{
    __shared__ LevelAShared sh;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x, nthreads = blockDim.x * blockDim.y;
    const vpt_kernel_params& kp = kernel_params;
    const int W = (int)kp.resolution.x, H = (int)kp.resolution.y;

    // ---- per-CTA scene staging straight from the caller's structures --------------------------------------------------------
    if (tid == 0) {
        SceneTables& sc = sh.fs.sc;
        sc.root_pmin[0] = oct_root->bbox.pmin.x; sc.root_pmin[1] = oct_root->bbox.pmin.y; sc.root_pmin[2] = oct_root->bbox.pmin.z;
        sc.root_pmax[0] = oct_root->bbox.pmax.x; sc.root_pmax[1] = oct_root->bbox.pmax.y; sc.root_pmax[2] = oct_root->bbox.pmax.z;
        sc.max_extinction = oct_root->max_extinction; sc.min_extinction = oct_root->min_extinction;
        sc.num_volumes = oct_root->num_volumes; sc.single_volume = (oct_root->num_volumes == 1) ? 1 : 0;
        sc.internal = nullptr; sc.leaf_list = nullptr; sc.leaf_indices = nullptr; sc.volumes = g_vrec; sc.leaf_nodes = sh.leaf_nodes;
        FrameArgs& fa = sh.fa;
        fa.cam = cam; fa.lights = lights; fa.kp = kernel_params; fa.sphere = &sphere; fa.scene = nullptr;
        fa.geom.width = W; fa.geom.height = H; fa.geom.local_rows = H; fa.geom.n_local = W * H; fa.geom.stripe_h = H > 0 ? H : 1; fa.geom.n_ranks = 1; fa.geom.rank = 0;
        fa.queue_dir = nullptr; fa.queue_id = nullptr; fa.queue_aux = nullptr; fa.thin_lens = cam.lens_radius != 0.0f ? 1 : 0;
        fa.bn_table = nullptr; fa.n_passes = 1; fa.passes_per_block = 1; fa.tiles_per_block = 1; fa.debug_flags = 0; fa.sched_min_lanes = 20; fa.queue_count = nullptr; fa.queue_head = nullptr;
        fa.planeA = fa.planeB = fa.planeC = nullptr;
        fa.planeD = reinterpret_cast<float4*>(kp.raw_buffer);          // env_pos scratch of the sphere branch: this pixel's raw_buffer entry, rewritten at the end
        fa.counters = nullptr; fa.cell_table = nullptr; fa.cell_nx = fa.cell_ny = fa.cell_nz = 0;
        sh.fs.vol0 = make_volume_rec(gpu_vdb[0]);
        sh.sph = load_sphere(&sphere);
        sh.tc.inv_max = 1.0f / sc.max_extinction;
        sh.tc.inv_mult = 1.0f / kp.density_mult;
        sh.tc.sigma_c = sc.min_extinction;
        sh.tc.sigma_r_inv = 1.0f / (sc.max_extinction - sh.tc.sigma_c);
        sh.tc.sun_dir = sun_direction(kp.azimuth, kp.elevation);
    }
    // internal nodes (root, 8, 64) from the pointer-linked tree, as k_prepare_scene flattens them
    for (int j = tid; j < kOctInternalNodes; j += nthreads) {
        const vpt_octnode* n = oct_root;
        bool exists = true;
        if (j >= 1 && j < 9) n = oct_ptr(oct_root->children[j - 1]);
        else if (j >= 9) {
            const vpt_octnode* p = oct_ptr(oct_root->children[(j - 9) >> 3]);
            if (p->num_volumes > 0) n = oct_ptr(p->children[(j - 9) & 7]); else exists = false;
        }
        OctInternal o;
        for (int a = 0; a < 3; ++a) { o.pmin[a] = 0.f; o.half[a] = 0.f; o.pmax[a] = 0.f; }
        o.child_empty = 0xffu; o.pad[0] = o.pad[1] = 0u;
        if (exists && n->num_volumes > 0) {
            o.pmin[0] = n->bbox.pmin.x; o.pmin[1] = n->bbox.pmin.y; o.pmin[2] = n->bbox.pmin.z;
            o.pmax[0] = n->bbox.pmax.x; o.pmax[1] = n->bbox.pmax.y; o.pmax[2] = n->bbox.pmax.z;
            const vpt_octnode* c0 = oct_ptr(n->children[0]);
            o.half[0] = c0->bbox.pmax.x; o.half[1] = c0->bbox.pmin.y; o.half[2] = c0->bbox.pmax.z;
            uint32_t mask = 0;
            for (int c = 0; c < 8; ++c) if (oct_ptr(n->children[c])->num_volumes == 0) mask |= 1u << c;
            o.child_empty = mask;
        }
        sh.fs.oct.node[j] = o;
    }
    const int n_vol = oct_root->num_volumes;
    if (n_vol > 1) {
        for (int l = tid; l < kOctLeaves; l += nthreads) {
            const void* leaf = nullptr;
            const vpt_octnode* p1 = oct_ptr(oct_root->children[l >> 6]);
            if (p1->num_volumes > 0) {
                const vpt_octnode* p2 = oct_ptr(p1->children[(l >> 3) & 7]);
                if (p2->num_volumes > 0) leaf = oct_ptr(p2->children[l & 7]);
            }
            sh.leaf_nodes[l] = leaf;
        }
        for (int v = tid; v < n_vol && v < VPT_OCT_MAX_VOLUMES; v += nthreads) g_vrec[v] = make_volume_rec(gpu_vdb[v]);
        __threadfence();
    }
    __syncthreads();

    const FrameShared& fs = sh.fs;
    const FrameArgs& fa = sh.fa;
    const SceneTables& sc = fs.sc;
    const SphereRec sph = sh.sph;
    const TraceConsts tc = sh.tc;

    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    const bool valid = x < W && y < H;
    const uint32_t idx = (uint32_t)y * (uint32_t)W + (uint32_t)x;
    const bool sampled = kp.render && kp.iteration < kp.max_interactions;

    PathState st;
    st.op = OP_IDLE;
    bool hit = false;
    if (valid && sampled) {
        st.lp = idx; st.pass = 0; st.qslot = 0;
        st.rng.init(idx, kp.iteration, 0u);
        // blue-noise jitter (:2238-2244), read before any CTA can advance the buffer (see the tail of this kernel)
        const float3* bn = reinterpret_cast<const float3*>(kp.blue_noise_buffer);
        const float3 bnv = bn[(y % 256) * 256 + (x % 256)];
        const float u = __fdividef(padd((float)x, bnv.x), (float)kp.resolution.x);
        const float v = __fdividef(padd((float)y, bnv.y), (float)kp.resolution.y);
        // thin-lens ray (camera::get_ray, camera.h:131-136): radical inverses of int(xi * 100) in bases 2 and 3, rejection loop
        float3 p;
        do {
            const float a = van_der_corput<2>(st.rng);
            const float b = van_der_corput<3>(st.rng);
            p = f3(pfma(a, 2.0f, -1.0f), pfma(b, 2.0f, -1.0f), 0.0f);
        } while (pfma(p.x, p.x, pmul(p.y, p.y)) >= 1.0f);
        const float3 rd = f3(pmul(cam.lens_radius, p.x), pmul(cam.lens_radius, p.y), 0.0f);
        const float3 offset = f3(pfma(cam.u.x, rd.x, pmul(cam.v.x, rd.y)), pfma(cam.u.y, rd.x, pmul(cam.v.y, rd.y)), pfma(cam.u.z, rd.x, pmul(cam.v.z, rd.y)));
        ++st.rng.k;                                                  // shutter-time draw
        st.org = f3(padd(cam.origin.x, offset.x), padd(cam.origin.y, offset.y), padd(cam.origin.z, offset.z));
        const float3 b = f3(psub(psub(pfma(cam.vertical.x, v, pfma(cam.horizontal.x, u, cam.lower_left_corner.x)), cam.origin.x), offset.x),
                            psub(psub(pfma(cam.vertical.y, v, pfma(cam.horizontal.y, u, cam.lower_left_corner.y)), cam.origin.y), offset.y),
                            psub(psub(pfma(cam.vertical.z, v, pfma(cam.horizontal.z, u, cam.lower_left_corner.z)), cam.origin.z), offset.z));
        st.dir = normalize(b);
        st.pos = st.org;
        st.beta = f3(1.0f); st.L = f3(.0f); st.alpha = .0f; st.depth = .0f;
        st.wpos = st.pos; st.wdir = st.dir; st.aux = f3(0.f); st.t = 0.f; st.distance = 0.f; st.trv = 1.f; st.T_c = 1.f;
        st.mi = false; st.first_walk = true; st.sphere_bounced = false; st.rd = 1; st.vd = 1; st.light_budget = 0; st.light_index = 0;
        st.mode = W_DELTA; st.exit_reason = EX_NONE; st.tr_kind = TR_SUN; st.sphere_free = false;
        st.obj_c = closest_object(sc, sph, st.pos, st.dir, st.tmin_c);
        st.have_closest = true;
        hit = st.obj_c != 0;
        if (hit) { st.phase = kp.integrator ? (int)VP_START : (int)PH_BOUNCE_TOP; st.op = OP_GLUE; }
    }

    // ---- the path: the warp votes between the tracking step and the bookkeeping, as k_trace does with its parked rays -------------
    uint32_t nlook = 0;
    for (;;) {
        const int nS = __popc(__ballot_sync(0xffffffffu, st.op == OP_STEP));
        const int nV = __popc(__ballot_sync(0xffffffffu, st.op != OP_STEP && st.op != OP_IDLE));
        if ((nS | nV) == 0) break;
        if (nV > 0 && (nV >= 12 || nS == 0 || nV > nS)) {
            if (st.op != OP_STEP && st.op != OP_IDLE) {
                if (st.op == OP_CLOSEST) {
                    st.obj_c = closest_object(sc, sph, st.pos, st.dir, st.tmin_c);
                    st.have_closest = true; st.op = OP_GLUE;
                }
                if (st.op == OP_GLUE) {
                    if (kp.integrator != 0) advance_vol(st, fs, fa, atmosphere, tc, sph);
                    else advance<false>(st, fs, fa, tc, sph);
                }
                if (st.op == OP_TRBEGIN) begin_ratio_walk(st, fs, tc, sph);
                if (st.op == OP_FINISH) st.op = OP_IDLE;
            }
            continue;
        }
        if (st.op == OP_STEP) walk_step<false>(st, fs, fa, tc, sph, nlook);
    }

    // ---- environment term, guard, running mean, tonemap, buffer writes (:1838-1850, :2262-2316) ----------------------------------------
    if (valid) {
        float3 env_pos = st.org;
        if (sampled && hit) {
            if (kp.integrator != 0) env_pos = length(st.beta) > 0.9999f ? st.org : st.pos;      // :1750
            else if (st.sphere_bounced) { const float4 D = fa.planeD[idx]; env_pos = f3(D.x, D.y, D.z); }
        }
        const bool sky_env = kp.environment_type == 0;
        if (kp.integrator != 0)  resolve_pixel<2>(fa, atmosphere, idx, sampled, hit, st.dir, st.L, st.beta, st.depth, st.alpha, env_pos);
        else if (sky_env)        resolve_pixel<1>(fa, atmosphere, idx, sampled, hit, st.dir, st.L, st.beta, st.depth, st.alpha, env_pos);
        else                     resolve_pixel<0>(fa, atmosphere, idx, sampled, hit, st.dir, st.L, st.beta, st.depth, st.alpha, env_pos);
    }

    // ---- blue-noise advance by the last CTA (:2319-2325 with the race removed) ---------------------------------------------------------
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        const unsigned total = gridDim.x * gridDim.y;
        sh.last_cta = (atomicAdd(&g_done_ctas, 1u) == total - 1u) ? 1 : 0;
    }
    __syncthreads();
    if (sh.last_cta) {
        __threadfence();
        float3* bn = reinterpret_cast<float3*>(kp.blue_noise_buffer);
        for (int i = tid; i < 256 * 256; i += nthreads) {
            if ((unsigned)i >= (unsigned)(W * H)) continue;            // the reference updates entry idx only for pixels that exist (idx < 65536 threads)
            float3 val = bn[i];
            val.x += (1.0f + sqrtf(5.0f)) / 2.0f; val.y += (1.0f + sqrtf(5.0f)) / 2.0f; val.z += (1.0f + sqrtf(5.0f)) / 2.0f;
            val.x = fmodf(val.x, 1.0f); val.y = fmodf(val.y, 1.0f); val.z = fmodf(val.z, 1.0f);
            bn[i] = val;
        }
        if (tid == 0) g_done_ctas = 0;
    }
}
