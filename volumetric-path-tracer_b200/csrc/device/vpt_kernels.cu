// vpt_kernels.cu -- sm_100a wavefront kernels that replace the reference megakernel
// `volume_rt_kernel` (source/render_kernel.cu:2216-2326), both integrators.
//
//   k_prepare_scene : GPU_VDB[] + OCTNode tree (the reference launch parameters) -> flat scene tables
//   k_bn_prepare    : per-chunk blue-noise jitter table + golden-ratio advance of the 256x256 buffer (race-free, quirk Q6)
//   k_generate      : one block per 32x4 pixel tile, all passes of the chunk: Philox stream, jitter, thin-lens ray,
//                     root/sphere test, draw-free prefix of the first tracking walk; misses write a 16-byte sample
//                     record, the rest are pushed into a warp-compacted ray queue (one atomic per warp)
//   k_trace<I, L>   : persistent; every lane owns three rays parked in shared memory (vpt_trace.cuh); I = integrator
//                     (0 direct, 1 volumetric path: vpt_trace_vol.cuh), L = lean instantiation for the common scene
//   k_resolve<S>    : per pixel, passes in order: environment term (S = 0 HDRI, 1 / 2 precomputed sky: vpt_atmosphere.cuh),
//                     NaN guard, running mean, ACES tonemap, display/raw/depth/cost writes (the tail of the reference kernel)
//   k_bn_advance, k_unpermute : blue-noise advance for non-sampling passes; stripe un-permutation after the multi-GPU gather
//
// Numerics: compiled with the reference's flags (--use_fast_math); decision-relevant expressions keep the reference
// build's operation order (read off its SASS) so a pixel's path is reproduced sample for sample (see vpt_math.cuh).
#include "vpt_frame.cuh"

namespace vpt {

// =====================================================================================================
// k_prepare_scene
// =====================================================================================================
// root == nullptr: the octree was built by vpt_octree_build, its flat tables already exist (`hdr` names them, any number of
// instances) and only the per-volume records -- which depend on the GPU_VDB[] array handed in at render time -- are made here.
// One kernel for both cases on purpose: the record arithmetic is then the very same machine code.
__global__ void k_prepare_scene(const vpt_gpu_vdb* __restrict__ vols, const vpt_octnode* __restrict__ root,
                                SceneTables* out, OctInternal* internal, uint2* leaf_list, int* leaf_indices,
                                VolumeRec* vrec, int max_volumes, const SceneTables hdr)
{
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nthreads = gridDim.x * blockDim.x;
    const int N = root ? root->num_volumes : hdr.num_volumes;
    if (!root && tid == 0) { SceneTables t = hdr; t.volumes = vrec; *out = t; }

    if (root && tid == 0) {
        out->root_pmin[0] = root->bbox.pmin.x; out->root_pmin[1] = root->bbox.pmin.y; out->root_pmin[2] = root->bbox.pmin.z;
        out->root_pmax[0] = root->bbox.pmax.x; out->root_pmax[1] = root->bbox.pmax.y; out->root_pmax[2] = root->bbox.pmax.z;
        out->max_extinction = root->max_extinction;
        out->min_extinction = root->min_extinction;
        out->num_volumes = N;
        out->single_volume = (N == 1) ? 1 : 0;
        out->internal = internal; out->leaf_list = leaf_list; out->leaf_indices = leaf_indices; out->volumes = vrec;
        out->leaf_nodes = nullptr;
    }

    // internal nodes: 0 = root, 1..8 = level 1, 9..72 = level 2
    for (int j = tid; root && j < kOctInternalNodes; j += nthreads) {
        const vpt_octnode* n = root;
        bool exists = true;
        if (j >= 1 && j < 9) { n = oct_ptr(root->children[j - 1]); }
        else if (j >= 9) {
            const int c1 = (j - 9) >> 3, c2 = (j - 9) & 7;
            const vpt_octnode* p = oct_ptr(root->children[c1]);
            if (p->num_volumes > 0) n = oct_ptr(p->children[c2]); else exists = false;
        }
        OctInternal o;
        for (int a = 0; a < 3; ++a) { o.pmin[a] = 0.f; o.half[a] = 0.f; o.pmax[a] = 0.f; }
        o.child_empty = 0xffu; o.pad[0] = o.pad[1] = 0u;
        if (exists && n->num_volumes > 0) {
            o.pmin[0] = n->bbox.pmin.x; o.pmin[1] = n->bbox.pmin.y; o.pmin[2] = n->bbox.pmin.z;
            o.pmax[0] = n->bbox.pmax.x; o.pmax[1] = n->bbox.pmax.y; o.pmax[2] = n->bbox.pmax.z;
            const vpt_octnode* c0 = oct_ptr(n->children[0]);       // child 0 = (x-, y+, z-)
            o.half[0] = c0->bbox.pmax.x; o.half[1] = c0->bbox.pmin.y; o.half[2] = c0->bbox.pmax.z;
            uint32_t mask = 0;
            for (int c = 0; c < 8; ++c) if (oct_ptr(n->children[c])->num_volumes == 0) mask |= 1u << c;
            o.child_empty = mask;
        }
        internal[j] = o;
    }

    // leaves: volume lists (instanced scenes); stride VPT_OCT_MAX_VOLUMES per leaf
    for (int l = tid; root && l < kOctLeaves; l += nthreads) {
        const int c1 = l >> 6, c2 = (l >> 3) & 7, c3 = l & 7;
        uint2 lst = make_uint2((uint32_t)l * VPT_OCT_MAX_VOLUMES, 0u);
        const vpt_octnode* p1 = oct_ptr(root->children[c1]);
        if (p1->num_volumes > 0) {
            const vpt_octnode* p2 = oct_ptr(p1->children[c2]);
            if (p2->num_volumes > 0) {
                const vpt_octnode* p3 = oct_ptr(p2->children[c3]);
                const int cnt = p3->num_volumes;
                lst.y = (uint32_t)cnt;
                if (N > 1) for (int i = 0; i < cnt; ++i) leaf_indices[lst.x + i] = p3->vol_indices[i];
            }
        }
        leaf_list[l] = lst;
    }

    // per-volume world->index affine
    for (int v = tid; v < N && v < max_volumes; v += nthreads) vrec[v] = make_volume_rec(vols[v]);
}

// =====================================================================================================
// k_generate
// =====================================================================================================
__global__ void __launch_bounds__(128)
k_generate(const FrameArgs fa)
{
    __shared__ FrameShared fs;
    __shared__ float vdc2[101], vdc3[101];                     // radical inverses of 0..100 in bases 2 and 3
    // the lens sampler only ever asks for vanDerCorput(int(xi * 100)): tabulate it with the reference's own loop
    if (threadIdx.x < 101) {
        { int n = threadIdx.x; float r = 0, denom = 1, inv = 1.f / 2; while (n) { denom *= 2; r = padd(r, __fdividef((float)(n % 2), denom)); n *= inv; } vdc2[threadIdx.x] = r; }
        { int n = threadIdx.x; float r = 0, denom = 1, inv = 1.f / 3; while (n) { denom *= 3; r = padd(r, __fdividef((float)(n % 3), denom)); n *= inv; } vdc3[threadIdx.x] = r; }
    }
    load_frame_shared(fs, fa.scene);
    const SceneTables& sc = fs.sc;
    const FrameGeom& g = fa.geom;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const SphereRec sph = load_sphere(fa.sphere);
    // one block = a run of 32x4 pixel tiles x a run of passes: enough (tile, pass) pairs per block to amortise the octree / table staging
    // above -- many passes of one tile when passes are fused, several tiles when the caller renders pass by pass; a small local frame
    // (multi-GPU shard, low resolution) splits the chunk's passes over blockIdx.z instead: see launch_generate
    const int tiles_x = (g.width + 31) / 32, n_tiles = tiles_x * ((g.local_rows + 3) / 4);
    for (int tile = blockIdx.x * fa.tiles_per_block; tile < min(n_tiles, (int)(blockIdx.x + 1) * fa.tiles_per_block); ++tile) {
    const int tile_y = tile / tiles_x, tile_x = tile - tile_y * tiles_x;
    const int x = tile_x * 32 + warp * 8 + (lane & 7);
    const int lr = tile_y * 4 + (lane >> 3);
    const int y = global_row(g, lr);
    const bool valid = (x < g.width) && (lr < g.local_rows) && (y < g.height);

    const int pass_begin = blockIdx.z * fa.passes_per_block;
    const int pass_end = min(fa.n_passes, pass_begin + fa.passes_per_block);
    // blue-noise jitter of each pass, from the per-chunk table written by k_bn_prepare; the value of the NEXT pass is requested one
    // iteration ahead (the load was the kernel's top stall: every pass started by waiting ~1 us for these 8 bytes)
    const int bn_index = valid ? (y % 256) * 256 + (x % 256) : 0;
    float2 bn_next = (valid && pass_begin < pass_end) ? __ldg(fa.bn_table + (size_t)pass_begin * 65536 + bn_index) : make_float2(0.f, 0.f);
    for (int pass = pass_begin; pass < pass_end; ++pass) {
    const float2 bnv = bn_next;
    if (valid && pass + 1 < pass_end) bn_next = __ldg(fa.bn_table + (size_t)(pass + 1) * 65536 + bn_index);
    bool hit = false;
    float3 org = f3(0.f), dir = f3(0.f, 0.f, 1.f);
    uint32_t kdraws = 0;
    int obj = 0; float t_min = 0.f;
    bool prestepped = false; float3 wstart = f3(0.f);
    const uint32_t lp = (uint32_t)lr * (uint32_t)g.width + (uint32_t)x;

    if (valid) {
        const vpt_kernel_params& kp = fa.kp;
        const vpt_camera& cam = fa.cam;
        const uint32_t idx = (uint32_t)y * (uint32_t)g.width + (uint32_t)x;
        Rng rng; rng.init(idx, kp.iteration + (uint32_t)pass, 0u);

        const float bnx = bnv.x, bny = bnv.y;
        const float u = __fdividef(padd((float)x, bnx), (float)kp.resolution.x);
        const float v = __fdividef(padd((float)y, bny), (float)kp.resolution.y);

        // thin-lens ray (reference camera::get_ray, camera.h:131-136).  The lens sample is drawn by a rejection loop on the pixel's
        // Philox stream BEFORE the ray exists -- but with a pinhole (lens_radius == 0) the sample is multiplied by zero: the ray
        // does not depend on it and the only thing the path needs from the loop is HOW MANY draws it consumed.  So the pinhole ray is
        // built first, the box / octree prefix below decides whether the sample can hit anything, and only the survivors run the
        // generator (70 % of the samples of the headline frame are misses and never touch it).  Bit-exactness: offset = u*0*p.x +
        // v*0*p.y is +-0; x + (+-0) == x and x - (+-0) == x for every x != 0, so lanes where a zero could meet a signed zero
        // (an origin or direction component that is exactly 0) take the literal order instead.
        const bool pinhole = (cam.lens_radius == 0.0f) && cam.origin.x != 0.0f && cam.origin.y != 0.0f && cam.origin.z != 0.0f;
        bool lens_pending = false;
        {
            const float3 b0 = f3(psub(pfma(cam.vertical.x, v, pfma(cam.horizontal.x, u, cam.lower_left_corner.x)), cam.origin.x),
                                 psub(pfma(cam.vertical.y, v, pfma(cam.horizontal.y, u, cam.lower_left_corner.y)), cam.origin.y),
                                 psub(pfma(cam.vertical.z, v, pfma(cam.horizontal.z, u, cam.lower_left_corner.z)), cam.origin.z));
            if (pinhole && b0.x != 0.0f && b0.y != 0.0f && b0.z != 0.0f) {
                org = ld3(cam.origin);
                dir = normalize(b0);
                lens_pending = true;
            } else {
                float3 p;
                do {
                    const float a = vdc2[int(rng.next() * 100)];
                    const float b = vdc3[int(rng.next() * 100)];
                    p = f3(pfma(a, 2.0f, -1.0f), pfma(b, 2.0f, -1.0f), 0.0f);
                } while (pfma(p.x, p.x, pmul(p.y, p.y)) >= 1.0f);
                const float3 rd = f3(pmul(cam.lens_radius, p.x), pmul(cam.lens_radius, p.y), 0.0f);
                const float3 offset = f3(pfma(cam.u.x, rd.x, pmul(cam.v.x, rd.y)), pfma(cam.u.y, rd.x, pmul(cam.v.y, rd.y)), pfma(cam.u.z, rd.x, pmul(cam.v.z, rd.y)));
                ++rng.k;                                                 // shutter time draw: consumed, value unused by the path
                org = f3(padd(cam.origin.x, offset.x), padd(cam.origin.y, offset.y), padd(cam.origin.z, offset.z));
                dir = normalize(f3(psub(b0.x, offset.x), psub(b0.y, offset.y), psub(b0.z, offset.z)));
                kdraws = rng.k;
            }
        }

        const bool sphere_clear = line_misses_sphere(sph, org, dir);   // then sphere::intersect is known to fail: skip it
        if (sphere_clear) { float tmax1; obj = aabb_intersect(sc.root_pmin, sc.root_pmax, org, dir, t_min, tmax1) ? 1 : 0; }
        else obj = closest_object(sc, sph, org, dir, t_min);
        hit = (obj != 0);

        // Draw-free prefix of the first delta walk: until the ray reaches a non-empty octree leaf the reference's `sample`
        // only hops over empty nodes (no random number is consumed).  Run those hops here, at full warp width; a ray that
        // leaves the box without ever meeting a populated leaf contributes exactly what a miss does and never enters the
        // queue, the others are queued at the position where stepping really starts.  (Pinhole camera and a ray whose line
        // provably misses the sphere only; everything else takes the generic route.)
        if (obj == 1 && kp.ray_depth >= 1 && kp.volume_depth >= 1 && cam.lens_radius == 0.0f && sphere_clear) {
            float3 p = madd3(org, dir, padd(t_min, VPT_EPS));
            int leaf = -2;
            if (!aabb_contains(sc.root_pmin, sc.root_pmax, p)) leaf = -1;
            for (int it = 0; it < 256 && leaf == -2; ++it) leaf = oct_locate_or_skip<true>(fs.oct, sc, p, dir);
            if (leaf == -1) {                                    // walked out through empty space: sample == miss sample
                hit = false;
                if (kp.integrator != 0) dir = normalize(dir);    // vol_integrator renormalises after a box hit (:1747)
            }
            else if (leaf >= 0) { prestepped = true; wstart = p; }
            // leaf == -2 after 256 hops: leave it to the generic route
        }

        if (hit && lens_pending) {
            // the rejection loop, for its draw count only (2 per trial + the shutter-time draw)
            float px, py;
            do {
                px = pfma(vdc2[int(rng.next() * 100)], 2.0f, -1.0f);
                py = pfma(vdc3[int(rng.next() * 100)], 2.0f, -1.0f);
            } while (pfma(px, px, pmul(py, py)) >= 1.0f);
            kdraws = rng.k + 1u;
        }

        if (!hit) {
            const size_t s = (size_t)pass * g.n_local + lp;
            // 16-byte miss record: direction + sentinel (L = 0, beta = 1, depth = 0, tr = 0 are implied; planes B/C untouched)
            fa.planeA[s] = make_float4(dir.x, dir.y, dir.z, __uint_as_float(kMissSentinel));
            if (fa.planeD) fa.planeD[s] = make_float4(org.x, org.y, org.z, 0.f);
        }
    }

    // warp-compacted push: one atomic per warp, records contiguous per 8x4 pixel tile
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (m) {
        unsigned base = 0;
        if (lane == __ffs(m) - 1) base = atomicAdd(fa.queue_count, __popc(m));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        if (hit) {
            // 24-byte record (+16 B origin when the lens is not a pinhole): direction + entry distance, ids + RNG position
            const unsigned slot = base + __popc(m & ((1u << lane) - 1u));
            fa.queue_dir[slot] = make_float4(dir.x, dir.y, dir.z, t_min);
            fa.queue_id[slot] = make_uint2(ray_pixel_word(g, lr, x), (uint32_t)pass | (kdraws << 6) | ((uint32_t)obj << 16) | ((uint32_t)prestepped << 18));
            if (prestepped) fa.queue_aux[slot] = make_float4(wstart.x, wstart.y, wstart.z, 0.f);      // where stepping starts
            else if (fa.thin_lens) fa.queue_aux[slot] = make_float4(org.x, org.y, org.z, 0.f);   // thin lens: per-ray origin
        }
    }
    }   // pass loop
    }   // tile loop
}


// =====================================================================================================
// k_resolve
// =====================================================================================================
// kSky 1: direct integrator with environment_type == 0 (Bruneton sky lookup, `atmo` is the caller's AtmosphereParameters);
// kSky 2: volumetric path integrator, which always ends on the sky (:1752); kSky 0: HDRI environment -- that variant
// takes a 16-byte dummy so it keeps its small parameter block and register budget.
struct NoSky { int pad[4]; };
struct PeerFlagPtrs { unsigned long long* p[kMaxPeers]; };

// The guard's load of the previous frame, out of line: inlined, it costs the HDRI variant 5 registers (32 -> 37) for a branch
// that finite samples never take.
__device__ __noinline__ float3 stale_pixel(const float3* accum_buf, uint32_t lp) { return accum_buf[lp]; }

template <int kSky>
__global__ void __launch_bounds__(256)
k_resolve(const FrameArgs fa, const typename std::conditional<kSky != 0, vpt_atmosphere, NoSky>::type atmo,
          const int n_passes, const int sampled, const int write_display, const PeerFrames peers)
{
    const FrameGeom& g = fa.geom;
    const vpt_kernel_params& kp = fa.kp;
    const vpt_camera& cam = fa.cam;
    const uint32_t lp = blockIdx.x * blockDim.x + threadIdx.x;
    if (lp >= (uint32_t)g.n_local) return;
    const int lr = lp / g.width;
    const int y = global_row(g, lr);
    if (y >= g.height) return;

    float3* accum_buf = reinterpret_cast<float3*>(kp.accum_buffer);
    float3* cost_buf = reinterpret_cast<float3*>(kp.cost_buffer);
    float*  depth_buf = reinterpret_cast<float*>(kp.depth_buffer);
    // output buffers are indexed by local pixel (== global pixel index for a single rank)
    float3 accum = f3(0.f), costv = f3(0.f); float depthv = 0.f;
    const bool have_prev = kp.iteration > 0;
    if (have_prev || !sampled) { accum = accum_buf[lp]; costv = cost_buf[lp]; depthv = depth_buf[lp]; }
    float tr = .0f;

    // one pass of the running mean; A (and B, C for a hit sample) are the pass's plane records, loaded by the caller
    auto one_pass = [&](const int p, const float4 A, const float4 B, const float4 C) {
        const uint32_t iteration = kp.iteration + (uint32_t)p;
        float3 value = f3(1.0f);                                // WHITE when nothing is sampled (:2248)
        float depth = .0f;
        tr = .0f;
        if (sampled) {
            const size_t s = (size_t)p * g.n_local + lp;
            const float3 ray_dir = f3(A.x, A.y, A.z);
            float3 beta = f3(1.0f), L = f3(0.0f);
            if (__float_as_uint(A.w) != kMissSentinel) {          // hit sample: the trace kernel wrote all three planes
                beta = f3(C.x, C.y, C.z); L = f3(B.x, B.y, B.z);
                depth = B.w; tr = A.w;
            }
            if constexpr (kSky == 1) {
                // precomputed sky seen from env_pos along the final direction (:1838-1841)
                const float4 D = fa.planeD[s];
                L += sample_atmosphere(atmo, kp.azimuth, kp.elevation, f3(D.x, D.y, D.z), ray_dir) * beta * kp.sky_mult * ld3(kp.sky_color);
            } else if constexpr (kSky == 2) {
                const float4 D = fa.planeD[s];                       // env_pos or the last path position (:1750-1752)
                L += beta * sample_atmosphere(atmo, kp.azimuth, kp.elevation, f3(D.x, D.y, D.z), ray_dir);
            } else {
                const float4 texval = tex2D<float4>((cudaTextureObject_t)kp.env_tex,
                    atan2f(ray_dir.z, ray_dir.x) * (float)(0.5 / 3.14159265358979323846) + 0.5f,
                    acosf(fmaxf(fminf(ray_dir.y, 1.0f), -1.0f)) * (float)(1.0 / 3.14159265358979323846));
                L += f3(texval.x, texval.y, texval.z) * ld3(kp.sky_color) * beta * (1.0f / (4.0f * VPT_PI_F));   // isotropic() returns the folded constant
            }
            tr = fminf(tr, 1.0f);
            value = L;
        }
        // NaN / Inf guard (:2263-2264): the pixel as the buffer holds it.  At iteration 0 that is the previous frame, which
        // `accum` was not loaded with; the load stays in this branch so finite samples do not pay for it
        if (any_nan(value) || any_inf(value)) value = iteration == 0 ? stale_pixel(accum_buf, lp) : accum;
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
    };
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    {
        for (int p = 0; p < n_passes; ++p) {
            float4 A = zero4, B = zero4, C = zero4;
            if (sampled) {
                const size_t s = (size_t)p * g.n_local + lp;
                A = fa.planeA[s];
                if (__float_as_uint(A.w) != kMissSentinel) { B = fa.planeB[s]; C = fa.planeC[s]; }
            }
            one_pass(p, A, B, C);
        }
    }
    accum_buf[lp] = accum; cost_buf[lp] = costv; depth_buf[lp] = depthv;

    if (write_display) {
        const float aces_in[9]  = { 0.59719f, 0.35458f, 0.04823f, 0.07600f, 0.90834f, 0.01566f, 0.02840f, 0.13383f, 0.83777f };
        const float aces_out[9] = { 1.60475f, -0.53108f, -0.07367f, -0.10208f, 1.10813f, -0.00605f, -0.00327f, -0.07276f, 1.07602f };
        float3 val = mat3_mul(aces_in, accum);
        val = aces_fit(val);
        val = mat3_mul(aces_out, val) * kp.exposure_scale;
        const unsigned int r = (unsigned int)(255.0f * fminf(powf(fmaxf(val.x, 0.0f), (float)(1.0 / 2.2)), 1.0f));
        const unsigned int gg = (unsigned int)(255.0f * fminf(powf(fmaxf(val.y, 0.0f), (float)(1.0 / 2.2)), 1.0f));
        const unsigned int b = (unsigned int)(255.0f * fminf(powf(fmaxf(val.z, 0.0f), (float)(1.0 / 2.2)), 1.0f));
        const unsigned int word = 0xff000000 | (r << 16) | (gg << 8) | b;
        reinterpret_cast<unsigned int*>(kp.display_buffer)[lp] = word;
        reinterpret_cast<float4*>(kp.raw_buffer)[lp] = make_float4(val.x, val.y, val.z, tr);
        if (peers.n > 0 && peers.display[0]) {
            const size_t gp = (size_t)y * g.width + (lp - (uint32_t)lr * (uint32_t)g.width);
            #pragma unroll
            for (int p = 0; p < kMaxPeers; ++p) if (p < peers.n) peers.display[p][gp] = word;
        }
    }
    // multi-GPU exchange fused into the producer: this pixel's running mean goes to its global position in every rank's full frame
    if (peers.n > 0 && peers.accum[0]) {
        const size_t gp = (size_t)y * g.width + (lp - (uint32_t)lr * (uint32_t)g.width);
        #pragma unroll
        for (int p = 0; p < kMaxPeers; ++p) if (p < peers.n) { float* a = peers.accum[p] + 3 * gp; a[0] = accum.x; a[1] = accum.y; a[2] = accum.z; }
    }
}

__global__ void k_peer_signal(PeerFlagPtrs fl, int n, int rank, int which, unsigned long long epoch)
{
    const int p = threadIdx.x;
    if (p >= n) return;
    __threadfence_system();                                    // everything this stream stored before (peer frames included) ...
    unsigned long long* slot = fl.p[p] + which * kPeerFlagStride + rank;
    asm volatile("st.release.sys.global.u64 [%0], %1;" :: "l"(slot), "l"(epoch) : "memory");   // ... is visible before the flag
}

__global__ void k_peer_wait(unsigned long long* local, int n, int which, unsigned long long epoch)
{
    const int p = threadIdx.x;
    if (p >= n) return;
    const unsigned long long* slot = local + which * kPeerFlagStride + p;
    unsigned long long t0 = 0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        unsigned long long v; asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(slot) : "memory");
        if (v >= epoch) break;
        unsigned long long t1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > 10000000000ull) { atomicAdd(local + 2 * kPeerFlagStride, 1ull); break; }     // 10 s: a rank is gone -- report, do not hang the GPU
        __nanosleep(200);
    }
}

// =====================================================================================================
// k_bn_advance: blue-noise buffer += golden ratio (mod 1), `n` passes worth (:2319-2325)
// =====================================================================================================
// Per-chunk jitter table: table[p][i] = (x, y) of blue-noise entry i after p advances, p = 0..np-1; the buffer
// itself is left advanced by `np` passes.  One launch replaces the per-thread replay in k_generate.
// `limit` = min(W*H, 65536): the reference advances entry idx = y*W + x from the thread of pixel (x, y), so a frame of fewer than
// 65536 pixels leaves the entries beyond W*H untouched (they are still READ as jitter through (y % 256) * 256 + x % 256).
__global__ void k_bn_prepare(float3* bn, float2* table, int np, int limit, unsigned* queue_counters)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx == 0 && queue_counters) { queue_counters[0] = 0u; queue_counters[1] = 0u; }   // first kernel of a round: also resets the ray queue (count, head)
    if (idx >= 256 * 256) return;
    float3 val = bn[idx];
    if (idx >= limit) {
        for (int i = 0; i < np; ++i) table[(size_t)i * 65536 + idx] = make_float2(val.x, val.y);
        return;
    }
    for (int i = 0; i < np; ++i) {
        table[(size_t)i * 65536 + idx] = make_float2(val.x, val.y);
        val.x += (1.0f + sqrtf(5.0f)) / 2.0f; val.y += (1.0f + sqrtf(5.0f)) / 2.0f; val.z += (1.0f + sqrtf(5.0f)) / 2.0f;
        val.x = fmodf(val.x, 1.0f); val.y = fmodf(val.y, 1.0f); val.z = fmodf(val.z, 1.0f);
    }
    bn[idx] = val;
}

__global__ void k_bn_advance(float3* bn, int n, int limit)
{
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 256 * 256 || idx >= limit) return;
    float3 val = bn[idx];
    for (int i = 0; i < n; ++i) {
        val.x += (1.0f + sqrtf(5.0f)) / 2.0f; val.y += (1.0f + sqrtf(5.0f)) / 2.0f; val.z += (1.0f + sqrtf(5.0f)) / 2.0f;
        val.x = fmodf(val.x, 1.0f); val.y = fmodf(val.y, 1.0f); val.z = fmodf(val.z, 1.0f);
    }
    bn[idx] = val;
}

// gather permutation for the multi-GPU path: rank-contiguous stripes -> full frame
__global__ void k_unpermute(const uint8_t* __restrict__ gathered, uint8_t* __restrict__ full, FrameGeom g, int elem_bytes)
{
    // one thread per (rank, local pixel) element of 4-byte words
    const size_t words_per_px = elem_bytes / 4;
    const size_t total = (size_t)g.n_ranks * g.n_local * words_per_px;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t px = i / words_per_px, w = i - px * words_per_px;
        const int rank = (int)(px / g.n_local);
        const size_t lp = px - (size_t)rank * g.n_local;
        const int lr = (int)(lp / g.width), x = (int)(lp - (size_t)lr * g.width);
        const int s = lr / g.stripe_h;
        const int y = (s * g.n_ranks + rank) * g.stripe_h + (lr - s * g.stripe_h);
        if (y < g.height)
            reinterpret_cast<uint32_t*>(full)[((size_t)y * g.width + x) * words_per_px + w] = reinterpret_cast<const uint32_t*>(gathered)[i];
    }
}

// =====================================================================================================
// host-callable launchers
// =====================================================================================================
cudaError_t launch_prepare_scene(const vpt_gpu_vdb* vols, const vpt_octnode* root, SceneTables* out, OctInternal* internal,
                                 uint2* leaf_list, int* leaf_indices, VolumeRec* vrec, int max_volumes, cudaStream_t s)
{
    SceneTables none; memset(&none, 0, sizeof(none));
    k_prepare_scene<<<4, 256, 0, s>>>(vols, root, out, internal, leaf_list, leaf_indices, vrec, max_volumes, none);
    return cudaGetLastError();
}

cudaError_t launch_prepare_volumes(const vpt_gpu_vdb* vols, const SceneTables& hdr, SceneTables* out, VolumeRec* vrec, cudaStream_t s)
{
    const int blocks = hdr.num_volumes > 4096 ? 32 : 4;
    k_prepare_scene<<<blocks, 256, 0, s>>>(vols, nullptr, out, nullptr, nullptr, nullptr, vrec, hdr.num_volumes, hdr);
    return cudaGetLastError();
}

cudaError_t launch_generate(const FrameArgs& fa, int n_passes, cudaStream_t s)
{
    FrameArgs a = fa; a.n_passes = n_passes;
    // one block = a run of 32x4 pixel tiles x a run of passes.  Keep >= ~8 waves of blocks (148 SMs x 7 resident blocks) so the tail of the
    // grid does not idle the SMs when the local frame is small; never fewer than 4 (tile, pass) pairs per block (amortises the table
    // staging: one pass per call used to spend half of this kernel on it).
    int ppb = n_passes;
    const long long tiles = (long long)((fa.geom.width + 31) / 32) * ((fa.geom.local_rows + 3) / 4);
    while (ppb > 4 && tiles * ((n_passes + ppb - 1) / ppb) < 8288) ppb = (ppb + 1) / 2;
    int tpb = 1;
    while (ppb * tpb < 4 && tiles / (tpb * 2) >= 2368) tpb *= 2;
    a.passes_per_block = ppb; a.tiles_per_block = tpb;
    dim3 grid((unsigned)((tiles + tpb - 1) / tpb), 1, (unsigned)((n_passes + ppb - 1) / ppb));
    k_generate<<<grid, 128, 0, s>>>(a);
    return cudaGetLastError();
}

static size_t trace_smem_bytes(int slots) { return (size_t)kTraceWarps * kRayWords * 32 * slots * sizeof(float); }

// atm != null selects the volumetric path integrator variant (Kernel_params.integrator != 0); lean selects the instantiation
// without multi-volume lists, emission walk and point lights (the caller guarantees none of them is in play); slots = rays per lane
template <int kInteg, bool kLean, int kSlots>
static cudaError_t launch_trace_t(const FrameArgs& fa, const vpt_atmosphere* atm, int n_ctas, cudaStream_t s)
{
    if constexpr (kInteg != 0) k_trace<kInteg, kLean, kSlots><<<n_ctas, kTraceThreads, trace_smem_bytes(kSlots), s>>>(fa, *atm);
    else                       k_trace<kInteg, kLean, kSlots><<<n_ctas, kTraceThreads, trace_smem_bytes(kSlots), s>>>(fa, NoAtmo{});
    return cudaGetLastError();
}

cudaError_t launch_trace(const FrameArgs& fa, const vpt_atmosphere* atm, bool lean, int slots, int n_ctas, cudaStream_t s)
{
    if (atm) return launch_trace_t<1, false, 3>(fa, atm, n_ctas, s);
    if (fa.cell_table) {                                                        // the host only sets it for lean scenes
        k_trace<0, true, 2, true><<<n_ctas, kTraceThreads, trace_smem_bytes(2), s>>>(fa, NoAtmo{});
        return cudaGetLastError();
    }
    if (slots == 2) return lean ? launch_trace_t<0, true, 2>(fa, nullptr, n_ctas, s) : launch_trace_t<0, false, 2>(fa, nullptr, n_ctas, s);
    return lean ? launch_trace_t<0, true, 3>(fa, nullptr, n_ctas, s) : launch_trace_t<0, false, 3>(fa, nullptr, n_ctas, s);
}

// Once per context (= per device): opt the instantiations into their dynamic shared memory and record how many CTAs of each fit
// on an SM.  The attribute is a per-device property of the function, so this must not be a process-wide static.
template <int kInteg, bool kLean, int kSlots>
static cudaError_t trace_init_t(int* max_ctas)
{
    cudaError_t e = cudaFuncSetAttribute(k_trace<kInteg, kLean, kSlots>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trace_smem_bytes(kSlots));
    if (e != cudaSuccess) return e;
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(max_ctas, k_trace<kInteg, kLean, kSlots>, kTraceThreads, trace_smem_bytes(kSlots));
}

static size_t brick_smem_bytes() { return (size_t)kBrickThreads * kBrickBytes; }

cudaError_t trace_kernels_init(int max_ctas[7])
{
    {
        cudaError_t e0 = cudaFuncSetAttribute(k_trace<0, true, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trace_smem_bytes(2));
        if (e0 == cudaSuccess) e0 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_ctas[6], k_trace<0, true, 2, true>, kTraceThreads, trace_smem_bytes(2));
        if (e0 != cudaSuccess) return e0;
    }
    cudaError_t e = trace_init_t<0, false, 3>(&max_ctas[0]);
    if (e == cudaSuccess) e = trace_init_t<0, true, 3>(&max_ctas[1]);
    if (e == cudaSuccess) e = trace_init_t<1, false, 3>(&max_ctas[2]);
    if (e == cudaSuccess) e = trace_init_t<0, false, 2>(&max_ctas[4]);
    if (e == cudaSuccess) e = trace_init_t<0, true, 2>(&max_ctas[5]);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_trace_brick, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)brick_smem_bytes());
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&max_ctas[3], k_trace_brick, kBrickThreads, brick_smem_bytes());
    return e;
}

cudaError_t launch_sampler_compare(unsigned long long tex, const float* pool, const int dims[3], int n, unsigned seed, double* d_out12, cudaStream_t s)
{
    BrickArgs ba;
    ba.pool = pool; ba.dimx = dims[0]; ba.dimy = dims[1]; ba.dimz = dims[2];
    ba.nbx = (dims[0] + 3) / 4; ba.nby = (dims[1] + 3) / 4; ba.nbz = (dims[2] + 3) / 4;
    k_sampler_compare<<<592, 256, 0, s>>>((cudaTextureObject_t)tex, ba, n, seed, d_out12);
    return cudaGetLastError();
}

cudaError_t launch_trace_brick(const FrameArgs& fa, const float* pool, const int dims[3], int n_ctas, cudaStream_t s)
{
    BrickArgs ba;
    ba.pool = pool; ba.dimx = dims[0]; ba.dimy = dims[1]; ba.dimz = dims[2];
    ba.nbx = (dims[0] + 3) / 4; ba.nby = (dims[1] + 3) / 4; ba.nbz = (dims[2] + 3) / 4;
    k_trace_brick<<<n_ctas, kBrickThreads, brick_smem_bytes(), s>>>(fa, ba);
    return cudaGetLastError();
}

cudaError_t launch_resolve(const FrameArgs& fa, const vpt_atmosphere* sky, int n_passes, int sampled, int write_display, const PeerFrames* peers, cudaStream_t s)
{
    const int threads = 256;
    const int blocks = (fa.geom.n_local + threads - 1) / threads;
    const PeerFrames pf = peers ? *peers : PeerFrames{};
    // (tried for frames of less than two waves of blocks -- multi-GPU shards: fetching the records of four passes at once before the
    // order-dependent running mean; slower there too, 0.28 vs 0.21 ms on a 1/8 shard of the 1080p frame)
    if (sky && fa.kp.integrator != 0) k_resolve<2><<<blocks, threads, 0, s>>>(fa, *sky, n_passes, sampled, write_display, pf);
    else if (sky)                     k_resolve<1><<<blocks, threads, 0, s>>>(fa, *sky, n_passes, sampled, write_display, pf);
    else                              k_resolve<0><<<blocks, threads, 0, s>>>(fa, NoSky{}, n_passes, sampled, write_display, pf);
    return cudaGetLastError();
}

cudaError_t launch_peer_signal(unsigned long long* const peer_flags[kMaxPeers], int n, int rank, int which, unsigned long long epoch, cudaStream_t s)
{
    PeerFlagPtrs fl; for (int p = 0; p < kMaxPeers; ++p) fl.p[p] = p < n ? peer_flags[p] : nullptr;
    k_peer_signal<<<1, 32, 0, s>>>(fl, n, rank, which, epoch);
    return cudaGetLastError();
}

cudaError_t launch_peer_wait(unsigned long long* local_flags, int n, int which, unsigned long long epoch, cudaStream_t s)
{
    k_peer_wait<<<1, 32, 0, s>>>(local_flags, n, which, epoch);
    return cudaGetLastError();
}

cudaError_t launch_bn_prepare(void* bn, float2* table, int np, int limit, unsigned* queue_counters, cudaStream_t s)
{
    k_bn_prepare<<<256, 256, 0, s>>>(reinterpret_cast<float3*>(bn), table, np, limit, queue_counters);
    return cudaGetLastError();
}

cudaError_t launch_bn_advance(void* bn, int n, int limit, cudaStream_t s)
{
    k_bn_advance<<<256, 256, 0, s>>>(reinterpret_cast<float3*>(bn), n, limit);
    return cudaGetLastError();
}

cudaError_t launch_unpermute(const void* gathered, void* full, const FrameGeom& g, int elem_bytes, cudaStream_t s)
{
    k_unpermute<<<1184, 256, 0, s>>>(reinterpret_cast<const uint8_t*>(gathered), reinterpret_cast<uint8_t*>(full), g, elem_bytes);
    return cudaGetLastError();
}

} // namespace vpt
