/*
 * ref_harness.cpp — TEST INFRASTRUCTURE (oracle side).  Headless CPU harness that
 * runs the reference's OWN code for the hot path:
 *   - scene loading:  reference Scene (src/scene/scene.cpp, compiled in place)
 *   - BVH build:      reference Bvh::BuildCPU (src/bvh.cpp, compiled in place)
 *   - env map:        reference LoadHDR (src/loaders/hdr_loader.cpp)
 *   - frame schedule: reference Integrator::Integrate (src/integrator/integrator.cpp)
 *   - kernels:        reference src/kernels/cl/*.cl compiled for the host through
 *                     oracle/ref_shim (see kernel_tu.cpp / clshim.h)
 * The only thing replaced is the OpenCL runtime: RefCpuIntegrator below stands in
 * for CLPathTraceIntegrator + CLContext (src/integrator/cl_pt_integrator.cpp,
 * src/gpu_wrappers/cl_context.cpp): it owns the same buffers
 * (cl_pt_integrator.cpp:194-249), binds the same arguments in the same order
 * (:261-363, :497-684) and "enqueues" each kernel over width*height work-items.
 * ResolveRadiance writes to a host RGBA32F image instead of a GL texture.
 *
 * Built only where /root/reference exists (oracle/build_ref.py) into
 * oracle/_ref/libref.so.  Nothing in the product path links or loads this.
 */
#include "integrator/integrator.hpp"
#include "bvh.hpp"
#include "scene/scene.hpp"
#include "loaders/image_loader.hpp"
#include "utils/blue_noise_sampler.hpp"

#include <unistd.h>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <string>
#include <vector>

typedef unsigned int uint;

// launchers exported by the kernel translation units (oracle/ref_shim/kernel_tu.cpp)
extern "C" {
void refk_RayGeneration_std(size_t, uint, uint, const void*, void*, void*, void*, void*, void*, void*, void*, void*, void*);
void refk_TraceBvh_std(size_t, void*, void*, void*, void*, void*);
void refk_TraceBvh_shadow(size_t, void*, void*, void*, void*, void*);
#define REF_DECL_MISS(s) void refk_Miss_##s(size_t, void*, void*, void*, void*, void*, float*, int, int, void*);
#define REF_DECL_HIT(s) void refk_HitSurface_##s(size_t, void*, void*, void*, void*, void*, void*, void*, void*, void*, void*, \
    uint, uint, uint, void*, const void*, void*, void*, void*, void*, void*, void*, void*, void*, void*, void*, void*, void*);
REF_DECL_MISS(std) REF_DECL_MISS(wf)
REF_DECL_HIT(std) REF_DECL_HIT(wf) REF_DECL_HIT(bn) REF_DECL_HIT(wfbn)
void refk_AccumulateDirectSamples_std(size_t, void*, void*, void*, void*, void*);
void refk_ClearCounter_std(size_t, void*);
void refk_IncrementCounter_std(size_t, void*);
void refk_ResetRadiance_std(size_t, uint, uint, void*);
void refk_GenerateAOV_std(size_t, void*, void*, void*, void*, void*, void*, void*, void*, uint, uint, const void*, const void*, void*, void*, void*, void*);
void refk_TemporalAccumulation_std(size_t, uint, uint, void*, void*, void*, void*, void*);
void refk_ResolveRadiance_std(size_t, uint, uint, uint, void*, void*, void*, void*, void*, void*, float*);
void refk_ResolveRadiance_dn(size_t, uint, uint, uint, void*, void*, void*, void*, void*, void*, float*);
}

namespace
{

// 64-byte aligned zero-initialised device-buffer stand-in
struct Buf
{
    void* p = nullptr;
    size_t size = 0;
    void alloc(size_t n) { release(); size = n; if (posix_memalign(&p, 64, n ? n : 64) != 0) abort(); memset(p, 0, n ? n : 64); }
    void release() { free(p); p = nullptr; size = 0; }
    ~Buf() { release(); }
};

struct ArrayAccel : public AccelerationStructure
{
    std::vector<LinearBVHNode> nodes;
    void BuildCPU(std::vector<Triangle>&) override {}
    std::vector<LinearBVHNode> const& GetNodes() const override { return nodes; }
};

struct SceneArrays
{
    std::vector<Triangle> triangles;
    std::vector<PackedMaterial> materials;
    std::vector<Light> lights;
    std::vector<Texture> textures;
    std::vector<std::uint32_t> texture_data;
    std::vector<std::uint32_t> emissive;
    std::vector<float> env;   // RGBA32F
    std::uint32_t env_width = 0, env_height = 0;
    SceneInfo info = {};
};

const int kMaxStatBounces = 64;
struct Stats
{
    std::uint32_t n_ext[kMaxStatBounces], n_miss[kMaxStatBounces], n_hit[kMaxStatBounces];
    std::uint32_t n_shadow[kMaxStatBounces], n_cont[kMaxStatBounces], n_unoccluded[kMaxStatBounces];
};

// sampling.h:50 indexes rankingTile with the un-wrapped dimension and so reads up to 247 ints past its end for the last
// tile pixels (undefined behaviour; on the host it would pick up whatever the linker placed next).  The kernels get a
// copy followed by 256 zeros, which is the behaviour include/rt_b200.h defines for those reads.
static const int* PaddedRankingTile()
{
    static std::vector<int> padded = [] {
        const size_t n = sizeof(rankingTile) / sizeof(rankingTile[0]);
        std::vector<int> v(n + 256, 0);
        for (size_t k = 0; k < n; ++k) v[k] = (int)rankingTile[k];
        return v;
    }();
    return padded.data();
}

// Tables that replace the compiled-in ones (ref_set_sampler_tables); empty: the reference's own tables.
static std::vector<int> g_sobol, g_scrambling, g_ranking;
static const void* SobolTable() { return g_sobol.empty() ? (const void*)sobol_256spp_256d : (const void*)g_sobol.data(); }
static const void* ScramblingTable() { return g_scrambling.empty() ? (const void*)scramblingTile : (const void*)g_scrambling.data(); }
static const void* RankingTable() { return g_ranking.empty() ? (const void*)PaddedRankingTile() : (const void*)g_ranking.data(); }

class RefCpuIntegrator : public Integrator
{
public:
    RefCpuIntegrator(std::uint32_t width, std::uint32_t height, AccelerationStructure& acc, SceneArrays& scene)
        : Integrator(width, height, acc), scene_(scene)
    {
        // cl_pt_integrator.cpp:194-249
        size_t n = (size_t)width_ * height_;
        radiance_.alloc(n * 16); prev_radiance_.alloc(n * 16);
        for (int i = 0; i < 2; ++i) { rays_[i].alloc(n * sizeof(Ray)); pixel_indices_[i].alloc(n * 4); ray_counter_[i].alloc(4); }
        shadow_rays_.alloc(n * sizeof(Ray)); shadow_pixel_indices_.alloc(n * 4); shadow_ray_counter_.alloc(4);
        hits_.alloc(n * sizeof(Hit)); shadow_hits_.alloc(n * 4); throughputs_.alloc(n * 16);
        sample_counter_.alloc(4); direct_light_samples_.alloc(n * 16);
        diffuse_albedo_.alloc(n * 16); depth_.alloc(n * 4); prev_depth_.alloc(n * 4);
        normal_.alloc(n * 16); velocity_.alloc(n * 8);
        resolved_.alloc(n * 16);
        tap_hits_.alloc(n * sizeof(Hit)); tap_rays_.alloc(n * sizeof(Ray));
        // cl_pt_integrator.cpp:392-402
        rt_triangles_.reserve(scene_.triangles.size());
        for (auto const& t : scene_.triangles)
            rt_triangles_.emplace_back(t.v1.position, t.v2.position, t.v3.position);
        CreateKernels();
        Reset();
    }

    void UploadGPUData(Scene const&, AccelerationStructure const&) override {}
    void SetCameraData(Camera const& camera) override { cur_camera_ = camera; aov_prev_camera_ = prev_camera_; prev_camera_ = camera; }
    void SetSamplerType(SamplerType t) override { if (t == sampler_type_) return; sampler_type_ = t; CreateKernels(); RequestReset(); }
    void SetAOV(AOV aov) override { if (aov == aov_) return; aov_ = aov; RequestReset(); }
    void EnableDenoiser(bool e) override { if (e == enable_denoiser_) return; enable_denoiser_ = e; CreateKernels(); RequestReset(); }

    std::uint32_t MaxBounces() const { return max_bounces_; }
    Stats stats = {};
    Buf radiance_, resolved_, tap_hits_, tap_rays_;
    Buf diffuse_albedo_, depth_, normal_, velocity_;
    std::uint32_t SampleCount() const { return *(std::uint32_t*)sample_counter_.p; }

protected:
    void CreateKernels() override {}   // variants are picked at call time from the option flags

    void Reset() override
    {
        if (!enable_denoiser_) refk_ClearCounter_std(1, sample_counter_.p);           // cl_pt_integrator.cpp:497-508
        refk_ResetRadiance_std(N(), width_, height_, radiance_.p);
    }
    void AdvanceSampleCount() override { refk_IncrementCounter_std(1, sample_counter_.p); }
    void GenerateRays() override
    {
        refk_RayGeneration_std(N(), width_, height_, &cur_camera_, sample_counter_.p, rays_[0].p, ray_counter_[0].p,
            pixel_indices_[0].p, throughputs_.p, diffuse_albedo_.p, depth_.p, normal_.p, velocity_.p);
        if (row_step_ > 1)
        {   // bounded sample for CPU timing (bench.py): keep only the rays of rows y % step == first.  This is a
            // host-side edit of the ray queue between two kernels; no kernel is modified.
            Ray* r = (Ray*)rays_[0].p; std::uint32_t* pi = (std::uint32_t*)pixel_indices_[0].p;
            std::uint32_t n = 0;
            for (std::uint32_t y = row_first_; y < height_; y += row_step_)
                for (std::uint32_t x = 0; x < width_; ++x) { r[n] = r[(size_t)y * width_ + x]; pi[n] = y * width_ + x; ++n; }
            *(std::uint32_t*)ray_counter_[0].p = n;
        }
    }
    public: std::uint32_t row_first_ = 0, row_step_ = 1; protected:
    void IntersectRays(std::uint32_t bounce) override
    {
        int in = bounce & 1;
        refk_TraceBvh_std(N(), rays_[in].p, ray_counter_[in].p, rt_triangles_.data(), (void*)acc_structure_.GetNodes().data(), hits_.p);
        std::uint32_t live = *(std::uint32_t*)ray_counter_[in].p;
        if (bounce < (std::uint32_t)kMaxStatBounces)
        {
            stats.n_ext[bounce] = live;
            std::uint32_t miss = 0;
            const Hit* h = (const Hit*)hits_.p;
            for (std::uint32_t i = 0; i < live; ++i) miss += (h[i].primitive_id == 0xFFFFFFFFu);
            stats.n_miss[bounce] = miss; stats.n_hit[bounce] = live - miss;
        }
        if (bounce == 0) { memcpy(tap_hits_.p, hits_.p, hits_.size); memcpy(tap_rays_.p, rays_[0].p, rays_[0].size); }
    }
    void ComputeAOVs() override
    {
        refk_GenerateAOV_std(N(), rays_[0].p, ray_counter_[0].p, pixel_indices_[0].p, hits_.p, scene_.triangles.data(),
            scene_.materials.data(), scene_.textures.data(), scene_.texture_data.data(), width_, height_,
            &cur_camera_, &aov_prev_camera_, diffuse_albedo_.p, depth_.p, normal_.p, velocity_.p);
    }
    void ShadeMissedRays(std::uint32_t bounce) override
    {
        int in = bounce & 1;
        auto fn = enable_white_furnace_ ? refk_Miss_wf : refk_Miss_std;
        fn(N(), rays_[in].p, ray_counter_[in].p, hits_.p, pixel_indices_[in].p, throughputs_.p,
            scene_.env.data(), (int)scene_.env_width, (int)scene_.env_height, radiance_.p);
    }
    void ShadeSurfaceHits(std::uint32_t bounce) override
    {
        int in = bounce & 1, out = (bounce + 1) & 1;
        bool bn = sampler_type_ == SamplerType::kBlueNoise;
        auto fn = enable_white_furnace_ ? (bn ? refk_HitSurface_wfbn : refk_HitSurface_wf) : (bn ? refk_HitSurface_bn : refk_HitSurface_std);
        fn(N(), rays_[in].p, ray_counter_[in].p, pixel_indices_[in].p, hits_.p, scene_.triangles.data(),
            scene_.lights.data(), scene_.emissive.data(), scene_.materials.data(), scene_.textures.data(),
            scene_.texture_data.data(), bounce, width_, height_, sample_counter_.p, &scene_.info,
            (void*)SobolTable(), (void*)ScramblingTable(), (void*)RankingTable(),
            throughputs_.p, rays_[out].p, ray_counter_[out].p, pixel_indices_[out].p,
            shadow_rays_.p, shadow_ray_counter_.p, shadow_pixel_indices_.p, direct_light_samples_.p, radiance_.p);
        if (bounce < (std::uint32_t)kMaxStatBounces)
        {
            stats.n_shadow[bounce] = *(std::uint32_t*)shadow_ray_counter_.p;
            stats.n_cont[bounce] = *(std::uint32_t*)ray_counter_[out].p;
        }
        cur_bounce_ = bounce;
    }
    void IntersectShadowRays() override
    {
        refk_TraceBvh_shadow(N(), shadow_rays_.p, shadow_ray_counter_.p, rt_triangles_.data(), (void*)acc_structure_.GetNodes().data(), shadow_hits_.p);
        if (cur_bounce_ < (std::uint32_t)kMaxStatBounces)
        {
            std::uint32_t live = *(std::uint32_t*)shadow_ray_counter_.p, un = 0;
            const std::uint32_t* h = (const std::uint32_t*)shadow_hits_.p;
            for (std::uint32_t i = 0; i < live; ++i) un += (h[i] == 0xFFFFFFFFu);
            stats.n_unoccluded[cur_bounce_] = un;
        }
    }
    void AccumulateDirectSamples() override
    {
        refk_AccumulateDirectSamples_std(N(), shadow_hits_.p, shadow_ray_counter_.p, shadow_pixel_indices_.p, direct_light_samples_.p, radiance_.p);
    }
    void ClearOutgoingRayCounter(std::uint32_t bounce) override { refk_ClearCounter_std(1, ray_counter_[(bounce + 1) & 1].p); }
    void ClearShadowRayCounter() override { refk_ClearCounter_std(1, shadow_ray_counter_.p); }
    void Denoise() override { refk_TemporalAccumulation_std(N(), width_, height_, radiance_.p, prev_radiance_.p, depth_.p, prev_depth_.p, velocity_.p); }
    void CopyHistoryBuffers() override { memcpy(prev_radiance_.p, radiance_.p, radiance_.size); memcpy(prev_depth_.p, depth_.p, depth_.size); }
    void ResolveRadiance() override
    {
        auto fn = enable_denoiser_ ? refk_ResolveRadiance_dn : refk_ResolveRadiance_std;
        fn(N(), width_, height_, (uint)aov_, radiance_.p, diffuse_albedo_.p, depth_.p, normal_.p, velocity_.p, sample_counter_.p, (float*)resolved_.p);
    }

private:
    size_t N() const { return (size_t)width_ * height_; }
    SceneArrays& scene_;
    std::vector<RTTriangle> rt_triangles_;
    Camera cur_camera_ = {}, aov_prev_camera_ = {};
    std::uint32_t cur_bounce_ = 0;
    Buf prev_radiance_, rays_[2], pixel_indices_[2], ray_counter_[2], shadow_rays_, shadow_pixel_indices_, shadow_ray_counter_;
    Buf hits_, shadow_hits_, throughputs_, sample_counter_, direct_light_samples_, prev_depth_;
};

struct RefHandle
{
    SceneArrays arrays;
    ArrayAccel accel;
    std::unique_ptr<RefCpuIntegrator> integrator;
    std::uint32_t width = 0, height = 0;
};

} // namespace

extern "C" {

// Load an OBJ the way the reference app does (main.cpp:55-58, render.cpp:60-67):
// Scene ctor -> AddDirectionalLight -> Bvh::BuildCPU (reorders triangles) -> Finalize.
void* ref_open_obj(const char* ref_root, const char* obj_rel_path, float scale, int flip_yz, int add_default_light)
{
    char cwd[4096];
    if (!getcwd(cwd, sizeof(cwd))) return nullptr;
    if (chdir(ref_root) != 0) return nullptr;   // Finalize() opens "assets/ibl/..." relative to the CWD (scene.cpp:360)
    RefHandle* h = nullptr;
    try
    {
        Scene scene(obj_rel_path, scale, flip_yz != 0);
        if (add_default_light) scene.AddDirectionalLight({ -0.6f, -1.5f, 3.5f }, { 15.0f, 10.0f, 5.0f });
        Bvh bvh;
        bvh.BuildCPU(scene.GetTriangles());
        scene.Finalize();
        h = new RefHandle;
        h->arrays.triangles = scene.GetTriangles();
        h->arrays.materials = scene.GetMaterials();
        h->arrays.lights = scene.GetLights();
        h->arrays.textures = scene.GetTextures();
        h->arrays.texture_data = scene.GetTextureData();
        h->arrays.emissive = scene.GetEmissiveIndices();
        h->arrays.info = scene.GetSceneInfo();
        Image const& env = scene.GetEnvImage();
        h->arrays.env_width = env.width; h->arrays.env_height = env.height;
        h->arrays.env.resize(env.data.size());
        memcpy(h->arrays.env.data(), env.data.data(), env.data.size() * 4);
        h->accel.nodes = bvh.GetNodes();
    }
    catch (std::exception& e)
    {
        fprintf(stderr, "ref_open_obj: %s\n", e.what());
        delete h; h = nullptr;
    }
    if (chdir(cwd) != 0) { /* nothing sensible to do */ }
    return h;
}

void* ref_open_arrays(const void* triangles, size_t n_triangles, const void* nodes, size_t n_nodes,
    const void* materials, size_t n_materials, const void* lights, size_t n_lights,
    const void* textures, size_t n_textures, const void* texels, size_t n_texels,
    const void* emissive, size_t n_emissive, const float* env, std::uint32_t env_w, std::uint32_t env_h,
    const void* scene_info)
{
    RefHandle* h = new RefHandle;
    auto fill = [](auto& vec, const void* src, size_t n) { vec.resize(n); if (n) memcpy((void*)vec.data(), src, n * sizeof(vec[0])); };
    // Triangle has a user constructor only; build via raw storage
    h->arrays.triangles.reserve(n_triangles);
    for (size_t i = 0; i < n_triangles; ++i) { Triangle t = ((const Triangle*)triangles)[i]; h->arrays.triangles.push_back(t); }
    fill(h->arrays.materials, materials, n_materials);
    fill(h->arrays.lights, lights, n_lights);
    fill(h->arrays.textures, textures, n_textures);
    fill(h->arrays.texture_data, texels, n_texels);
    fill(h->arrays.emissive, emissive, n_emissive);
    h->arrays.env.assign(env, env + (size_t)env_w * env_h * 4);
    h->arrays.env_width = env_w; h->arrays.env_height = env_h;
    memcpy(&h->arrays.info, scene_info, sizeof(SceneInfo));
    fill(h->accel.nodes, nodes, n_nodes);
    return h;
}

// which: 0 triangles 1 nodes 2 materials 3 lights 4 textures 5 texels 6 emissive 7 env(float) 8 scene_info
int ref_scene_query(void* handle, int which, const void** ptr, size_t* count, std::uint32_t* extra0, std::uint32_t* extra1)
{
    RefHandle* h = (RefHandle*)handle;
    SceneArrays& a = h->arrays;
    *extra0 = *extra1 = 0;
    switch (which)
    {
    case 0: *ptr = a.triangles.data(); *count = a.triangles.size(); return 0;
    case 1: *ptr = h->accel.nodes.data(); *count = h->accel.nodes.size(); return 0;
    case 2: *ptr = a.materials.data(); *count = a.materials.size(); return 0;
    case 3: *ptr = a.lights.data(); *count = a.lights.size(); return 0;
    case 4: *ptr = a.textures.data(); *count = a.textures.size(); return 0;
    case 5: *ptr = a.texture_data.data(); *count = a.texture_data.size(); return 0;
    case 6: *ptr = a.emissive.data(); *count = a.emissive.size(); return 0;
    case 7: *ptr = a.env.data(); *count = a.env.size(); *extra0 = a.env_width; *extra1 = a.env_height; return 0;
    case 8: *ptr = &a.info; *count = 1; return 0;
    }
    return -1;
}

int ref_begin(void* handle, std::uint32_t width, std::uint32_t height)
{
    RefHandle* h = (RefHandle*)handle;
    h->width = width; h->height = height;
    h->integrator.reset(new RefCpuIntegrator(width, height, h->accel, h->arrays));
    return 0;
}

void ref_set_camera(void* handle, const void* camera) { Camera c; memcpy(&c, camera, sizeof(Camera)); ((RefHandle*)handle)->integrator->SetCameraData(c); }
void ref_set_max_bounces(void* handle, std::uint32_t b) { ((RefHandle*)handle)->integrator->SetMaxBounces(b); }
void ref_enable_white_furnace(void* handle, int e) { ((RefHandle*)handle)->integrator->EnableWhiteFurnace(e != 0); }
// The three sampler tables of utils/blue_noise_sampler.hpp as the reference compiled them in (tests read them from here
// rather than from a committed copy).
void ref_sampler_tables(const int** sobol, const int** scrambling, const int** ranking)
{
    *sobol = (const int*)sobol_256spp_256d; *scrambling = (const int*)scramblingTile; *ranking = (const int*)rankingTile;
}
// Other tables of the same sizes for the blue-noise kernels (the ranking table gets the same 256 zeros of padding as the
// compiled-in one); null pointers restore the compiled-in tables.
void ref_set_sampler_tables(const int* sobol, const int* scrambling, const int* ranking)
{
    if (!sobol || !scrambling || !ranking) { g_sobol.clear(); g_scrambling.clear(); g_ranking.clear(); return; }
    const size_t n_sobol = sizeof(sobol_256spp_256d) / sizeof(int), n_scrambling = sizeof(scramblingTile) / sizeof(int),
                 n_ranking = sizeof(rankingTile) / sizeof(rankingTile[0]);
    g_sobol.assign(sobol, sobol + n_sobol);
    g_scrambling.assign(scrambling, scrambling + n_scrambling);
    g_ranking.assign(ranking, ranking + n_ranking);
    g_ranking.resize(n_ranking + 256, 0);
}
void ref_set_sampler(void* handle, int blue_noise) { ((RefHandle*)handle)->integrator->SetSamplerType(blue_noise ? Integrator::SamplerType::kBlueNoise : Integrator::SamplerType::kRandom); }
void ref_enable_denoiser(void* handle, int e) { ((RefHandle*)handle)->integrator->EnableDenoiser(e != 0); }
void ref_set_aov(void* handle, int aov) { ((RefHandle*)handle)->integrator->SetAOV((Integrator::AOV)aov); }
void ref_set_row_sample(void* handle, std::uint32_t first, std::uint32_t step) { auto& it = *((RefHandle*)handle)->integrator; it.row_first_ = first; it.row_step_ = step ? step : 1; }
void ref_request_reset(void* handle) { ((RefHandle*)handle)->integrator->RequestReset(); }
void ref_integrate(void* handle) { ((RefHandle*)handle)->integrator->Integrate(); }

// which: 0 radiance(float4/pixel) 1 resolved image(float4/pixel) 2 primary hits (Hit/ray) 3 primary rays (Ray/ray)
//        4 stats (6 x 64 uint32) 5 sample count (1 uint32) 6 albedo(float4) 7 depth(float) 8 normal(float4) 9 velocity(float2)
int ref_read(void* handle, int which, void* dst)
{
    RefHandle* h = (RefHandle*)handle;
    RefCpuIntegrator& it = *h->integrator;
    switch (which)
    {
    case 0: memcpy(dst, it.radiance_.p, it.radiance_.size); return 0;
    case 1: memcpy(dst, it.resolved_.p, it.resolved_.size); return 0;
    case 2: memcpy(dst, it.tap_hits_.p, it.tap_hits_.size); return 0;
    case 3: memcpy(dst, it.tap_rays_.p, it.tap_rays_.size); return 0;
    case 4: memcpy(dst, &it.stats, sizeof(Stats)); return 0;
    case 5: { std::uint32_t c = it.SampleCount(); memcpy(dst, &c, 4); return 0; }
    case 6: memcpy(dst, it.diffuse_albedo_.p, it.diffuse_albedo_.size); return 0;
    case 7: memcpy(dst, it.depth_.p, it.depth_.size); return 0;
    case 8: memcpy(dst, it.normal_.p, it.normal_.size); return 0;
    case 9: memcpy(dst, it.velocity_.p, it.velocity_.size); return 0;
    }
    return -1;
}

void ref_close(void* handle) { delete (RefHandle*)handle; }

int ref_libm_variant() {
#if defined(RT_REF_LIBM) && RT_REF_LIBM
    return 1;
#else
    return 0;
#endif
}

} // extern "C"
