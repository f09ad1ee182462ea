// api.cu — context, buffers, programs and bindings of the C ABI (include/rt_core.h).
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.cuh"

static thread_local char g_error[512] = "";

void rt_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

extern "C" {

const char *rt_last_error(void) { return g_error; }
const char *rt_version(void) { return "rt_core 0.1 (sm_100a, CUDA " RT_STR(CUDART_VERSION) ")"; }

int rt_context_create(int device, rt_context **out) {
    RT_REQUIRE(out != nullptr, "out");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        rt_set_error("no CUDA device available (%s); rt_core has no CPU fallback", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return RT_ERR_CUDA;
    }
    RT_REQUIRE(device >= 0 && device < count, "device ordinal out of range");
    RT_CUDA(cudaSetDevice(device));
    rt_context *ctx = new rt_context();
    ctx->device = device;
    cudaDeviceProp prop;
    RT_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx->num_sms = prop.multiProcessorCount;
    RT_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->owns_stream = true;
    RT_CUDA(cudaMalloc(&ctx->status, 256));
    RT_CUDA(cudaMemset(ctx->status, 0, 256));
    RT_CUDA(cudaMalloc(&ctx->ray_counts, 256));
    RT_CUDA(cudaMemset(ctx->ray_counts, 0, 256));
    *out = ctx;
    return RT_OK;
}

int rt_context_destroy(rt_context *ctx) {
    if (!ctx) return RT_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->ws.base) cudaFree(ctx->ws.base);
    for (auto &b : ctx->band_streams)
        for (cudaStream_t q : b)
            if (q) cudaStreamDestroy(q);
    for (auto &b : ctx->band_events)
        for (cudaEvent_t e : b)
            if (e) cudaEventDestroy(e);
    if (ctx->ev_band_fork) cudaEventDestroy(ctx->ev_band_fork);
    if (ctx->side_stream) cudaStreamDestroy(ctx->side_stream);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->status) cudaFree(ctx->status);
    if (ctx->hit_programs) cudaFree(ctx->hit_programs);
    if (ctx->ray_counts) cudaFree(ctx->ray_counts);
    if (ctx->ev_ready)
        for (auto &e : ctx->ev) cudaEventDestroy(e);
    if (ctx->owns_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return RT_OK;
}

int rt_context_set_stream(rt_context *ctx, void *stream) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    if (ctx->owns_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    ctx->stream = static_cast<cudaStream_t>(stream);
    ctx->owns_stream = false;
    return RT_OK;
}

int rt_sync(rt_context *ctx) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

int rt_get_status(rt_context *ctx) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    uint32_t s = 0;
    RT_CUDA(cudaMemcpyAsync(&s, ctx->status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    if (s & 2u) {
        // not sticky: it describes the dispatches since the last check, not the context
        const uint32_t cleared = s & ~2u;
        RT_CUDA(cudaMemcpyAsync(ctx->status, &cleared, 4, cudaMemcpyHostToDevice, ctx->stream));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    if (s & 8u) {
        const uint32_t cleared = s & ~14u;
        RT_CUDA(cudaMemcpyAsync(ctx->status, &cleared, 4, cudaMemcpyHostToDevice, ctx->stream));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        rt_set_error("a ray hit an instance whose hit-group record index lies beyond the bound records "
                     "(InstanceContributionToHitGroupIndex + ray type >= records set with rt_bindings_set_hit_record)");
        return RT_ERR_INVALID_ARG;
    }
    if (s & 4u) {
        const uint32_t cleared = s & ~6u;
        RT_CUDA(cudaMemcpyAsync(ctx->status, &cleared, 4, cudaMemcpyHostToDevice, ctx->stream));
        RT_CUDA(cudaStreamSynchronize(ctx->stream));
        rt_set_error("a top-level build was given an instance whose BLAS address is null or does not hold a finished bottom-level "
                     "build of this library; such instances were made inactive");
        return RT_ERR_INVALID_ARG;
    }
    if (s & 1u) {
        rt_set_error("traversal stack overflow: a ray needed more than 64 stack entries");
        return RT_ERR_OVERFLOW;
    }
    if (s & 2u) {
        rt_set_error("the acceleration structure holds procedural primitives but the dispatch's hit groups are of type TRIANGLES "
                     "(no intersection program): every ray was reported as a miss; use rt_trace_rays_hit_groups");
        return RT_ERR_UNSUPPORTED;
    }
    return RT_OK;
}

uint64_t rt_launch_count(const rt_context *ctx) { return ctx ? ctx->launches : 0; }

int rt_malloc(rt_context *ctx, uint64_t bytes, void **dev) {
    RT_REQUIRE(ctx && dev, "null argument");
    RT_CUDA(cudaSetDevice(ctx->device));
    RT_CUDA(cudaMalloc(dev, bytes ? bytes : 1));
    return RT_OK;
}
int rt_free(rt_context *ctx, void *dev) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    if (!dev) return RT_OK;
    RT_CUDA(cudaSetDevice(ctx->device));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    RT_CUDA(cudaFree(dev));
    return RT_OK;
}
int rt_memset(rt_context *ctx, void *dev, int value, uint64_t bytes) {
    RT_REQUIRE(ctx && (dev || bytes == 0), "null argument");
    RT_CUDA(cudaSetDevice(ctx->device));
    RT_CUDA(cudaMemsetAsync(dev, value, bytes, ctx->stream));
    return RT_OK;
}
int rt_upload(rt_context *ctx, void *dev, const void *host, uint64_t bytes) {
    RT_REQUIRE(ctx && (bytes == 0 || (dev && host)), "null argument");
    RT_CUDA(cudaSetDevice(ctx->device));
    if (bytes) RT_CUDA(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return RT_OK;
}
int rt_download(rt_context *ctx, void *host, const void *dev, uint64_t bytes) {
    RT_REQUIRE(ctx && (bytes == 0 || (dev && host)), "null argument");
    RT_CUDA(cudaSetDevice(ctx->device));
    if (bytes) RT_CUDA(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}
int rt_host_alloc_pinned(uint64_t bytes, void **host) {
    RT_REQUIRE(host != nullptr, "host");
    RT_CUDA(cudaMallocHost(host, bytes ? bytes : 1));
    return RT_OK;
}
int rt_host_free_pinned(void *host) {
    if (host) RT_CUDA(cudaFreeHost(host));
    return RT_OK;
}

// ---------------------------------------------------------------------------------------------- programs
int rt_program_create(rt_context *ctx, rt_program_kind kind, uint32_t hit_group_count, uint32_t miss_count, rt_program **out) {
    RT_REQUIRE(ctx && out, "null argument");
    RT_REQUIRE(kind == RT_PROGRAM_PROGRESSIVE || kind == RT_PROGRAM_REALTIME, "program kind");
    // both shader libraries declare hit groups {Primary, Shadow} and miss shaders {PrimaryMiss, ShadowMiss}
    // (src/ProgressiveRaytracingPipeline.cpp:36-39); the instance contribution is i * hit_group_count.
    RT_REQUIRE(hit_group_count >= 1 && hit_group_count <= 8, "hit_group_count");
    RT_REQUIRE(miss_count >= 1 && miss_count <= 8, "miss_count");
    rt_program *p = new rt_program();
    p->ctx = ctx;
    p->kind = kind;
    p->hit_group_count = hit_group_count;
    p->miss_count = miss_count;
    *out = p;
    return RT_OK;
}

int rt_program_destroy(rt_program *p) {
    if (!p) return RT_OK;
    if (p->ctx) {
        cudaSetDevice(p->ctx->device);
        cudaStreamSynchronize(p->ctx->stream);
    }
    if (p->dev_recs) cudaFree(p->dev_recs);
    free(p->host_recs);
    delete p;
    return RT_OK;
}

int rt_bindings_set_hit_record(rt_program *p, uint32_t ray_type, uint32_t instance, const void *vb, const void *ib,
                               const rt_material_params *mat) {
    RT_REQUIRE(p && mat, "null argument");
    RT_REQUIRE(ray_type < p->hit_group_count, "ray type beyond the program's hit groups");  // std::logic_error in RtBindings.cpp:77-79
    RT_REQUIRE(instance < (1u << 22), "instance index");
    RT_REQUIRE(vb != nullptr && ib != nullptr, "hit record needs a vertex and an index buffer");
    RT_REQUIRE((uintptr_t(vb) & 3) == 0 && (uintptr_t(ib) & 3) == 0, "buffer alignment");
    const uint32_t idx = instance * p->hit_group_count + ray_type;
    if (idx >= p->cap_recs) {
        uint32_t cap = p->cap_recs ? p->cap_recs : 16;
        while (cap <= idx) cap *= 2;
        rt_hit_record_dev *h = static_cast<rt_hit_record_dev *>(calloc(cap, sizeof(rt_hit_record_dev)));
        RT_REQUIRE(h != nullptr, "out of host memory");
        if (p->host_recs) memcpy(h, p->host_recs, sizeof(rt_hit_record_dev) * p->n_recs);
        free(p->host_recs);
        p->host_recs = h;
        RT_CUDA(cudaSetDevice(p->ctx->device));
        RT_CUDA(cudaStreamSynchronize(p->ctx->stream));
        if (p->dev_recs) RT_CUDA(cudaFree(p->dev_recs));
        RT_CUDA(cudaMalloc(&p->dev_recs, sizeof(rt_hit_record_dev) * cap));
        p->cap_recs = cap;
    }
    rt_hit_record_dev &r = p->host_recs[idx];
    r.vb = static_cast<const float *>(vb);
    r.ib = static_cast<const uint32_t *>(ib);
    r.mat = *mat;
    if (idx + 1 > p->n_recs) p->n_recs = idx + 1;
    p->dirty = true;
    return RT_OK;
}

int rt_bindings_set_miss_record(rt_program *p, uint32_t ray_type, const float *env, uint32_t size) {
    RT_REQUIRE(p != nullptr, "program");
    RT_REQUIRE(ray_type < p->miss_count, "ray type beyond the program's miss shaders");
    RT_REQUIRE((uintptr_t(env) & 15) == 0, "environment texels must be 16-byte aligned");
    if (ray_type == 0) {  // PrimaryMiss samples the cube; ShadowMiss has no resources that matter
        p->env_texels = env;
        p->env_size = env ? size : 0;
    }
    return RT_OK;
}

// ---------------------------------------------------------------------------------------------- per-dispatch state
int rt_set_frame_constants(rt_context *ctx, const rt_per_frame_constants *f) {
    RT_REQUIRE(ctx && f, "null argument");
    ctx->frame = *f;
    return RT_OK;
}
int rt_set_output(rt_context *ctx, uint32_t slot, float *rgba, uint64_t pitch) {
    RT_REQUIRE(ctx != nullptr && slot < 2, "slot");
    RT_REQUIRE((uintptr_t(rgba) & 15) == 0 && pitch % 16 == 0, "output alignment");
    ctx->output[slot] = rgba;
    ctx->pitch[slot] = pitch;
    return RT_OK;
}
int rt_set_aov_output(rt_context *ctx, uint32_t aov, float *rgba, uint64_t pitch) {
    RT_REQUIRE(ctx != nullptr && aov < RT_AOV_COUNT, "unknown AOV id");
    RT_REQUIRE((uintptr_t(rgba) & 15) == 0 && pitch % 16 == 0, "AOV output alignment");
    ctx->aov[aov] = rgba;
    ctx->aov_pitch[aov] = pitch;
    return RT_OK;
}
int rt_set_instance_motion(rt_context *ctx, const float *world_to_previous_world, uint32_t n) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    RT_REQUIRE((world_to_previous_world == nullptr) == (n == 0), "motion matrices: NULL with n = 0, or a pointer with n > 0");
    RT_REQUIRE((uintptr_t(world_to_previous_world) & 15) == 0, "motion matrices must be 16-byte aligned");
    RT_REQUIRE(n <= 0xFFFFFFu, "more than 2^24 - 1 motion matrices (InstanceIndex is 24 bits)");
    ctx->motion = world_to_previous_world;
    ctx->n_motion = n;
    return RT_OK;
}
int rt_set_instance_deformation(rt_context *ctx, const rt_deformation_desc *descs, uint32_t n) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    RT_REQUIRE((descs == nullptr) == (n == 0), "deformation descriptors: NULL with n = 0, or a pointer with n > 0");
    RT_REQUIRE((uintptr_t(descs) & 15) == 0, "deformation descriptors must be 16-byte aligned");
    RT_REQUIRE(n <= 0xFFFFFFu, "more than 2^24 - 1 deformation descriptors (InstanceIndex is 24 bits)");
    ctx->deform = descs;
    ctx->n_deform = n;
    return RT_OK;
}
int rt_set_adaptive_sampling(rt_context *ctx, uint32_t *counts, float *moments) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    RT_REQUIRE((counts == nullptr) == (moments == nullptr), "counts and moments are both given or both NULL");
    RT_REQUIRE((uintptr_t(counts) & 3) == 0 && (uintptr_t(moments) & 7) == 0, "counts must be 4-byte and moments 8-byte aligned");
    ctx->adaptive_counts = counts;
    ctx->adaptive_moments = moments;
    return RT_OK;
}
int rt_set_render_options(rt_context *ctx, const rt_render_options *o) {
    RT_REQUIRE(ctx && o, "null argument");
    RT_REQUIRE(o->max_radiance_ray_depth == 1 || o->max_radiance_ray_depth == 2, "max_radiance_ray_depth must be 1 or 2");
    RT_REQUIRE(o->half_render_targets <= 1, "half_render_targets must be 0 or 1");
    ctx->render_options = *o;
    return RT_OK;
}
int rt_set_tlas(rt_context *ctx, const void *tlas) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    ctx->tlas = tlas;
    return RT_OK;
}

int rt_get_ray_counts(rt_context *ctx, rt_ray_counts *counts, int reset) {
    RT_REQUIRE(ctx && counts, "null argument");
    unsigned long long h[3];
    RT_CUDA(cudaMemcpyAsync(h, ctx->ray_counts, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    counts->primary = h[0], counts->secondary = h[1], counts->shadow = h[2];
    if (reset) RT_CUDA(cudaMemsetAsync(ctx->ray_counts, 0, 64, ctx->stream));
    return RT_OK;
}

int rt_enable_trace_stats(rt_context *ctx, int enable) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    ctx->collect_stats = enable != 0;
    return RT_OK;
}

int rt_get_trace_stats(rt_context *ctx, rt_trace_stats *primary, rt_trace_stats *secondary, rt_trace_stats *shadow, int reset) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    unsigned long long h[32];
    RT_CUDA(cudaMemcpyAsync(h, ctx->ray_counts, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    rt_trace_stats *out[3] = {primary, secondary, shadow};
    for (int s = 0; s < 3; ++s)
        if (out[s]) {
            const unsigned long long *p = h + 8 * (s + 1);
            out[s]->rays = p[0], out[s]->internal_visits = p[1], out[s]->leaf_visits = p[2], out[s]->instance_visits = p[3], out[s]->max_stack = p[4];
        }
    if (reset) RT_CUDA(cudaMemsetAsync(ctx->ray_counts + 8, 0, 192, ctx->stream));
    return RT_OK;
}

int rt_enable_stage_timing(rt_context *ctx, int enable) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    ctx->timing = enable != 0;
    return RT_OK;
}

int rt_get_stage_timing(rt_context *ctx, double *primary_ms, double *secondary_ms, double *shadow_ms, int reset) {
    RT_REQUIRE(ctx != nullptr, "ctx");
    RT_CUDA(cudaStreamSynchronize(ctx->stream));
    if (secondary_ms) *secondary_ms = ctx->t_secondary;
    if (primary_ms) *primary_ms = ctx->t_primary;
    if (shadow_ms) *shadow_ms = ctx->t_shadow;
    if (reset) ctx->t_secondary = ctx->t_primary = ctx->t_shadow = 0;
    return RT_OK;
}

}  // extern "C"
