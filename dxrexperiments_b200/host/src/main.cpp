// main.cpp — dxr_headless: the headless replacement of the reference's Win32 app shell
// (src/Main.cpp:18, src/DXRExperimentsApp.cpp:25-229).  It owns an RtContext, an RtScene, the two pipelines and
// the DenoiseCompositor, drives update()/render() for a number of frames and writes the result as PFM.
//
//   dxr_headless --model scene.obj --pipeline progressive --spp 16 --width 1920 --height 1080 --out frame.pfm
//   dxr_headless --scene cornell --pipeline realtime --out direct.pfm --out2 spec.pfm --denoise composite.pfm
//   dxr_headless ... --exr frame.exr [--exr-half]        OpenEXR output (fp32, or HALF = the reference's R16G16B16A16_FLOAT)
//   dxr_headless --pipeline progressive ... --aov albedo albedo.pfm --aov normal normal.exr   AOV outputs, accumulated from the
//     same rays as --out (direct, indirect-diffuse, indirect-specular, albedo, fresnel, normal; EXR when the path ends in .exr)
//   dxr_headless --pipeline progressive ... --denoise-progressive clean.pfm   the beauty output filtered with the albedo and
//     normal AOVs as guides (rt_denoise_progressive; the flag enables both AOVs; EXR when the path ends in .exr)
//   dxr_headless --pipeline progressive ... --orbit 0.5 --spp 16 --denoise-temporal clean.pfm   one sample per frame from a
//     camera orbiting --at by 0.5 degrees per frame, every frame filtered by rt_denoise_temporal; writes the last frame's output
//   dxr_headless --pipeline progressive ... --spp 256 --adaptive 0.1 [--adaptive-min 8] [--adaptive-every 4] --sample-counts n.pfm
//     adaptive sampling: --spp is the per-pixel sample cap; rt_adaptive_update runs every 4 dispatches and the run stops when
//     no pixel is active; --sample-counts writes each pixel's sample count as a grey heat map
// Multi-GPU (one process per GPU, replicated scene; the frame's samples and strips are sharded, one NCCL reduce at the end):
//   for r in 0 1; do dxr_headless ... --spp 64 --world 2 --rank $r --comm-file /tmp/id [--strip-groups 2] --out frame.pfm & done
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <map>

#include "../include/DenoiseCompositor.h"
#include "../include/ImageIO.h"
#include "../include/RealtimeRaytracingPipeline.h"

using namespace DXRFramework;

static void addQuad(std::vector<Vertex> &v, std::vector<uint32_t> &idx, const float p[4][3]) {
    const float e1[3] = {p[1][0] - p[0][0], p[1][1] - p[0][1], p[1][2] - p[0][2]}, e2[3] = {p[2][0] - p[0][0], p[2][1] - p[0][1], p[2][2] - p[0][2]};
    float n[3] = {e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]};
    const float l = sqrtf(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    for (float &c : n) c /= l;
    const uint32_t base = uint32_t(v.size());
    for (int i = 0; i < 4; ++i) v.push_back({{p[i][0], p[i][1], p[i][2]}, {n[0], n[1], n[2]}});
    const uint32_t q[6] = {0, 1, 2, 0, 2, 3};
    for (uint32_t k : q) idx.push_back(base + k);
}

static void addBox(std::vector<Vertex> &v, std::vector<uint32_t> &idx, const float lo[3], const float hi[3], bool inward, int skipFace) {
    const float x0 = lo[0], y0 = lo[1], z0 = lo[2], x1 = hi[0], y1 = hi[1], z1 = hi[2];
    const float faces[6][4][3] = {{{x1, y0, z0}, {x1, y1, z0}, {x1, y1, z1}, {x1, y0, z1}}, {{x0, y0, z0}, {x0, y0, z1}, {x0, y1, z1}, {x0, y1, z0}},
                                  {{x0, y1, z0}, {x0, y1, z1}, {x1, y1, z1}, {x1, y1, z0}}, {{x0, y0, z0}, {x1, y0, z0}, {x1, y0, z1}, {x0, y0, z1}},
                                  {{x0, y0, z1}, {x1, y0, z1}, {x1, y1, z1}, {x0, y1, z1}}, {{x0, y0, z0}, {x0, y1, z0}, {x1, y1, z0}, {x1, y0, z0}}};
    for (int f = 0; f < 6; ++f) {
        if (f == skipFace) continue;
        float p[4][3];
        for (int i = 0; i < 4; ++i) {
            const int s = inward ? (i == 0 ? 0 : 4 - i) : i;  // reverse the winding for inward-facing boxes
            std::memcpy(p[i], faces[f][s], sizeof(p[i]));
        }
        addQuad(v, idx, p);
    }
}

// The procedural Cornell box of config C1 (same geometry as dxrexperiments_b200/scenes.py:cornell_box).
static void makeCornell(std::vector<Vertex> &v, std::vector<uint32_t> &idx) {
    const float lo[3] = {-1, -1, -1}, hi[3] = {1, 1, 1};
    addBox(v, idx, lo, hi, true, 4);
    const float light[4][3] = {{-0.25f, 0.995f, -0.25f}, {0.25f, 0.995f, -0.25f}, {0.25f, 0.995f, 0.25f}, {-0.25f, 0.995f, 0.25f}};
    addQuad(v, idx, light);
    const float tlo[3] = {-0.65f, -1.0f, -0.6f}, thi[3] = {-0.1f, 0.2f, -0.05f}, slo[3] = {0.1f, -1.0f, 0.0f}, shi[3] = {0.65f, -0.4f, 0.55f};
    addBox(v, idx, tlo, thi, false, -1);
    addBox(v, idx, slo, shi, false, -1);
}

struct Args {
    std::map<std::string, std::vector<std::string>> kv;
    bool has(const std::string &k) const { return kv.count(k) != 0; }
    std::string str(const std::string &k, const std::string &d) const { return has(k) && !kv.at(k).empty() ? kv.at(k)[0] : d; }
    double num(const std::string &k, double d, size_t i = 0) const { return has(k) && kv.at(k).size() > i ? std::atof(kv.at(k)[i].c_str()) : d; }
};

static int usage() {
    std::puts("dxr_headless [--model file.obj | --scene cornell|triangle] [--pipeline progressive|realtime] [--width W] [--height H]\n"
              "             [--spp N] [--seed S] [--no-jitter] [--eye x y z] [--at x y z] [--light-pos x y z] [--env-dds file | --env-raw file size]\n"
              "             [--out file.pfm] [--out2 file.pfm] [--denoise file.pfm] [--exr file.exr [--exr-half]] [--dump-frames file.bin] [--device N]\n"
              "             [--radiance-depth 1|2] [--fp16-targets] [--denoise-mock direct.pfm specular.pfm --denoise out.pfm [--kernel-size K]]\n"
              "             [--aov direct|indirect-diffuse|indirect-specular|albedo|fresnel|normal|position|previous-position file.pfm|file.exr]...\n"
              "                                                                    (progressive only)\n"
              "             [--denoise-progressive file.pfm|file.exr]   (progressive only: the beauty output filtered with the albedo and normal AOVs)\n"
              "             [--orbit DEGREES]   (frame f: the eye rotated about --at around +y by f * DEGREES)\n"
              "             [--move DX DY DZ]   (frame f: instance 0 translated by f * (DX, DY, DZ); the camera stays unless --orbit)\n"
              "             [--deform DX DY DZ] (frame f: every vertex of model 0 at its rest position + f * (DX, DY, DZ) * h, h its rest\n"
              "                                  height normalised to [0, 1]: a shear, refitted per frame; progressive pipeline only)\n"
              "             [--denoise-temporal file.pfm|file.exr]   (progressive, one GPU: accumulation off, every frame filtered by rt_denoise_temporal)\n"
              "             [--adaptive THRESHOLD [--adaptive-min N] [--adaptive-every K] [--sample-counts file.pfm|file.exr]]\n"
              "                                                                    (progressive, one GPU: --spp is the sample cap)\n"
              "             [--world N --rank R --comm-file path [--strip-groups G] [--strip-rows 32] [--band-shard]]   (one process per GPU)");
    return 0;
}

int main(int argc, char **argv) {
    Args a;
    for (int i = 1; i < argc; ++i) {
        if (std::strncmp(argv[i], "--", 2) == 0) {
            std::string key = argv[i] + 2;
            a.kv[key];
            while (i + 1 < argc && !(std::strncmp(argv[i + 1], "--", 2) == 0 && !std::isdigit((unsigned char)argv[i + 1][2]) && argv[i + 1][2] != '.'))
                a.kv[key].push_back(argv[++i]);
        }
    }
    if (a.has("help")) return usage();
    const UINT width = UINT(a.num("width", 1920)), height = UINT(a.num("height", 1080)), spp = UINT(a.num("spp", 1));
    const std::string pipelineName = a.str("pipeline", "progressive");
    const int world = int(a.num("world", 1)), rank = int(a.num("rank", 0));
    try {
        if (world < 1 || rank < 0 || rank >= world) throw std::runtime_error("--world / --rank");
        const bool denoiseProgressive = a.has("denoise-progressive");
        if (denoiseProgressive && (pipelineName == "realtime" || a.str("denoise-progressive", "").empty()))
            throw std::runtime_error("--denoise-progressive takes a path and needs --pipeline progressive (--denoise filters the realtime pipeline)");
        const bool denoiseTemporal = a.has("denoise-temporal");
        if (denoiseTemporal && (pipelineName == "realtime" || world > 1 || a.str("denoise-temporal", "").empty()))
            throw std::runtime_error("--denoise-temporal takes a path and needs --pipeline progressive on one GPU (no --world > 1)");
        const bool adaptive = a.has("adaptive");
        if (adaptive && (pipelineName == "realtime" || world > 1 || denoiseTemporal || a.str("adaptive", "").empty()))
            throw std::runtime_error("--adaptive takes a threshold and needs --pipeline progressive on one GPU, without --denoise-temporal");
        if (a.has("sample-counts") && (!adaptive || a.str("sample-counts", "").empty()))
            throw std::runtime_error("--sample-counts takes a path and needs --adaptive");
        const bool deform = a.has("deform");
        if (deform && (pipelineName == "realtime" || a.kv.at("deform").size() != 3))
            throw std::runtime_error("--deform takes DX DY DZ and needs --pipeline progressive (the realtime program has no previous-position AOV)");
        const UINT adaptiveEvery = UINT(a.num("adaptive-every", 4));
        if (adaptive && (adaptiveEvery < 1 || spp < 1)) throw std::runtime_error("--adaptive-every and --spp must be at least 1");
        auto context = RtContext::create(int(a.num("device", rank)));
        if (a.has("denoise-mock")) {
            // DenoiseCompositor with mock inputs (src/DenoiseCompositor.cpp:52-60 loads DirectLighting.png / IndirectSpecular.png and
            // dispatch() falls back to them when it is handed null SRVs, :113-116): --denoise-mock direct.pfm specular.pfm --denoise out.pfm
            std::vector<float> d, sp;
            uint32_t dw = 0, dh = 0, sw = 0, sh = 0;
            if (a.kv.at("denoise-mock").size() < 2 || !ImageIO::readPFM(a.kv.at("denoise-mock")[0], d, dw, dh) ||
                !ImageIO::readPFM(a.kv.at("denoise-mock")[1], sp, sw, sh) || dw != sw || dh != sh)
                throw std::runtime_error("--denoise-mock needs two PFM images of equal size");
            auto denoiser = DenoiseCompositor::create(context);
            denoiser->loadResources(3, true);
            denoiser->setMockResources(context->createBuffer(d.data(), d.size() * sizeof(float)), context->createBuffer(sp.data(), sp.size() * sizeof(float)));
            denoiser->createOutputResource(DXGI_FORMAT_R16G16B16A16_FLOAT, dw, dh);
            if (a.has("kernel-size")) denoiser->mConstantBuffer.maxKernelSize = int(a.num("kernel-size", 12));
            denoiser->dispatch({0, 0}, 0, dw, dh);
            context->waitForGpu();
            std::vector<float> out(size_t(dw) * dh * 4);
            denoiser->getOutputResource()->download(out.data(), out.size() * sizeof(float));
            if (!ImageIO::writePFM(a.str("denoise", "denoised.pfm"), out.data(), dw, dh)) throw std::runtime_error("cannot write the denoised image");
            std::printf("{\"denoise_mock\": true, \"width\": %u, \"height\": %u, \"kernel_launches\": %llu, \"core\": \"%s\"}\n", dw, dh,
                        (unsigned long long)context->launchCount(), rt_version());
            return 0;
        }
        // shard plan (dxrexperiments_b200/sharding.py): rank = sampleGroup * stripGroups + stripGroup
        UINT stripGroups = UINT(a.num("strip-groups", 0));
        if (stripGroups == 0) {  // samples first, strips when the samples run out
            stripGroups = 1;
            while (UINT(world) / stripGroups > std::max<UINT>(spp, 1) || UINT(world) % stripGroups) ++stripGroups;
        }
        if (UINT(world) % stripGroups) throw std::runtime_error("--world must be a multiple of --strip-groups");
        const UINT sampleGroups = UINT(world) / stripGroups, sampleGroup = UINT(rank) / stripGroups, stripGroup = UINT(rank) % stripGroups;
        if (world > 1) {
            if (!a.has("comm-file")) throw std::runtime_error("--world > 1 needs --comm-file (the side channel for the NCCL unique id)");
            context->joinCommunicator(world, rank, a.str("comm-file", ""));
        }

        // ---- scene (DXRExperimentsApp::InitRaytracing, src/DXRExperimentsApp.cpp:78-138)
        auto scene = RtScene::create();
        RtModel::SharedPtr model;
        if (a.has("model")) model = RtModel::create(context, a.str("model", ""));
        else if (a.str("scene", "cornell") == "cornell") {
            std::vector<Vertex> v;
            std::vector<uint32_t> idx;
            makeCornell(v, idx);
            model = RtModel::create(context, v, idx);
        } else model = RtModel::create(context, std::string("<none>"));  // the reference's fallback triangle
        scene->addModel(model, DirectX::XMMatrixIdentity());
        if (deform) model->setDynamic(true);
        const std::vector<Vertex> restVertices = deform ? model->getVertices() : std::vector<Vertex>();

        RaytracingPipeline::Material material{};
        material.params.albedo[0] = 0.95f, material.params.albedo[1] = 0.05f, material.params.albedo[2] = 0.0f, material.params.albedo[3] = 1.0f;
        material.params.specular[0] = material.params.specular[1] = material.params.specular[2] = 0.58f, material.params.specular[3] = 1.0f;
        material.params.roughness = 0.5f;
        material.params.reflectivity = 0.7f;
        material.params.type = 1;

        auto camera = std::make_shared<Math::Camera>();
        camera->SetAspectRatio(float(width) / float(height));
        const bool cornell = !a.has("model") && a.str("scene", "cornell") == "cornell";
        Math::Vector3 eye{float(a.num("eye", cornell ? 0.0 : 8.0, 0)), float(a.num("eye", cornell ? 0.0 : 10.0, 1)), float(a.num("eye", cornell ? 3.5 : 30.0, 2))};
        Math::Vector3 at{float(a.num("at", 0.0, 0)), float(a.num("at", cornell ? 0.0 : 1.5, 1)), float(a.num("at", 0.0, 2))};
        camera->SetEyeAtUp(eye, at, {0, 1, 0});
        camera->SetZRange(1.0f, 10000.0f);

        std::shared_ptr<RaytracingPipelineBase> pipeline;
        if (pipelineName == "realtime") pipeline = RealtimeRaytracingPipeline::create(context);
        else pipeline = ProgressiveRaytracingPipeline::create(context);
        pipeline->setScene(scene);
        pipeline->addMaterial(material);
        pipeline->setCamera(camera);
        pipeline->setJitterSeed(uint32_t(a.num("seed", 1234)));
        if (a.has("light-pos"))
            pipeline->pointLightPos = {float(a.num("light-pos", 0, 0)), float(a.num("light-pos", 0, 1)), float(a.num("light-pos", 0, 2)), 1.0f};
        else if (cornell) pipeline->pointLightPos = {0.0f, 0.5f, 0.0f, 1.0f};
        if (a.has("env-dds") && !pipeline->loadEnvironmentDDS(a.str("env-dds", ""))) throw std::runtime_error("cannot read DDS cube " + a.str("env-dds", ""));
        if (a.has("env-raw")) {
            const uint32_t size = uint32_t(a.num("env-raw", 0, 1));
            std::vector<float> texels(size_t(6) * size * size * 4);
            std::ifstream in(a.str("env-raw", ""), std::ios::binary);
            in.read(reinterpret_cast<char *>(texels.data()), texels.size() * sizeof(float));
            if (!in) throw std::runtime_error("cannot read raw environment texels");
            auto tex = std::make_shared<RtTexture>();
            tex->texels = context->createBuffer(texels.data(), texels.size() * sizeof(float));
            tex->size = size;
            tex->cubemap = true;
            pipeline->setEnvironment(tex);
        }
        // --aov NAME PATH, repeatable: names in rt_aov id order
        static const char *const kAovNames[RT_AOV_COUNT] = {"direct", "indirect-diffuse", "indirect-specular", "albedo", "fresnel", "normal",
                                                                   "position", "previous-position"};
        std::vector<std::pair<int, std::string>> aovFiles;
        if (a.has("aov")) {
            const auto &v = a.kv.at("aov");
            if (pipelineName == "realtime") throw std::runtime_error("--aov needs --pipeline progressive");
            if (v.empty() || v.size() % 2) throw std::runtime_error("--aov takes a name and a path");
            for (size_t i = 0; i < v.size(); i += 2) {
                int id = -1;
                for (int k = 0; k < RT_AOV_COUNT; ++k)
                    if (v[i] == kAovNames[k]) id = k;
                if (id < 0) throw std::runtime_error("unknown AOV name " + v[i]);
                pipeline->enableAov(rt_aov(id));
                aovFiles.emplace_back(id, v[i + 1]);
            }
        }
        if (denoiseProgressive) pipeline->enableAov(RT_AOV_ALBEDO), pipeline->enableAov(RT_AOV_NORMAL);
        const auto progressive = std::dynamic_pointer_cast<ProgressiveRaytracingPipeline>(pipeline);
        if (denoiseTemporal) {
            pipeline->enableAov(RT_AOV_ALBEDO), pipeline->enableAov(RT_AOV_NORMAL), pipeline->enableAov(RT_AOV_POSITION);
            if (a.has("move") || deform) pipeline->enableAov(RT_AOV_PREVIOUS_POSITION);  // moving instances or a deforming model: the motion variant
            progressive->mFrameAccumulationEnabled = false;
        }
        pipeline->loadResources(3);
        pipeline->createOutputResource(DXGI_FORMAT_R16G16B16A16_FLOAT, width, height);
        pipeline->setRenderOptions(UINT(a.num("radiance-depth", 1)), a.has("fp16-targets"));
        if (adaptive) {  // threshold, floor, min_samples (capped at --spp), max_samples = --spp
            rt_adaptive_params ap = RT_ADAPTIVE_DEFAULTS;
            ap.threshold = float(a.num("adaptive", 0.0));
            ap.min_samples = std::min<uint32_t>(uint32_t(a.num("adaptive-min", ap.min_samples)), spp);
            ap.max_samples = spp;
            progressive->setAdaptiveSampling(ap);
        }
        // --band-shard (realtime pipeline + --denoise, one frame): rank r renders AND filters its row band plus the filter's reach;
        // the reduce composites the filtered bands instead of the AOVs (dxrexperiments_b200/sharding.py band_plan)
        const bool bandShard = a.has("band-shard") && world > 1;
        UINT core0 = 0, core1 = height, row0 = 0, row1 = height;
        const UINT halo = 12;  // DenoiseCompositor's maxKernelSize (src/DenoiseCompositor.cpp:49)
        if (bandShard) {
            if (pipelineName != "realtime" || !a.has("denoise") || spp != 1) throw std::runtime_error("--band-shard needs --pipeline realtime --denoise --spp 1");
            core0 = UINT(uint64_t(height) * rank / world), core1 = UINT(uint64_t(height) * (rank + 1) / world);
            row0 = core0 > halo ? core0 - halo : 0, row1 = std::min(height, core1 + halo);
            pipeline->setRowBand(row0, row1);
        } else if (stripGroups > 1) pipeline->setStripShard(UINT(a.num("strip-rows", 32)), stripGroups, stripGroup);

        auto t0 = std::chrono::steady_clock::now();
        pipeline->buildAccelerationStructures();
        context->waitForGpu();
        auto t1 = std::chrono::steady_clock::now();

        // ---- frames (OnUpdate / OnRender)
        std::ofstream frames;
        if (a.has("dump-frames")) frames.open(a.str("dump-frames", ""), std::ios::binary);
        UINT mySamples = 0;
        const rt_temporal_denoise_params temporalParams = RT_TEMPORAL_DENOISE_DEFAULTS;
        RtBuffer::SharedPtr temporalOut;
        UINT dispatches = 0;
        for (UINT f = 0; f < spp; ++f) {
            if (a.has("orbit")) {  // the eye rotated about `at` around +y (scenes.orbit)
                const double ang = double(f) * a.num("orbit", 0.0) * 3.14159265358979323846 / 180.0, c = std::cos(ang), s = std::sin(ang);
                const double dx = double(eye.x) - at.x, dz = double(eye.z) - at.z;
                camera->SetEyeAtUp({float(at.x + c * dx + s * dz), eye.y, float(at.z - s * dx + c * dz)}, at, {0, 1, 0});
            }
            if (deform && f > 0) {  // model 0 sheared by f * (DX, DY, DZ) (scenes.sheared_positions): a BLAS refit
                float lo = restVertices[0].position.y, hi = lo;
                for (const Vertex &v : restVertices) lo = std::min(lo, v.position.y), hi = std::max(hi, v.position.y);
                const double off[3] = {double(f) * a.num("deform", 0.0, 0), double(f) * a.num("deform", 0.0, 1), double(f) * a.num("deform", 0.0, 2)};
                std::vector<Vertex> v = restVertices;
                for (Vertex &x : v) {
                    const double h = hi > lo ? (double(x.position.y) - lo) / (double(hi) - lo) : 0.0;
                    x.position = {float(x.position.x + h * off[0]), float(x.position.y + h * off[1]), float(x.position.z + h * off[2])};
                }
                model->setVertices(context, v);
            }
            if (a.has("move") && f > 0)  // instance 0 at f * (DX, DY, DZ)
                scene->setTransform(0, DirectX::XMMatrixTranslation(float(f * a.num("move", 0.0, 0)), float(f * a.num("move", 0.0, 1)),
                                                                    float(f * a.num("move", 0.0, 2))));
            if ((a.has("move") || deform) && f > 0) scene->update(context);  // a TLAS refit, and the motion since frame f - 1
            if (!bandShard && f % sampleGroups != sampleGroup) {  // another sample group's frame: keep the jitter sequence in step
                pipeline->skipFrame();
                continue;
            }
            ++mySamples;
            pipeline->update(0.0f, f, (f + 2) % 3, f % 3, width, height);
            if (a.has("no-jitter")) {
                auto &fc = const_cast<PerFrameConstants &>(pipeline->getFrameConstants());
                fc.cameraParams.jitters[0] = fc.cameraParams.jitters[1] = 0.0f;
            }
            if (frames) frames.write(reinterpret_cast<const char *>(&pipeline->getFrameConstants()), sizeof(PerFrameConstants));
            pipeline->render(f % 3, width, height);
            ++dispatches;
            if (denoiseTemporal) temporalOut = progressive->denoiseTemporal(temporalParams);
            if (adaptive && (f + 1) % adaptiveEvery == 0 && progressive->adaptiveUpdate() == 0) break;  // every pixel converged
        }
        // ---- the path's one collective: every output is summed onto rank 0, weighted by the rank's share of the samples
        std::vector<RtBuffer::SharedPtr> finalOut;
        for (int i = 0; i < pipeline->getNumOutputs(); ++i) finalOut.push_back(pipeline->getOutputResource(i));
        std::shared_ptr<DenoiseCompositor> bandDenoiser;
        RtBuffer::SharedPtr bandFrame;
        if (bandShard) {
            bandDenoiser = DenoiseCompositor::create(context);
            bandDenoiser->loadResources(3, false);
            bandDenoiser->createOutputResource(DXGI_FORMAT_R16G16B16A16_FLOAT, width, height);
            bandDenoiser->dispatchBand({finalOut[0]->gpuHandle(), finalOut[1]->gpuHandle()}, width, height, row0, row1, core0, core1);
            const uint64_t floats = uint64_t(width) * height * 4;
            bandFrame = rank == 0 ? context->createBuffer(floats * 4) : nullptr;
            context->reduceAccumulation(bandDenoiser->getOutputResource(), bandFrame, floats, 1.0f, 0);
        } else if (world > 1) {
            // in place: on the root the pipeline's own buffers then hold the frame, which is what denoise() filters.  The
            // enabled AOVs are running means like the beauty output, so they reduce with the same weights.
            const uint64_t floats = uint64_t(width) * height * 4;
            std::vector<RtBuffer::SharedPtr> reduced = finalOut;
            for (int k = 0; k < RT_AOV_COUNT; ++k)
                if (auto b = pipeline->getAovResource(rt_aov(k))) reduced.push_back(b);
            for (const auto &b : reduced) context->reduceAccumulation(b, rank == 0 ? b : nullptr, floats, float(mySamples) / float(spp), 0);
        }
        context->waitForGpu();
        context->checkDeviceStatus();
        auto t2 = std::chrono::steady_clock::now();

        std::vector<float> img(size_t(width) * height * 4);
        auto save = [&](RtBuffer::SharedPtr buf, const std::string &path) {
            if (rank != 0) return;  // only the root holds the frame
            buf->download(img.data(), img.size() * sizeof(float));
            const bool exr = path.size() > 4 && path.substr(path.size() - 4) == ".exr";
            const bool ok = exr ? ImageIO::writeEXR(path, img.data(), width, height, a.has("exr-half")) : ImageIO::writePFM(path, img.data(), width, height);
            if (!ok) throw std::runtime_error("cannot write " + path);
        };
        if (a.has("out")) save(finalOut[0], a.str("out", ""));
        if (a.has("exr")) save(finalOut[0], a.str("exr", ""));
        if (a.has("out2") && finalOut.size() > 1) save(finalOut[1], a.str("out2", ""));
        for (const auto &f : aovFiles) save(pipeline->getAovResource(rt_aov(f.first)), f.second);
        if (denoiseProgressive && rank == 0) {
            const rt_progressive_denoise_params params = RT_PROGRESSIVE_DENOISE_DEFAULTS;
            auto clean = std::static_pointer_cast<ProgressiveRaytracingPipeline>(pipeline)->denoise(params);
            context->waitForGpu();
            save(clean, a.str("denoise-progressive", ""));
        }
        if (denoiseTemporal && temporalOut) save(temporalOut, a.str("denoise-temporal", ""));
        if (a.has("sample-counts")) {  // n_p as a grey heat map (the converged bit masked off)
            std::vector<uint32_t> counts(size_t(width) * height);
            progressive->getSampleCountResource()->download(counts.data(), counts.size() * sizeof(uint32_t));
            for (size_t i = 0; i < counts.size(); ++i) {
                const float n = float(counts[i] & ~RT_ADAPTIVE_CONVERGED);
                img[4 * i] = img[4 * i + 1] = img[4 * i + 2] = n, img[4 * i + 3] = 1.0f;
            }
            const std::string path = a.str("sample-counts", "");
            const bool exr = path.size() > 4 && path.substr(path.size() - 4) == ".exr";
            if (!(exr ? ImageIO::writeEXR(path, img.data(), width, height, false) : ImageIO::writePFM(path, img.data(), width, height)))
                throw std::runtime_error("cannot write " + path);
        }
        if (bandShard) {
            save(bandFrame, a.str("denoise", ""));
        } else if (a.has("denoise") && rank == 0) {
            if (pipeline->getNumOutputs() < 2) throw std::runtime_error("--denoise needs --pipeline realtime");
            auto denoiser = DenoiseCompositor::create(context);
            denoiser->loadResources(3, false);
            denoiser->createOutputResource(DXGI_FORMAT_R16G16B16A16_FLOAT, width, height);
            denoiser->dispatch({finalOut[0]->gpuHandle(), finalOut[1]->gpuHandle()}, 0, width, height);
            context->waitForGpu();
            save(denoiser->getOutputResource(), a.str("denoise", ""));
        }
        rt_ray_counts rc{};
        rt_get_ray_counts(context->getNative(), &rc, 0);
        const double buildMs = std::chrono::duration<double, std::milli>(t1 - t0).count(), renderMs = std::chrono::duration<double, std::milli>(t2 - t1).count();
        const double rays = double(rc.primary + rc.secondary + rc.shadow);
        std::printf("{\"pipeline\": \"%s\", \"triangles\": %u, \"width\": %u, \"height\": %u, \"frames\": %u, \"build_ms\": %.3f, \"render_ms\": %.3f, "
                    "\"rays\": %.0f, \"mrays_per_s\": %.1f, \"kernel_launches\": %llu, \"world\": %d, \"rank\": %d, \"strip_groups\": %u, "
                    "\"samples_on_rank\": %u, \"dispatches\": %u, \"primary_rays\": %llu, \"core\": \"%s\"}\n",
                    pipeline->getName(), model->getNumTriangles(), width, height, spp, buildMs, renderMs, rays, rays / (renderMs * 1e3),
                    (unsigned long long)context->launchCount(), world, rank, stripGroups, mySamples, dispatches, (unsigned long long)rc.primary,
                    rt_version());
    } catch (const std::exception &e) {
        std::fprintf(stderr, "dxr_headless: %s\n", e.what());
        return 1;
    }
    return 0;
}
