// ProgressiveRaytracingPipeline.h / RealtimeRaytracingPipeline (see RealtimeRaytracingPipeline.h) — headless
// counterparts of include/ProgressiveRaytracingPipeline.h:14-77 and include/RealtimeRaytracingPipeline.h.
// Both reference pipelines share almost all of their host code; here that code lives once in
// RaytracingPipelineBase and the two classes differ in shader library, outputs and accumulation.
#pragma once
#include <array>

#include "RaytracingPipeline.h"

class RaytracingPipelineBase : public RaytracingPipeline {
public:
    void userInterface() override {}
    void render(UINT frameIndex, UINT width, UINT height) override;
    void loadResources(UINT frameCount) override;
    void buildAccelerationStructures() override;
    void addMaterial(Material material) override { mMaterials.push_back(material); }
    void setCamera(std::shared_ptr<Math::Camera> camera) override { mCamera = camera; }
    void setScene(DXRFramework::RtScene::SharedPtr scene) override;
    void createOutputResource(DXGI_FORMAT format, UINT width, UINT height) override;
    DXRFramework::RtBuffer::SharedPtr getOutputResource(UINT id) override { return mOutputResource.at(id); }
    uint64_t getOutputUavHandle(UINT id) override { return mOutputResource.at(id)->gpuHandle(); }
    uint64_t getOutputSrvHandle(UINT id) override { return mOutputResource.at(id)->gpuHandle(); }
    bool *isActive() override { return &mActive; }
    void setJitterSeed(uint32_t seed) override { mRng = std::mt19937(seed); }
    const PerFrameConstants &getFrameConstants() const override { return mConstantBuffer; }

    // Multi-GPU sharding of a frame (SURVEY.md 8e; the reference is single-GPU).  setStripShard: render() covers only
    // every `groups`-th strip of `stripRows` image rows, starting with strip `group` (RtContext::raytraceStrips).
    // skipFrame: consume the jitter of a sample another rank renders, so that every rank draws the SAME jitter for
    // sample s as a single GPU would (update() takes its jitter from a sequential generator, :191-193).
    void setStripShard(UINT stripRows, UINT groups, UINT group) { mStripRows = stripRows, mStripGroups = groups, mStripGroup = group; }
    void skipFrame() { (void)mRngDist(mRng), (void)mRngDist(mRng); }
    // setRowBand: render() covers image rows [row0, row1) only (RtContext::raytraceRegion) — the band of a realtime frame
    // this rank renders and filters (its core rows plus the filter's reach, DenoiseCompositor::dispatchBand).
    void setRowBand(UINT row0, UINT row1) { mBandRow0 = row0, mBandRow1 = row1; }
    // MAX_RADIANCE_RAY_DEPTH (1 in the reference's shaders; 2 = one more Phong-lobe bounce) and emulation of the
    // R16G16B16A16_FLOAT render targets createOutputResource() is asked for (rt_set_render_options); applied by render().
    void setRenderOptions(UINT maxRadianceRayDepth, bool halfRenderTargets) { mRenderOptions = {maxRadianceRayDepth, halfRenderTargets ? 1u : 0u}; }
    // AOV outputs (rt_set_aov_output; progressive pipeline only): enableAov before createOutputResource, which allocates the
    // enabled ones next to the beauty output; render() then accumulates them from the same rays.  getAovResource is null
    // for an AOV that is not enabled.  render() binds all RT_AOV_COUNT slots on every call (null for disabled ones), so a
    // pipeline without AOVs sharing the context with one that has them never dispatches into the other's buffers.
    void enableAov(rt_aov aov) { mAovEnabled.at(aov) = true; }
    DXRFramework::RtBuffer::SharedPtr getAovResource(rt_aov aov) const { return mAovResource.at(aov); }

    // Environment: a procedural sky by default; loadEnvironmentDDS replaces it with an R16G16B16A16F / R32G32B32A32F
    // cube map file such as the reference's assets/textures/CathedralRadiance.dds.
    bool loadEnvironmentDDS(const std::string &path);
    void setEnvironment(DXRFramework::RtTexture::SharedPtr tex) { mEnvCube = tex; }

    bool mAnimationPaused = true;
    DebugOptions mShaderDebugOptions;
    DirectX::XMFLOAT4 pointLightColor{0.2f, 0.8f, 0.6f, 2.0f};  // src/ProgressiveRaytracingPipeline.cpp:13-14
    DirectX::XMFLOAT4 dirLightColor{0.9f, 0.9f, 0.9f, 1.0f};
    DirectX::XMFLOAT4 pointLightPos{0.0f, 0.0f, 0.0f, 1.0f};

protected:
    RaytracingPipelineBase(DXRFramework::RtContext::SharedPtr context, const uint8_t *library, UINT librarySize, UINT maxPayloadSize, UINT numOutputs);
    void fillCommonConstants(float elapsedTime, UINT elapsedFrames, UINT width, UINT height);

    DXRFramework::RtContext::SharedPtr mRtContext;
    DXRFramework::RtProgram::SharedPtr mRtProgram;
    DXRFramework::RtBindings::SharedPtr mRtBindings;
    DXRFramework::RtState::SharedPtr mRtState;
    DXRFramework::RtScene::SharedPtr mRtScene;
    std::vector<Material> mMaterials;
    std::shared_ptr<Math::Camera> mCamera;
    std::vector<DXRFramework::RtBuffer::SharedPtr> mOutputResource;
    std::array<bool, RT_AOV_COUNT> mAovEnabled{};
    std::array<DXRFramework::RtBuffer::SharedPtr, RT_AOV_COUNT> mAovResource;
    // adaptive sampling (ProgressiveRaytracingPipeline::setAdaptiveSampling): per-pixel counts and moments, null when off;
    // render() binds them (or unbinds) on every call
    DXRFramework::RtBuffer::SharedPtr mAdaptiveCounts, mAdaptiveMoments;
    UINT mNumOutputs;
    UINT mOutputWidth = 0, mOutputHeight = 0;  // of the last createOutputResource
    PerFrameConstants mConstantBuffer{};
    DXRFramework::RtTexture::SharedPtr mEnvCube;
    bool mActive = true;
    UINT mStripRows = 32, mStripGroups = 1, mStripGroup = 0;
    UINT mBandRow0 = 0, mBandRow1 = 0;  // row1 > row0: render only these rows
    rt_render_options mRenderOptions{1u, 0u};
    std::mt19937 mRng;
    std::uniform_real_distribution<float> mRngDist;
};

class ProgressiveRaytracingPipeline : public RaytracingPipelineBase {
public:
    using SharedPtr = std::shared_ptr<ProgressiveRaytracingPipeline>;
    static SharedPtr create(DXRFramework::RtContext::SharedPtr context) { return SharedPtr(new ProgressiveRaytracingPipeline(context)); }

    void update(float elapsedTime, UINT elapsedFrames, UINT prevFrameIndex, UINT frameIndex, UINT width, UINT height) override;
    int getNumOutputs() override { return 1; }
    const char *getName() override { return "Progressive Ray Tracing Pipeline"; }

    bool mFrameAccumulationEnabled = true;
    UINT getAccumCount() const { return mAccumCount; }
    void restartAccumulation() { mHasLastCamera = false; }  // what a UI change does (mLastCameraVPMatrix = Matrix4())
    // The beauty output filtered by rt_denoise_progressive, with the albedo and normal AOVs as guides (both must be enabled
    // with enableAov).  Stream-ordered after the last render(); the filter's scratch and the returned output are allocated on
    // first use and reused by later calls, so the result is valid until the next denoise().
    DXRFramework::RtBuffer::SharedPtr denoise(const rt_progressive_denoise_params &params);
    // The beauty output filtered by rt_denoise_temporal: the frames filtered since the last resetTemporal() are the history,
    // reprojected through the position AOV into the camera of the last render().  Needs the albedo, normal and position
    // AOVs enabled and mFrameAccumulationEnabled false (one sample per frame).  Call once after every render(); the result
    // is valid until the next call.
    DXRFramework::RtBuffer::SharedPtr denoiseTemporal(const rt_temporal_denoise_params &params);
    void resetTemporal() { mHasTemporalHistory = false; }
    // Adaptive sampling (rt_set_adaptive_sampling): call after createOutputResource.  Allocates zeroed per-pixel sample counts
    // and luminance moments, which every later render() binds; converged pixels are skipped.  A restart of the accumulation
    // (a camera move, restartAccumulation, accumulation off) zeroes them, so every pixel is active again.
    void setAdaptiveSampling(const rt_adaptive_params &params);
    // rt_adaptive_update with the parameters of setAdaptiveSampling: marks converged pixels and returns how many pixels are
    // still active (synchronises).
    UINT adaptiveUpdate();
    // width x height uint32: n_p in bits 0-30, converged in bit 31 (null unless setAdaptiveSampling was called)
    DXRFramework::RtBuffer::SharedPtr getSampleCountResource() const { return mAdaptiveCounts; }

private:
    explicit ProgressiveRaytracingPipeline(DXRFramework::RtContext::SharedPtr context);
    UINT mAccumCount = 0;
    float mLastCameraVP[16] = {};
    bool mHasLastCamera = false;
    DXRFramework::RtBuffer::SharedPtr mDenoiseTmp, mDenoiseOut;
    uint64_t mDenoiseBytes = 0;
    // rt_denoise_temporal: the history pair (mTemporalHistory[0] = the last call's), its scratch and output, and the camera
    // of the frame the last call filtered
    DXRFramework::RtBuffer::SharedPtr mTemporalHistory[2], mTemporalTmp, mTemporalOut;
    uint64_t mTemporalBytes = 0;
    CameraParams mPrevCamera{};
    bool mHasTemporalHistory = false;
    rt_adaptive_params mAdaptiveParams = RT_ADAPTIVE_DEFAULTS;
    DXRFramework::RtBuffer::SharedPtr mAdaptiveActive;  // one uint32: rt_adaptive_update's active count
};
