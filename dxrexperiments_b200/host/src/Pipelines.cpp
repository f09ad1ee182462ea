// Pipelines.cpp — host side of the two ray-tracing pipelines and the denoise compositor, re-hosted on the C ABI.
// Follows src/ProgressiveRaytracingPipeline.cpp:27-247, src/RealtimeRaytracingPipeline.cpp:27-235 and
// src/DenoiseCompositor.cpp:15-148 of the reference (constants, update() arithmetic, record layout, dispatch order).
#include <algorithm>
#include <cmath>

#include "../include/DenoiseCompositor.h"
#include "../include/ImageIO.h"
#include "../include/RealtimeRaytracingPipeline.h"

using namespace DXRFramework;
using namespace DirectX;

static const UINT kSizeOfMaterialInUint32 = sizeof(MaterialParams) / sizeof(uint32_t);

RaytracingPipelineBase::RaytracingPipelineBase(RtContext::SharedPtr context, const uint8_t *library, UINT librarySize, UINT maxPayloadSize,
                                               UINT numOutputs)
    : mRtContext(context), mNumOutputs(numOutputs), mRngDist(0.0f, 1.0f) {
    RtProgram::Desc programDesc;
    {
        std::vector<std::wstring> libraryExports = {L"RayGen", L"PrimaryClosestHit", L"PrimaryMiss", L"ShadowClosestHit", L"ShadowAnyHit", L"ShadowMiss"};
        programDesc.addShaderLibrary(library, librarySize, libraryExports);
        programDesc.setRayGen("RayGen");
        programDesc.addHitGroup(0, "PrimaryClosestHit", "").addMiss(0, "PrimaryMiss");
        programDesc.addHitGroup(1, "ShadowClosestHit", "ShadowAnyHit").addMiss(1, "ShadowMiss");
        programDesc.configureGlobalRootSignature([](RootSignatureGenerator &config) {
            config.AddRootParameter(RootParameterType::SRV, 0);  // t0: acceleration structure
            config.AddHeapRangesParameter(0, 0);                 // u0: output view(s)
            config.AddRootParameter(RootParameterType::CBV, 0);  // b0: per-frame constants
        });
        programDesc.configureHitGroupRootSignature([](RootSignatureGenerator &config) {
            config.AddHeapRangesParameter(0, 1);  // t0, space1: vertex buffer
            config.AddHeapRangesParameter(1, 1);  // t1, space1: index buffer
            config.AddRootParameter(RootParameterType::Constants32Bit, 0, 1, kSizeOfMaterialInUint32);  // b0, space1
        });
        programDesc.configureMissRootSignature([](RootSignatureGenerator &config) {
            config.AddHeapRangesParameter(0, 2);  // t0, space2: lat-long environment map (unused by the shader)
            config.AddHeapRangesParameter(1, 2);  // t1, space2: environment cube map
        });
    }
    mRtProgram = RtProgram::create(context, programDesc);
    mRtState = RtState::create(context);
    mRtState->setProgram(mRtProgram);
    mRtState->setMaxTraceRecursionDepth(4);
    mRtState->setMaxAttributeSize(8);
    mRtState->setMaxPayloadSize(maxPayloadSize);

    std::memset(&mShaderDebugOptions, 0, sizeof(mShaderDebugOptions));
    mShaderDebugOptions.maxIterations = 1024;
    mShaderDebugOptions.cosineHemisphereSampling = 1;
    mShaderDebugOptions.environmentStrength = 1.0f;
    mRng = std::mt19937(1234u);
}

void RaytracingPipelineBase::setScene(RtScene::SharedPtr scene) {
    mRtScene = scene;
    mRtBindings = RtBindings::create(mRtContext, mRtProgram, scene);
}

void RaytracingPipelineBase::buildAccelerationStructures() { mRtScene->build(mRtContext, mRtProgram->getHitProgramCount()); }

void RaytracingPipelineBase::loadResources(UINT /*frameCount*/) {
    if (!mEnvCube) {
        std::vector<float> texels;
        const uint32_t size = 64;
        ImageIO::proceduralSkyCube(size, texels);
        auto tex = std::make_shared<RtTexture>();
        tex->texels = mRtContext->createBuffer(texels.data(), texels.size() * sizeof(float));
        tex->size = size;
        tex->cubemap = true;
        mEnvCube = tex;
    }
}

bool RaytracingPipelineBase::loadEnvironmentDDS(const std::string &path) {
    std::vector<float> texels;
    uint32_t size = 0;
    if (!ImageIO::readDDSCube(path, texels, size)) return false;
    auto tex = std::make_shared<RtTexture>();
    tex->texels = mRtContext->createBuffer(texels.data(), texels.size() * sizeof(float));
    tex->size = size;
    tex->cubemap = true;
    mEnvCube = tex;
    return true;
}

void RaytracingPipelineBase::createOutputResource(DXGI_FORMAT /*format*/, UINT width, UINT height) {
    mOutputResource.clear();
    mOutputWidth = width, mOutputHeight = height;
    for (UINT i = 0; i < mNumOutputs; ++i) {
        auto b = mRtContext->createBuffer(uint64_t(width) * height * 16);
        b->clear();
        mOutputResource.push_back(b);
    }
    for (int k = 0; k < RT_AOV_COUNT; ++k) {
        mAovResource[k] = nullptr;
        if (!mAovEnabled[k]) continue;
        mAovResource[k] = mRtContext->createBuffer(uint64_t(width) * height * 16);
        mAovResource[k]->clear();
    }
}

// calculateCameraVariables (src/ProgressiveRaytracingPipeline.cpp:151-168)
static void calculateCameraVariables(Math::Camera &camera, float aspectRatio, float U[4], float V[4], float W[4]) {
    Math::Vector3 w = camera.GetForwardVec();  // not normalised again: its length is the focal length
    float wlen = Math::Length(w);
    Math::Vector3 u = Math::Normalize(Math::Cross(w, camera.GetUpVec()));
    Math::Vector3 v = Math::Normalize(Math::Cross(u, w));
    float vlen = wlen * tanf(0.5f * camera.GetFOV());
    float ulen = vlen * aspectRatio;
    u = u * ulen;
    v = v * vlen;
    U[0] = u.x, U[1] = u.y, U[2] = u.z, U[3] = 0.0f;
    V[0] = v.x, V[1] = v.y, V[2] = v.z, V[3] = 0.0f;
    W[0] = w.x, W[1] = w.y, W[2] = w.z, W[3] = 0.0f;
}

void RaytracingPipelineBase::fillCommonConstants(float elapsedTime, UINT elapsedFrames, UINT width, UINT height) {
    if (mAnimationPaused) elapsedTime = 142.0f;
    CameraParams &cameraParams = mConstantBuffer.cameraParams;
    Math::Vector3 eye = mCamera->GetPosition();
    cameraParams.worldEyePos[0] = eye.x, cameraParams.worldEyePos[1] = eye.y, cameraParams.worldEyePos[2] = eye.z, cameraParams.worldEyePos[3] = 1.0f;
    calculateCameraVariables(*mCamera, mCamera->GetAspectRatio(), cameraParams.U, cameraParams.V, cameraParams.W);
    float xJitter = (mRngDist(mRng) - 0.5f) / float(width);
    float yJitter = (mRngDist(mRng) - 0.5f) / float(height);
    cameraParams.jitters[0] = xJitter, cameraParams.jitters[1] = yJitter;
    cameraParams.frameCount = elapsedFrames;

    XMFLOAT4 dirLightVector{0.3f, -0.2f, -1.0f, 0.0f};
    XMMATRIX rotation = XMMatrixRotationY(sinf(elapsedTime * 0.2f) * 3.14f * 0.5f);
    dirLightVector = XMVector4Transform(dirLightVector, rotation);
    float *fd = mConstantBuffer.directionalLight.forwardDir;
    fd[0] = dirLightVector.x, fd[1] = dirLightVector.y, fd[2] = dirLightVector.z, fd[3] = dirLightVector.w;
    float *dc = mConstantBuffer.directionalLight.color;
    dc[0] = dirLightColor.x, dc[1] = dirLightColor.y, dc[2] = dirLightColor.z, dc[3] = dirLightColor.w;
    float *pp = mConstantBuffer.pointLight.worldPos;
    pp[0] = pointLightPos.x, pp[1] = pointLightPos.y, pp[2] = pointLightPos.z, pp[3] = pointLightPos.w;
    float *pc = mConstantBuffer.pointLight.color;
    pc[0] = pointLightColor.x, pc[1] = pointLightColor.y, pc[2] = pointLightColor.z, pc[3] = pointLightColor.w;
}

void RaytracingPipelineBase::render(UINT /*frameIndex*/, UINT width, UINT height) {
    // Update shader table root arguments (src/ProgressiveRaytracingPipeline.cpp:218-234)
    auto program = mRtBindings->getProgram();
    for (UINT rayType = 0; rayType < program->getHitProgramCount(); ++rayType) {
        for (UINT instance = 0; instance < mRtScene->getNumInstances(); ++instance) {
            auto &hitVars = mRtBindings->getHitVars(rayType, instance);
            hitVars->appendHeapRanges(mRtScene->getModel(instance)->getVertexBufferSrvHandle());
            hitVars->appendHeapRanges(mRtScene->getModel(instance)->getIndexBufferSrvHandle());
            const Material &m = mMaterials.at(instance < mMaterials.size() ? instance : mMaterials.size() - 1);
            hitVars->append32BitConstants(&m.params, kSizeOfMaterialInUint32);
        }
    }
    for (UINT rayType = 0; rayType < program->getMissProgramCount(); ++rayType) {
        auto &missVars = mRtBindings->getMissVars(rayType);
        missVars->appendHeapRanges(0);  // lat-long map: never sampled
        missVars->appendHeapRanges(createTextureSRVHandle(mEnvCube));
    }
    mRtBindings->apply(mRtContext, mRtState);

    // Set global root arguments (:236-242)
    rt_context *ctx = mRtContext->getNative();
    ThrowIfFailed(rt_set_frame_constants(ctx, &mConstantBuffer), "rt_set_frame_constants");
    for (UINT i = 0; i < mNumOutputs; ++i)
        ThrowIfFailed(rt_set_output(ctx, i, static_cast<float *>(mOutputResource.at(i)->ptr()), uint64_t(width) * 16), "rt_set_output");
    for (uint32_t k = 0; k < RT_AOV_COUNT; ++k)
        ThrowIfFailed(rt_set_aov_output(ctx, k, mAovResource[k] ? static_cast<float *>(mAovResource[k]->ptr()) : nullptr, uint64_t(width) * 16),
                      "rt_set_aov_output");
    ThrowIfFailed(rt_set_tlas(ctx, mRtScene->getTlasWrappedPtr()), "rt_set_tlas");
    // the scene's instance motion for the previous-position AOV; NULL otherwise, so that no earlier binding is inherited
    const float *motion = mAovResource[RT_AOV_PREVIOUS_POSITION] ? mRtScene->getMotionPtr() : nullptr;
    ThrowIfFailed(rt_set_instance_motion(ctx, motion, motion ? mRtScene->getNumInstances() : 0), "rt_set_instance_motion");
    // likewise its deforming models' previous positions (RtScene::update)
    const rt_deformation_desc *deform = mAovResource[RT_AOV_PREVIOUS_POSITION] ? mRtScene->getDeformationPtr() : nullptr;
    ThrowIfFailed(rt_set_instance_deformation(ctx, deform, deform ? mRtScene->getNumInstances() : 0), "rt_set_instance_deformation");
    ThrowIfFailed(rt_set_adaptive_sampling(ctx, mAdaptiveCounts ? static_cast<uint32_t *>(mAdaptiveCounts->ptr()) : nullptr,
                                           mAdaptiveMoments ? static_cast<float *>(mAdaptiveMoments->ptr()) : nullptr),
                  "rt_set_adaptive_sampling");
    ThrowIfFailed(rt_set_render_options(ctx, &mRenderOptions), "rt_set_render_options");

    if (mBandRow1 > mBandRow0) mRtContext->raytraceRegion(mRtBindings, mRtState, width, height, 0, mBandRow0, width, std::min(mBandRow1, height));
    else if (mStripGroups > 1) mRtContext->raytraceStrips(mRtBindings, mRtState, width, height, mStripRows, mStripGroups, mStripGroup);
    else mRtContext->raytrace(mRtBindings, mRtState, width, height, 3);
    for (auto &o : mOutputResource) mRtContext->insertUAVBarrier(o);
    for (auto &o : mAovResource)
        if (o) mRtContext->insertUAVBarrier(o);
}

// ------------------------------------------------------------------------------------------------ progressive
ProgressiveRaytracingPipeline::ProgressiveRaytracingPipeline(RtContext::SharedPtr context)
    : RaytracingPipelineBase(context, kProgressiveRaytracingLibrary, kProgressiveRaytracingLibrarySize, 20, 1) {}

void ProgressiveRaytracingPipeline::update(float elapsedTime, UINT elapsedFrames, UINT, UINT, UINT width, UINT height) {
    float vp[16];
    mCamera->GetViewProjSignature(vp);
    const bool moved = !mHasLastCamera || std::memcmp(vp, mLastCameraVP, sizeof(vp)) != 0;  // hasCameraMoved
    if (moved || !mFrameAccumulationEnabled) {
        mAccumCount = 0;
        std::memcpy(mLastCameraVP, vp, sizeof(vp));
        mHasLastCamera = true;
        if (mAdaptiveCounts) mAdaptiveCounts->clear(), mAdaptiveMoments->clear();  // the running means restart with n_p = 0
    }
    fillCommonConstants(elapsedTime, elapsedFrames, width, height);
    mConstantBuffer.cameraParams.accumCount = mAccumCount++;
    mConstantBuffer.options = mShaderDebugOptions;
}

void ProgressiveRaytracingPipeline::setAdaptiveSampling(const rt_adaptive_params &params) {
    ThrowIfFalse(mOutputWidth > 0 && mOutputHeight > 0, "ProgressiveRaytracingPipeline::setAdaptiveSampling needs createOutputResource first");
    const uint64_t pixels = uint64_t(mOutputWidth) * mOutputHeight;
    mAdaptiveCounts = mRtContext->createBuffer(4 * pixels);
    mAdaptiveMoments = mRtContext->createBuffer(8 * pixels);
    mAdaptiveActive = mRtContext->createBuffer(4);
    mAdaptiveCounts->clear(), mAdaptiveMoments->clear();
    mAdaptiveParams = params;
}

UINT ProgressiveRaytracingPipeline::adaptiveUpdate() {
    ThrowIfFalse(mAdaptiveCounts != nullptr, "ProgressiveRaytracingPipeline::adaptiveUpdate needs setAdaptiveSampling first");
    ThrowIfFailed(rt_adaptive_update(mRtContext->getNative(), static_cast<const float *>(mAdaptiveMoments->ptr()),
                                     static_cast<uint32_t *>(mAdaptiveCounts->ptr()), mOutputWidth, mOutputHeight, &mAdaptiveParams,
                                     static_cast<uint32_t *>(mAdaptiveActive->ptr())),
                  "rt_adaptive_update");
    uint32_t active = 0;
    mAdaptiveActive->download(&active, sizeof(active));  // synchronises
    return active;
}

RtBuffer::SharedPtr ProgressiveRaytracingPipeline::denoise(const rt_progressive_denoise_params &params) {
    const auto albedo = mAovResource[RT_AOV_ALBEDO], normal = mAovResource[RT_AOV_NORMAL];
    ThrowIfFalse(albedo && normal, "ProgressiveRaytracingPipeline::denoise needs the albedo and normal AOVs enabled");
    const uint64_t bytes = uint64_t(mOutputWidth) * mOutputHeight * 16;
    if (!mDenoiseOut || mDenoiseBytes != bytes) {
        mDenoiseTmp = mRtContext->createBuffer(2 * bytes);
        mDenoiseOut = mRtContext->createBuffer(bytes);
        mDenoiseBytes = bytes;
    }
    ThrowIfFailed(rt_denoise_progressive(mRtContext->getNative(), static_cast<const float *>(mOutputResource.at(0)->ptr()),
                                         static_cast<const float *>(albedo->ptr()), static_cast<const float *>(normal->ptr()),
                                         static_cast<float *>(mDenoiseTmp->ptr()), static_cast<float *>(mDenoiseOut->ptr()), mOutputWidth,
                                         mOutputHeight, &params),
                  "rt_denoise_progressive");
    return mDenoiseOut;
}

RtBuffer::SharedPtr ProgressiveRaytracingPipeline::denoiseTemporal(const rt_temporal_denoise_params &params) {
    const auto albedo = mAovResource[RT_AOV_ALBEDO], normal = mAovResource[RT_AOV_NORMAL], position = mAovResource[RT_AOV_POSITION];
    ThrowIfFalse(albedo && normal && position, "ProgressiveRaytracingPipeline::denoiseTemporal needs the albedo, normal and position AOVs enabled");
    ThrowIfFalse(!mFrameAccumulationEnabled, "ProgressiveRaytracingPipeline::denoiseTemporal needs mFrameAccumulationEnabled = false");
    const uint64_t bytes = uint64_t(mOutputWidth) * mOutputHeight * 16;
    if (!mTemporalOut || mTemporalBytes != bytes) {
        mTemporalHistory[0] = mRtContext->createBuffer(4 * bytes);
        mTemporalHistory[1] = mRtContext->createBuffer(4 * bytes);
        mTemporalTmp = mRtContext->createBuffer(2 * bytes);
        mTemporalOut = mRtContext->createBuffer(bytes);
        mTemporalBytes = bytes;
        mHasTemporalHistory = false;
    }
    std::swap(mTemporalHistory[0], mTemporalHistory[1]);  // [1] = the last call's history, [0] = this call's
    const rt_camera_params *prevCamera = mHasTemporalHistory ? &mPrevCamera : nullptr;
    const float *prevHistory = mHasTemporalHistory ? static_cast<const float *>(mTemporalHistory[1]->ptr()) : nullptr;
    if (const auto previous = mAovResource[RT_AOV_PREVIOUS_POSITION])  // moving instances: reproject through their motion
        ThrowIfFailed(rt_denoise_temporal_motion(mRtContext->getNative(), static_cast<const float *>(mOutputResource.at(0)->ptr()),
                                                 static_cast<const float *>(albedo->ptr()), static_cast<const float *>(normal->ptr()),
                                                 static_cast<const float *>(position->ptr()), static_cast<const float *>(previous->ptr()),
                                                 prevCamera, prevHistory, static_cast<float *>(mTemporalHistory[0]->ptr()),
                                                 static_cast<float *>(mTemporalTmp->ptr()), static_cast<float *>(mTemporalOut->ptr()),
                                                 mOutputWidth, mOutputHeight, &params),
                      "rt_denoise_temporal_motion");
    else
        ThrowIfFailed(rt_denoise_temporal(mRtContext->getNative(), static_cast<const float *>(mOutputResource.at(0)->ptr()),
                                          static_cast<const float *>(albedo->ptr()), static_cast<const float *>(normal->ptr()),
                                          static_cast<const float *>(position->ptr()), prevCamera, prevHistory,
                                          static_cast<float *>(mTemporalHistory[0]->ptr()), static_cast<float *>(mTemporalTmp->ptr()),
                                          static_cast<float *>(mTemporalOut->ptr()), mOutputWidth, mOutputHeight, &params),
                      "rt_denoise_temporal");
    mPrevCamera = mConstantBuffer.cameraParams;
    mHasTemporalHistory = true;
    return mTemporalOut;
}

// ------------------------------------------------------------------------------------------------ realtime
RealtimeRaytracingPipeline::RealtimeRaytracingPipeline(RtContext::SharedPtr context)
    : RaytracingPipelineBase(context, kRealtimeRaytracingLibrary, kRealtimeRaytracingLibrarySize, 60, 2) {}

void RealtimeRaytracingPipeline::update(float elapsedTime, UINT elapsedFrames, UINT, UINT, UINT width, UINT height) {
    fillCommonConstants(elapsedTime, elapsedFrames, width, height);
    mConstantBuffer.cameraParams.accumCount = 0;
    std::memset(&mConstantBuffer.options, 0, sizeof(mConstantBuffer.options));
    mConstantBuffer.options.environmentStrength = 1.0f;  // src/RealtimeRaytracingPipeline.cpp:196
}

// ------------------------------------------------------------------------------------------------ denoise compositor
DenoiseCompositor::DenoiseCompositor(RtContext::SharedPtr context) : mRtContext(context) {
    mConstantBuffer.exposure = 1.0f;  // src/DenoiseCompositor.cpp:45-50
    mConstantBuffer.gamma = 2.2f;
    mConstantBuffer.tonemap = 1;
    mConstantBuffer.gammaCorrect = 0;
    mConstantBuffer.maxKernelSize = 12;
    mConstantBuffer.debugVisualize = 0;
}

void DenoiseCompositor::loadResources(UINT, bool) {}
void DenoiseCompositor::setMockResources(RtBuffer::SharedPtr direct, RtBuffer::SharedPtr indirectSpecular) {
    mMock[0] = direct;
    mMock[1] = indirectSpecular;
}

void DenoiseCompositor::createOutputResource(DXGI_FORMAT, UINT width, UINT height) {
    for (auto &o : mOutputResource) o = mRtContext->createBuffer(uint64_t(width) * height * 16);
}

// Multi-GPU (SURVEY.md 8e-ii; the reference is single-GPU): filter image rows [row0, row1) only and keep the core rows
// [core0, core1) of the result — the rest of the output stays / becomes zero, so that the weight-1 sum of the ranks' outputs
// (RtContext::reduceAccumulation) is the frame.  With row0 <= core0 - maxKernelSize and row1 >= core1 + maxKernelSize
// (clipped at the image border) the core rows are the rows dispatch() produces on the whole frame, bit for bit: the
// filter reaches maxKernelSize rows up and down (BilateralFilter.hlsli:92-115).
void DenoiseCompositor::dispatchBand(InputComponents inputs, UINT width, UINT height, UINT row0, UINT row1, UINT core0, UINT core1) {
    ThrowIfFalse(inputs.directLightingSrv != 0 && inputs.indirectSpecularSrv != 0, "DenoiseCompositor::dispatchBand: no inputs");
    ThrowIfFalse(mOutputResource[0] && mOutputResource[1], "DenoiseCompositor: createOutputResource was not called");
    ThrowIfFalse(row0 <= core0 && core0 <= core1 && core1 <= row1 && row1 <= height && row0 < row1, "DenoiseCompositor::dispatchBand: rows");
    rt_context *ctx = mRtContext->getNative();
    const uint64_t row = uint64_t(width) * 4;  // floats per row
    float *tmp = static_cast<float *>(mOutputResource[0]->ptr()), *out = static_cast<float *>(mOutputResource[1]->ptr());
    ThrowIfFailed(rt_memset(ctx, out, 0, uint64_t(height) * row * 4), "rt_memset");
    ThrowIfFailed(rt_denoise(ctx, reinterpret_cast<const float *>(inputs.directLightingSrv) + row0 * row,
                             reinterpret_cast<const float *>(inputs.indirectSpecularSrv) + row0 * row, tmp + row0 * row, out + row0 * row, width,
                             row1 - row0, &mConstantBuffer),
                  "rt_denoise");
    if (core0 > row0) ThrowIfFailed(rt_memset(ctx, out + row0 * row, 0, uint64_t(core0 - row0) * row * 4), "rt_memset");
    if (row1 > core1) ThrowIfFailed(rt_memset(ctx, out + core1 * row, 0, uint64_t(row1 - core1) * row * 4), "rt_memset");
}

void DenoiseCompositor::dispatch(InputComponents inputs, UINT, UINT width, UINT height) {
    if (inputs.directLightingSrv == 0) {  // mock inputs (src/DenoiseCompositor.cpp:113-116)
        ThrowIfFalse(mMock[0] && mMock[1], "DenoiseCompositor: no inputs and no mock resources");
        inputs.directLightingSrv = mMock[0]->gpuHandle();
        inputs.indirectSpecularSrv = mMock[1]->gpuHandle();
    }
    ThrowIfFalse(mOutputResource[0] && mOutputResource[1], "DenoiseCompositor: createOutputResource was not called");
    // pass 0 (H) -> mOutputResource[0]; pass 1 (V) -> mOutputResource[1]
    ThrowIfFailed(rt_denoise(mRtContext->getNative(), reinterpret_cast<const float *>(inputs.directLightingSrv),
                             reinterpret_cast<const float *>(inputs.indirectSpecularSrv), static_cast<float *>(mOutputResource[0]->ptr()),
                             static_cast<float *>(mOutputResource[1]->ptr()), width, height, &mConstantBuffer),
                  "rt_denoise");
}
