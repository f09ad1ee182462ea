// RtScene.h — headless counterpart of libs/DXRFramework/RtScene.h:9-45: a list of (model, transform) instances
// and the TLAS built over them (RtScene.cpp:18-52).
#pragma once
#include "RtModel.h"

namespace DXRFramework {

class RtScene {
public:
    using SharedPtr = std::shared_ptr<RtScene>;
    static SharedPtr create() { return SharedPtr(new RtScene()); }
    ~RtScene() = default;

    void addModel(RtModel::SharedPtr model, DirectX::XMMATRIX transform) { mInstances.push_back({model, transform}); }
    RtModel::SharedPtr getModel(UINT index) const { return mInstances.at(index).model; }
    UINT getNumInstances() const { return static_cast<UINT>(mInstances.size()); }

    RtBuffer::SharedPtr getTlasResource() const { return mTlasBuffer; }
    const void *getTlasWrappedPtr() const { return mTlasBuffer ? mTlasBuffer->ptr() : nullptr; }

    // Builds every model's BLAS, then the TLAS with InstanceID = i, InstanceContributionToHitGroupIndex =
    // i * hitGroupCount, mask 0xFF, flags NONE (RtScene.cpp:27-30, Helpers/TopLevelASGenerator.cpp:343-362).
    void build(RtContext::SharedPtr context, UINT hitGroupCount);

    // Moving instances (new work: the reference's scene is static).  setTransform changes an instance's object->world
    // transform; update refits the TLAS in place (PERFORM_UPDATE) and makes the motion the change from the transforms of
    // the previous build or update to these: one row-major 3x4 world -> previous-world matrix per instance,
    // prevObjectToWorld * inverse(objectToWorld) in double and rounded to float, for rt_set_instance_motion.
    void setTransform(UINT index, DirectX::XMMATRIX transform) { mInstances.at(index).transform = transform; }
    void update(RtContext::SharedPtr context);
    // the device array of the motion matrices, nullptr before the first update
    const float *getMotionPtr() const { return mMotionBuffer ? static_cast<const float *>(mMotionBuffer->ptr()) : nullptr; }
    // update also describes deforming models (RtModel::setVertices): one rt_deformation_desc per instance with its model's
    // previous positions (NULL for a model that has none) and the row-major 3x4 of the instance's transform before this
    // update.  The device array, nullptr while no instance has previous positions.
    const rt_deformation_desc *getDeformationPtr() const {
        return mDeformBuffer ? static_cast<const rt_deformation_desc *>(mDeformBuffer->ptr()) : nullptr;
    }

private:
    RtScene() = default;
    struct Node {
        RtModel::SharedPtr model;
        DirectX::XMMATRIX transform;
    };
    std::vector<Node> mInstances;
    std::vector<DirectX::XMMATRIX> mBuiltTransforms;  // the transforms of the last build or update
    UINT mHitGroupCount = 0;
    RtBuffer::SharedPtr mTlasBuffer, mMotionBuffer, mDeformBuffer;
    void buildTlas(RtContext::SharedPtr context, bool performUpdate);
};

}  // namespace DXRFramework
