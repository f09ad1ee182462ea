// RtModel.h — headless counterpart of libs/DXRFramework/RtModel.h:8-38.
//
// A model is one interleaved {position, normal} vertex buffer (stride 24) + one uint32 index buffer + one BLAS
// (libs/DXRFramework/RtModel.cpp:13-17,73-118).  The reference loads any Assimp-supported file; only Assimp's
// headers and Windows binaries are vendored there, so this host always ships a built-in Wavefront OBJ reader
// (triangulation, per-mesh merge, smooth normals when the file has none — the post-processing RtModel.cpp:26
// asks Assimp for) and procedural creation from arrays, and compiles the Assimp path only when RT_HAVE_ASSIMP
// is defined and libassimp is available at build time.
#pragma once
#include "RtContext.h"

namespace DXRFramework {

struct Vertex {  // RtModel.cpp:13-17
    DirectX::XMFLOAT3 position;
    DirectX::XMFLOAT3 normal;
};

class RtModel {
public:
    using SharedPtr = std::shared_ptr<RtModel>;

    // Reference signature: create(context, filePath).  Unreadable files fall back to the reference's built-in
    // single triangle (RtModel.cpp:59-69).
    static SharedPtr create(RtContext::SharedPtr context, const std::string &filePath);
    // Procedural meshes (all BASELINE configs are synthetic).
    static SharedPtr create(RtContext::SharedPtr context, const std::vector<Vertex> &vertices, const std::vector<uint32_t> &indices);
    // Procedural-primitive model (D3D12_RAYTRACING_GEOMETRY_TYPE_PROCEDURAL_PRIMITIVE_AABBS, FL/LoadProceduralGeometry.hlsl):
    // 6 floats {min xyz, max xyz} per primitive; hit through an intersection shader of the hit group (RtContext::traceRays).
    static SharedPtr createProcedural(RtContext::SharedPtr context, const std::vector<float> &aabbs, bool opaque = true);
    ~RtModel();
    bool isProcedural() const { return mProcedural; }

    RtBuffer::SharedPtr getVertexBuffer() const { return mVertexBuffer; }
    RtBuffer::SharedPtr getIndexBuffer() const { return mIndexBuffer; }
    uint64_t getVertexBufferSrvHandle() const { return mVertexBufferSrvHandle; }
    uint64_t getIndexBufferSrvHandle() const { return mIndexBufferSrvHandle; }
    UINT getNumVertices() const { return mNumVertices; }
    UINT getNumTriangles() const { return mNumTriangles; }
    RtBuffer::SharedPtr getBlasBuffer() const { return mBlasBuffer; }

    // Deforming meshes (new work: the reference's models are static).  setDynamic(true) before the scene is built selects
    // RT_BUILD_FLAG_ALLOW_UPDATE for the BLAS (the default stays RT_BUILD_FLAG_NONE).  setVertices replaces every vertex
    // (same count and order) in the vertex buffer the hit records point to, refits the BLAS in place (PERFORM_UPDATE) and
    // makes the vertices from before the call the previous positions that RtScene::update describes for
    // rt_set_instance_deformation.  Call it once per frame, then RtScene::update, which refits the TLAS.
    void setDynamic(bool dynamic) { mDynamic = dynamic; }
    void setVertices(RtContext::SharedPtr context, const std::vector<Vertex> &vertices);
    const std::vector<Vertex> &getVertices() const { return mVertices; }  // the host copy of the current vertices
    // the device copy of the vertices before the last setVertices (stride sizeof(Vertex)), nullptr before the first
    const float *getPreviousPositionsPtr() const { return mPrevPositions ? static_cast<const float *>(mPrevPositions->ptr()) : nullptr; }

    // Parses an OBJ file into the interleaved layout; returns false if the file cannot be read.
    static bool loadObj(const std::string &path, std::vector<Vertex> &vertices, std::vector<uint32_t> &indices);
    // The reference's loader (RtModel.cpp:26-58): Assimp import with Triangulate | GenSmoothNormals | FlipUVs |
    // JoinIdenticalVertices | PreTransformVertices, all meshes merged with a per-mesh vertex offset.  Defined in
    // RtModelAssimp.cpp, compiled when RT_HAVE_ASSIMP is set (make ASSIMP_INCLUDE=... ASSIMP_LIB=...).
    static bool loadWithAssimp(const std::string &path, std::vector<Vertex> &vertices, std::vector<uint32_t> &indices);

private:
    friend class RtScene;
    RtModel(RtContext::SharedPtr context, std::vector<Vertex> vertices, std::vector<uint32_t> indices);
    void build(RtContext::SharedPtr context);  // RtModel.cpp:86-118

    bool mHasIndexBuffer = false;
    bool mProcedural = false, mOpaque = true, mDynamic = false;
    std::vector<Vertex> mVertices;
    UINT mNumVertices = 0;
    UINT mNumTriangles = 0;
    RtBuffer::SharedPtr mVertexBuffer, mIndexBuffer, mBlasBuffer, mPrevPositions;
    rt_geometry_desc geometryDesc() const;
    uint64_t mVertexBufferSrvHandle = 0, mIndexBufferSrvHandle = 0;
};

}  // namespace DXRFramework
