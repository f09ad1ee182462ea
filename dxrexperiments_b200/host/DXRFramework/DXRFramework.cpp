// DXRFramework.cpp — implementation of the headless DXRFramework layer over the rt_core C ABI.
// Mirrors the behaviour of libs/DXRFramework/Rt{Context,Model,Scene,Program,Params,Bindings}.cpp of the reference.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <fstream>
#include <map>
#include <chrono>
#include <sstream>
#include <thread>
#include <tuple>

#include "RtBindings.h"
#include "RtContext.h"
#include "RtModel.h"
#include "RtProgram.h"
#include "RtScene.h"

using namespace DirectX;

namespace DXRFramework {

// ============================================================================================ RtBuffer / RtContext
RtBuffer::RtBuffer(rt_context *ctx, uint64_t bytes) : mCtx(ctx), mBytes(bytes) { ThrowIfFailed(rt_malloc(ctx, bytes, &mPtr), "rt_malloc"); }
RtBuffer::~RtBuffer() {
    if (mPtr) rt_free(mCtx, mPtr);
}
void RtBuffer::upload(const void *host, uint64_t bytes, uint64_t offset) {
    ThrowIfFalse(offset + bytes <= mBytes, "RtBuffer::upload out of range");
    ThrowIfFailed(rt_upload(mCtx, static_cast<uint8_t *>(mPtr) + offset, host, bytes), "rt_upload");
    ThrowIfFailed(rt_sync(mCtx), "rt_sync");  // the source may be pageable and short-lived
}
void RtBuffer::download(void *host, uint64_t bytes, uint64_t offset) const {
    ThrowIfFalse(offset + bytes <= mBytes, "RtBuffer::download out of range");
    ThrowIfFailed(rt_download(mCtx, host, static_cast<const uint8_t *>(mPtr) + offset, bytes), "rt_download");
}
void RtBuffer::clear() { ThrowIfFailed(rt_memset(mCtx, mPtr, 0, mBytes), "rt_memset"); }

RtContext::SharedPtr RtContext::create(int deviceOrdinal) { return SharedPtr(new RtContext(deviceOrdinal)); }
RtContext::RtContext(int deviceOrdinal) { ThrowIfFailed(rt_context_create(deviceOrdinal, &mCtx), "rt_context_create"); }
RtContext::~RtContext() {
    rt_comm_destroy(mComm);
    rt_context_destroy(mCtx);
}

void RtContext::joinCommunicator(int worldSize, int rank, const std::string &idFile) {
    ThrowIfFalse(mComm == nullptr, "joinCommunicator: already joined");
    ThrowIfFalse(worldSize >= 1 && rank >= 0 && rank < worldSize && !idFile.empty(), "joinCommunicator: world / rank / id file");
    uint8_t id[RT_COMM_ID_BYTES];
    if (rank == 0) {
        ThrowIfFailed(rt_comm_get_unique_id(id), "rt_comm_get_unique_id");
        const std::string tmp = idFile + ".tmp";
        {
            std::ofstream f(tmp, std::ios::binary);
            f.write(reinterpret_cast<const char *>(id), sizeof(id));
            ThrowIfFalse(bool(f), "joinCommunicator: cannot write the id file");
        }
        ThrowIfFalse(std::rename(tmp.c_str(), idFile.c_str()) == 0, "joinCommunicator: cannot publish the id file");
    } else {
        bool got = false;
        for (int tries = 0; tries < 12000 && !got; ++tries) {  // up to two minutes
            std::ifstream f(idFile, std::ios::binary);
            if (f && f.read(reinterpret_cast<char *>(id), sizeof(id)) && f.gcount() == std::streamsize(sizeof(id))) got = true;
            else std::this_thread::sleep_for(std::chrono::milliseconds(10));
        }
        ThrowIfFalse(got, "joinCommunicator: no NCCL unique id appeared in the id file");
    }
    ThrowIfFailed(rt_comm_create(mCtx, id, worldSize, rank, &mComm), "rt_comm_create");
    mWorld = worldSize, mRank = rank;
}

void RtContext::reduceAccumulation(const RtBuffer::SharedPtr &send, const RtBuffer::SharedPtr &recv, uint64_t floats, float weight, int root) {
    ThrowIfFalse(mComm != nullptr, "reduceAccumulation: joinCommunicator first");
    ThrowIfFalse(send && send->size() >= floats * 4 && (!recv || recv->size() >= floats * 4), "reduceAccumulation: buffer sizes");
    ThrowIfFailed(rt_accum_reduce(mCtx, mComm, static_cast<const float *>(send->ptr()), recv ? static_cast<float *>(recv->ptr()) : nullptr, floats,
                                  weight, root), "rt_accum_reduce");
}

RtBuffer::SharedPtr RtContext::createBuffer(uint64_t bytes) { return RtBuffer::SharedPtr(new RtBuffer(mCtx, bytes)); }
RtBuffer::SharedPtr RtContext::createBuffer(const void *initialData, uint64_t bytes) {
    auto b = createBuffer(bytes);
    if (bytes) b->upload(initialData, bytes);
    return b;
}
void RtContext::waitForGpu() { ThrowIfFailed(rt_sync(mCtx), "rt_sync"); }
void RtContext::checkDeviceStatus() { ThrowIfFailed(rt_get_status(mCtx), "rt_get_status"); }
uint64_t RtContext::launchCount() const { return rt_launch_count(mCtx); }

void RtContext::raytrace(std::shared_ptr<RtBindings> bindings, std::shared_ptr<RtState> state, uint32_t width, uint32_t height, uint32_t depth) {
    ThrowIfFalse(bindings && state && state->getProgram(), "raytrace: bindings/state without a program");
    ThrowIfFailed(rt_dispatch_rays(mCtx, state->getProgram()->getNative(), width, height, depth), "rt_dispatch_rays");
}

void RtContext::raytraceStrips(std::shared_ptr<RtBindings> bindings, std::shared_ptr<RtState> state, uint32_t width, uint32_t height,
                               uint32_t stripRows, uint32_t groups, uint32_t group) {
    ThrowIfFalse(bindings && state && state->getProgram(), "raytraceStrips: bindings/state without a program");
    ThrowIfFailed(rt_dispatch_rays_interleaved(mCtx, state->getProgram()->getNative(), width, height, stripRows, groups, group),
                  "rt_dispatch_rays_interleaved");
}

void RtContext::raytraceRegion(std::shared_ptr<RtBindings> bindings, std::shared_ptr<RtState> state, uint32_t width, uint32_t height,
                               uint32_t x0, uint32_t y0, uint32_t x1, uint32_t y1) {
    ThrowIfFalse(bindings && state && state->getProgram(), "raytraceRegion: bindings/state without a program");
    ThrowIfFailed(rt_dispatch_rays_region(mCtx, state->getProgram()->getNative(), width, height, x0, y0, x1, y1), "rt_dispatch_rays_region");
}

void RtContext::traceRays(std::shared_ptr<RtProgram> program, std::shared_ptr<RtScene> scene, const rt_ray *rays, uint64_t n, uint32_t rayFlags,
                          uint32_t instanceMask, uint32_t rayContribution, uint32_t geometryMultiplier, rt_hit *hits) {
    ThrowIfFalse(program && scene && scene->getTlasWrappedPtr(), "traceRays: program / built scene");
    ThrowIfFalse(n == 0 || (rays && hits), "traceRays: null ray or hit array");
    // one table entry per shader-table hit record: [instance][ray type], as RtBindings lays them out (RtBindings.cpp:131-164)
    const uint32_t groups = program->getHitProgramCount();
    std::vector<rt_hit_group_programs> table(size_t(scene->getNumInstances()) * groups);
    for (size_t r = 0; r < table.size(); ++r) table[r] = program->getHitGroupPrograms(uint32_t(r % groups));
    auto dRays = createBuffer(rays, std::max<uint64_t>(n * sizeof(rt_ray), 32));
    auto dHits = createBuffer(std::max<uint64_t>(n * sizeof(rt_hit), 32));
    ThrowIfFailed(rt_trace_rays_hit_groups(mCtx, scene->getTlasWrappedPtr(), static_cast<const rt_ray *>(dRays->ptr()), n, rayFlags, instanceMask,
                                           rayContribution, geometryMultiplier, table.data(), uint32_t(table.size()),
                                           static_cast<rt_hit *>(dHits->ptr())), "rt_trace_rays_hit_groups");
    if (n) dHits->download(hits, n * sizeof(rt_hit));
    checkDeviceStatus();
}

// ============================================================================================ RtModel
static XMFLOAT3 sub(XMFLOAT3 a, XMFLOAT3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
static XMFLOAT3 cross(XMFLOAT3 a, XMFLOAT3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

bool RtModel::loadObj(const std::string &path, std::vector<Vertex> &vertices, std::vector<uint32_t> &indices) {
    std::ifstream in(path);
    if (!in) return false;
    std::vector<XMFLOAT3> pos, nrm;
    std::map<std::pair<int, int>, uint32_t> remap;  // (position, normal) -> merged vertex (JoinIdenticalVertices)
    bool missingNormals = false;
    std::string line;
    auto resolve = [](int idx, size_t count) { return idx > 0 ? idx - 1 : int(count) + idx; };
    while (std::getline(in, line)) {
        std::istringstream ls(line);
        std::string tag;
        ls >> tag;
        if (tag == "v") {
            XMFLOAT3 p{};
            ls >> p.x >> p.y >> p.z;
            pos.push_back(p);
        } else if (tag == "vn") {
            XMFLOAT3 n{};
            ls >> n.x >> n.y >> n.z;
            nrm.push_back(n);
        } else if (tag == "f") {
            std::vector<uint32_t> face;
            std::string tok;
            while (ls >> tok) {
                int vi = 0, ni = 0;
                size_t s1 = tok.find('/');
                vi = std::stoi(tok.substr(0, s1));
                if (s1 != std::string::npos) {
                    size_t s2 = tok.find('/', s1 + 1);
                    if (s2 != std::string::npos && s2 + 1 < tok.size()) ni = std::stoi(tok.substr(s2 + 1));
                }
                int p = resolve(vi, pos.size());
                int n = ni != 0 ? resolve(ni, nrm.size()) : -1;
                if (p < 0 || p >= int(pos.size())) return false;
                if (n < 0) missingNormals = true;
                auto key = std::make_pair(p, n);
                auto it = remap.find(key);
                if (it == remap.end()) {
                    Vertex v{pos[p], n >= 0 && n < int(nrm.size()) ? nrm[n] : XMFLOAT3{0, 0, 0}};
                    it = remap.emplace(key, uint32_t(vertices.size())).first;
                    vertices.push_back(v);
                }
                face.push_back(it->second);
            }
            for (size_t k = 1; k + 1 < face.size(); ++k) {  // aiProcess_Triangulate: fan
                indices.push_back(face[0]);
                indices.push_back(face[k]);
                indices.push_back(face[k + 1]);
            }
        }
    }
    if (missingNormals) {  // aiProcess_GenSmoothNormals: area-weighted vertex normals
        std::vector<XMFLOAT3> acc(vertices.size(), XMFLOAT3{0, 0, 0});
        for (size_t t = 0; t + 2 < indices.size(); t += 3) {
            XMFLOAT3 n = cross(sub(vertices[indices[t + 1]].position, vertices[indices[t]].position),
                               sub(vertices[indices[t + 2]].position, vertices[indices[t]].position));
            for (int k = 0; k < 3; ++k) {
                XMFLOAT3 &a = acc[indices[t + k]];
                a.x += n.x, a.y += n.y, a.z += n.z;
            }
        }
        for (size_t i = 0; i < vertices.size(); ++i) {
            float l = sqrtf(acc[i].x * acc[i].x + acc[i].y * acc[i].y + acc[i].z * acc[i].z);
            if (l > 0) vertices[i].normal = {acc[i].x / l, acc[i].y / l, acc[i].z / l};
        }
    }
    return !indices.empty();
}

RtModel::SharedPtr RtModel::create(RtContext::SharedPtr context, const std::string &filePath) {
    std::vector<Vertex> vertices;
    std::vector<uint32_t> indices;
    bool ok = false;
    const bool isObj = filePath.size() > 4 && (filePath.substr(filePath.size() - 4) == ".obj" || filePath.substr(filePath.size() - 4) == ".OBJ");
    if (isObj) ok = loadObj(filePath, vertices, indices);
#if defined(RT_HAVE_ASSIMP)
    if (!ok) ok = loadWithAssimp(filePath, vertices, indices);
#endif
    if (!ok) {
        // the reference's fallback when aiImportFile fails (RtModel.cpp:59-69)
        vertices = {{{0.0f, 0.25f, 0.0f}, {0.0f, 0.0f, 1.0f}}, {{0.25f, -0.25f, 0.0f}, {0.0f, 0.0f, 1.0f}}, {{-0.25f, -0.25f, 0.0f}, {0.0f, 0.0f, 1.0f}}};
        indices = {0, 2, 1};
    }
    return SharedPtr(new RtModel(context, std::move(vertices), std::move(indices)));
}

RtModel::SharedPtr RtModel::create(RtContext::SharedPtr context, const std::vector<Vertex> &vertices, const std::vector<uint32_t> &indices) {
    return SharedPtr(new RtModel(context, vertices, indices));
}

RtModel::RtModel(RtContext::SharedPtr context, std::vector<Vertex> vertices, std::vector<uint32_t> indices) {
    mNumVertices = static_cast<UINT>(vertices.size());
    mNumTriangles = static_cast<UINT>(indices.size() / 3);
    mHasIndexBuffer = !indices.empty();
    ThrowIfFalse(mNumVertices > 0, "RtModel: empty vertex buffer");
    mVertexBuffer = context->createBuffer(vertices.data(), vertices.size() * sizeof(Vertex));
    mVertices = std::move(vertices);
    if (mHasIndexBuffer) mIndexBuffer = context->createBuffer(indices.data(), indices.size() * sizeof(uint32_t));
    else {  // the hit shaders always read an index buffer (Load3x32BitIndices): synthesise 0,1,2,...
        std::vector<uint32_t> iota(mNumVertices);
        for (UINT i = 0; i < mNumVertices; ++i) iota[i] = i;
        mIndexBuffer = context->createBuffer(iota.data(), iota.size() * sizeof(uint32_t));
        mNumTriangles = mNumVertices / 3;
    }
}

RtModel::~RtModel() = default;

RtModel::SharedPtr RtModel::createProcedural(RtContext::SharedPtr context, const std::vector<float> &aabbs, bool opaque) {
    ThrowIfFalse(!aabbs.empty() && aabbs.size() % 6 == 0, "createProcedural: 6 floats {min, max} per AABB");
    // the AABB buffer takes the place of the vertex buffer (stride 24 = D3D12_RAYTRACING_AABB); there is no index buffer,
    // but closest-hit records still bind one, so a one-element placeholder keeps the record complete
    std::vector<Vertex> boxes(aabbs.size() / 6);
    std::memcpy(boxes.data(), aabbs.data(), aabbs.size() * sizeof(float));
    SharedPtr m(new RtModel(context, std::move(boxes), {}));
    m->mProcedural = true;
    m->mOpaque = opaque;
    m->mNumTriangles = m->mNumVertices;  // primitives
    return m;
}

rt_geometry_desc RtModel::geometryDesc() const {
    // blasGenerator.AddVertexBuffer(VB, 0, nVerts, sizeof(Vertex), IB, 0, nTris*3, R32_UINT, nullptr, 0), opaque
    rt_geometry_desc g{};
    g.vertex_buffer = mVertexBuffer->ptr();
    g.vertex_count = mNumVertices;
    g.vertex_stride_bytes = sizeof(Vertex);
    if (mProcedural) {
        g.type = RT_GEOMETRY_TYPE_PROCEDURAL_AABBS;
    } else {
        g.index_buffer = mIndexBuffer->ptr();
        g.index_count = mNumTriangles * 3;
        g.index_format = 32;
    }
    g.transform3x4 = nullptr;
    g.flags = mOpaque ? RT_GEOMETRY_FLAG_OPAQUE : RT_GEOMETRY_FLAG_NONE;
    return g;
}

void RtModel::build(RtContext::SharedPtr context) {
    const rt_geometry_desc g = geometryDesc();
    const uint32_t flags = mDynamic ? RT_BUILD_FLAG_ALLOW_UPDATE : RT_BUILD_FLAG_NONE;  // the reference: no update
    rt_prebuild_info info{};
    ThrowIfFailed(rt_blas_prebuild(context->getNative(), &g, 1, flags, &info), "rt_blas_prebuild");
    auto scratch = context->createBuffer(info.scratch_bytes);
    mBlasBuffer = context->createBuffer(info.result_bytes);
    ThrowIfFailed(rt_blas_build(context->getNative(), &g, 1, flags, scratch->ptr(), scratch->size(), mBlasBuffer->ptr(),
                                mBlasBuffer->size()), "rt_blas_build");
    context->waitForGpu();  // scratch goes out of scope, as after WaitForGpu in the reference
    mVertexBufferSrvHandle = context->createBufferSRVHandle(mVertexBuffer);
    mIndexBufferSrvHandle = context->createBufferSRVHandle(mIndexBuffer);
}

void RtModel::setVertices(RtContext::SharedPtr context, const std::vector<Vertex> &vertices) {
    ThrowIfFalse(mDynamic && !mProcedural && mBlasBuffer, "RtModel::setVertices needs a triangle model built after setDynamic(true)");
    ThrowIfFalse(vertices.size() == mVertices.size(), "RtModel::setVertices: the vertex count must not change");
    const uint64_t bytes = mVertices.size() * sizeof(Vertex);
    if (!mPrevPositions) mPrevPositions = context->createBuffer(bytes);
    mPrevPositions->upload(mVertices.data(), bytes);
    mVertexBuffer->upload(vertices.data(), bytes);
    mVertices = vertices;
    const rt_geometry_desc g = geometryDesc();
    rt_prebuild_info info{};
    ThrowIfFailed(rt_blas_prebuild(context->getNative(), &g, 1, RT_BUILD_FLAG_ALLOW_UPDATE, &info), "rt_blas_prebuild");
    auto scratch = context->createBuffer(std::max<uint64_t>(info.update_scratch_bytes ? info.update_scratch_bytes : info.scratch_bytes, 16));
    ThrowIfFailed(rt_blas_build(context->getNative(), &g, 1, RT_BUILD_FLAG_ALLOW_UPDATE | RT_BUILD_FLAG_PERFORM_UPDATE, scratch->ptr(),
                                scratch->size(), mBlasBuffer->ptr(), mBlasBuffer->size()), "rt_blas_build (update)");
    context->waitForGpu();
}

// ============================================================================================ RtScene
void RtScene::build(RtContext::SharedPtr context, UINT hitGroupCount) {
    mHitGroupCount = hitGroupCount;
    buildTlas(context, false);
}

// the instance desc's row-major 3x4 (the transpose of the row-vector XMMATRIX, TopLevelASGenerator.cpp:353-355) in double
static void affine3x4(const XMMATRIX &transform, double out[12]) {
    float m[16];
    const XMMATRIX t = XMMatrixTranspose(transform);
    std::memcpy(m, &t, sizeof(m));
    for (int k = 0; k < 12; ++k) out[k] = m[k];
}

void RtScene::update(RtContext::SharedPtr context) {
    const size_t n = mInstances.size();
    std::vector<float> motion(12 * std::max<size_t>(n, 1));
    for (size_t i = 0; i < n; ++i) {
        double p[12], c[12], inv[12], r[12];
        affine3x4(mBuiltTransforms[i], p);
        affine3x4(mInstances[i].transform, c);
        // inverse of [A t]: [A^-1, -A^-1 t], A^-1 = adj(A) / det(A)
        const double a00 = c[0], a01 = c[1], a02 = c[2], a10 = c[4], a11 = c[5], a12 = c[6], a20 = c[8], a21 = c[9], a22 = c[10];
        const double det = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20);
        ThrowIfFalse(det != 0.0 && std::isfinite(det), "RtScene::update: an instance transform is not invertible");
        const double adj[9] = {a11 * a22 - a12 * a21, a02 * a21 - a01 * a22, a01 * a12 - a02 * a11,
                               a12 * a20 - a10 * a22, a00 * a22 - a02 * a20, a02 * a10 - a00 * a12,
                               a10 * a21 - a11 * a20, a01 * a20 - a00 * a21, a00 * a11 - a01 * a10};
        for (int row = 0; row < 3; ++row) {
            for (int col = 0; col < 3; ++col) inv[4 * row + col] = adj[3 * row + col] / det;
            inv[4 * row + 3] = -(inv[4 * row] * c[3] + inv[4 * row + 1] * c[7] + inv[4 * row + 2] * c[11]);
        }
        for (int row = 0; row < 3; ++row) {
            for (int col = 0; col < 4; ++col)
                r[4 * row + col] = p[4 * row] * inv[col] + p[4 * row + 1] * inv[4 + col] + p[4 * row + 2] * inv[8 + col] + (col == 3 ? p[4 * row + 3] : 0.0);
        }
        for (int k = 0; k < 12; ++k) motion[12 * i + k] = float(r[k]);
    }
    if (!mMotionBuffer) mMotionBuffer = context->createBuffer(motion.data(), motion.size() * sizeof(float));
    else mMotionBuffer->upload(motion.data(), motion.size() * sizeof(float));
    // deforming models: their previous positions and the transforms before this update (rt_set_instance_deformation)
    std::vector<rt_deformation_desc> deform(std::max<size_t>(n, 1));
    bool deforming = false;
    for (size_t i = 0; i < n; ++i) {
        const RtModel &m = *mInstances[i].model;
        rt_deformation_desc &d = deform[i];
        std::memset(&d, 0, sizeof(d));
        d.previous_positions = m.getPreviousPositionsPtr();
        d.stride_bytes = sizeof(Vertex);
        d.vertex_count = m.mNumVertices;
        double p[12];
        affine3x4(mBuiltTransforms[i], p);
        for (int k = 0; k < 12; ++k) d.object_to_previous_world[k] = float(p[k]);
        deforming = deforming || d.previous_positions;
    }
    if (!deforming) mDeformBuffer.reset();
    else if (!mDeformBuffer) mDeformBuffer = context->createBuffer(deform.data(), deform.size() * sizeof(rt_deformation_desc));
    else mDeformBuffer->upload(deform.data(), deform.size() * sizeof(rt_deformation_desc));
    buildTlas(context, true);
}

void RtScene::buildTlas(RtContext::SharedPtr context, bool performUpdate) {
    std::vector<rt_instance_desc> descs(mInstances.size());
    for (size_t i = 0; i < mInstances.size(); ++i) {
        if (!mInstances[i].model->mBlasBuffer) mInstances[i].model->build(context);
        rt_instance_desc &d = descs[i];
        std::memset(&d, 0, sizeof(d));
        // the instance desc is row major 3x4 = the transpose of the row-vector XMMATRIX (TopLevelASGenerator.cpp:353-355)
        XMMATRIX m = XMMatrixTranspose(mInstances[i].transform);
        std::memcpy(d.transform, &m, sizeof(d.transform));
        d.instance_id_and_mask = (uint32_t(i) & 0xFFFFFFu) | (0xFFu << 24);
        d.hit_group_and_flags = (uint32_t(i * mHitGroupCount) & 0xFFFFFFu) | (uint32_t(RT_INSTANCE_FLAG_NONE) << 24);
        d.blas = reinterpret_cast<uint64_t>(mInstances[i].model->mBlasBuffer->ptr());
    }
    const uint32_t n = static_cast<uint32_t>(descs.size());
    rt_prebuild_info info{};
    ThrowIfFailed(rt_tlas_prebuild(context->getNative(), n, RT_BUILD_FLAG_ALLOW_UPDATE, &info), "rt_tlas_prebuild");
    auto scratch = context->createBuffer(std::max<uint64_t>(performUpdate && info.update_scratch_bytes ? info.update_scratch_bytes : info.scratch_bytes, 16));
    if (!performUpdate) mTlasBuffer = context->createBuffer(info.result_bytes);
    auto instanceDesc = context->createBuffer(descs.data(), std::max<uint64_t>(sizeof(rt_instance_desc) * n, 64));
    const uint32_t flags = uint32_t(RT_BUILD_FLAG_ALLOW_UPDATE) | (performUpdate ? uint32_t(RT_BUILD_FLAG_PERFORM_UPDATE) : 0u);
    ThrowIfFailed(rt_tlas_build(context->getNative(), static_cast<const rt_instance_desc *>(instanceDesc->ptr()), n, flags, scratch->ptr(),
                                scratch->size(), mTlasBuffer->ptr(), mTlasBuffer->size()), "rt_tlas_build");
    context->waitForGpu();
    mBuiltTransforms.clear();
    for (const Node &node : mInstances) mBuiltTransforms.push_back(node.transform);
}

// ============================================================================================ RtProgram
const uint8_t kProgressiveRaytracingLibrary[] = "rt_core:ProgressiveRaytracing";
const UINT kProgressiveRaytracingLibrarySize = sizeof(kProgressiveRaytracingLibrary);
const uint8_t kRealtimeRaytracingLibrary[] = "rt_core:RealtimeRaytracing";
const UINT kRealtimeRaytracingLibrarySize = sizeof(kRealtimeRaytracingLibrary);
const uint8_t kHitGroupProgramsLibrary[] = "rt_core:HitGroupPrograms";
const UINT kHitGroupProgramsLibrarySize = sizeof(kHitGroupProgramsLibrary);

static const char *kLibraryExports[] = {"RayGen", "PrimaryClosestHit", "PrimaryMiss", "ShadowClosestHit", "ShadowAnyHit", "ShadowMiss"};
// exports of kHitGroupProgramsLibrary and the program ids they stand for (include/rt_types.h)
static const struct {
    const char *name;
    RtShader::Type type;
    uint32_t id;
} kHitGroupExports[] = {{"AnyHitAccept", RtShader::Type::AnyHit, RT_ANYHIT_ACCEPT},          {"AnyHitIgnore", RtShader::Type::AnyHit, RT_ANYHIT_IGNORE},
                        {"AnyHitEndSearch", RtShader::Type::AnyHit, RT_ANYHIT_END_SEARCH},   {"AnyHitCutout", RtShader::Type::AnyHit, RT_ANYHIT_CUTOUT},
                        {"IntersectBox", RtShader::Type::Intersection, RT_INTERSECTION_BOX}, {"IntersectSphere", RtShader::Type::Intersection, RT_INTERSECTION_SPHERE},
                        {"ProceduralClosestHit", RtShader::Type::ClosestHit, 0}};

static uint32_t anyHitId(const std::string &name) {
    if (name.empty()) return RT_ANYHIT_NONE;
    if (name == "ShadowAnyHit") return RT_ANYHIT_ACCEPT;  // the application's no-op any-hit shader (ProgressiveRaytracing.hlsl:172-176)
    for (const auto &e : kHitGroupExports)
        if (e.type == RtShader::Type::AnyHit && name == e.name) return e.id;
    throw std::logic_error("'" + name + "' is not an any-hit shader");
}
static uint32_t intersectionId(const std::string &name) {
    if (name.empty()) return RT_INTERSECTION_NONE;
    for (const auto &e : kHitGroupExports)
        if (e.type == RtShader::Type::Intersection && name == e.name) return e.id;
    throw std::logic_error("'" + name + "' is not an intersection shader");
}

UINT RootSignatureGenerator::argumentBytes() const {
    UINT off = 0;
    for (const auto &p : mParams) {
        if (p.type == RootParameterType::Constants32Bit) {
            off = (off + 3u) & ~3u;
            off += 4 * p.numConstants;
        } else {
            off = (off + 7u) & ~7u;
            off += 8;
        }
    }
    return off;
}

static std::string narrow(const std::wstring &w) { return std::string(w.begin(), w.end()); }

RtProgram::Desc &RtProgram::Desc::addShaderLibrary(const uint8_t *bytecode, UINT bytecodeSize, const std::vector<std::wstring> &symbolExports) {
    ThrowIfFalse(bytecode != nullptr, "addShaderLibrary: null library");
    const std::string token(reinterpret_cast<const char *>(bytecode), strnlen(reinterpret_cast<const char *>(bytecode), bytecodeSize));
    bool hitGroupLibrary = false;
    if (token == reinterpret_cast<const char *>(kProgressiveRaytracingLibrary)) mLibrary = RT_PROGRAM_PROGRESSIVE;
    else if (token == reinterpret_cast<const char *>(kRealtimeRaytracingLibrary)) mLibrary = RT_PROGRAM_REALTIME;
    else if (token == reinterpret_cast<const char *>(kHitGroupProgramsLibrary)) hitGroupLibrary = true;
    else throw std::logic_error("addShaderLibrary: unknown shader library (shaders are compiled into librt_core.so; pass "
                                "kProgressiveRaytracingLibrary, kRealtimeRaytracingLibrary or kHitGroupProgramsLibrary)");
    for (const auto &w : symbolExports) {
        std::string e = narrow(w);
        bool known = false;
        if (hitGroupLibrary) {
            for (const auto &k : kHitGroupExports) known |= (e == k.name);
        } else {
            for (const char *k : kLibraryExports) known |= (e == k);
        }
        if (!known) throw std::logic_error("addShaderLibrary: the library does not export '" + e + "'");
        mExports.push_back(e);
    }
    return *this;
}

static void requireExport(const std::vector<std::string> &exports, const std::string &name) {
    if (name.empty()) return;
    if (std::find(exports.begin(), exports.end(), name) == exports.end())
        throw std::logic_error("unknown shader identifier '" + name + "'");  // RtBindings.cpp:77-79 throws the same way
}

RtProgram::Desc &RtProgram::Desc::setRayGen(const std::string &raygen) {
    requireExport(mExports, raygen);
    mRayGen = raygen;
    return *this;
}
RtProgram::Desc &RtProgram::Desc::addMiss(uint32_t missIndex, const std::string &miss) {
    requireExport(mExports, miss);
    if (missIndex >= mMiss.size()) mMiss.resize(missIndex + 1);
    mMiss[missIndex] = miss;
    return *this;
}
RtProgram::Desc &RtProgram::Desc::addHitGroup(uint32_t hitIndex, const std::string &closestHit, const std::string &anyHit, const std::string &intersection) {
    requireExport(mExports, closestHit);
    requireExport(mExports, anyHit);
    requireExport(mExports, intersection);
    (void)anyHitId(anyHit), (void)intersectionId(intersection);  // the names must be shaders of the right kind
    ThrowIfFalse(hitIndex < 8, "addHitGroup: at most 8 hit groups");
    if (hitIndex >= mHit.size()) mHit.resize(hitIndex + 1);
    mHit[hitIndex] = {intersection, anyHit, closestHit};
    return *this;
}
RtProgram::Desc &RtProgram::Desc::configureGlobalRootSignature(RootSignatureConfigurator c) { c(mGlobalRootSignatureConfig); return *this; }
RtProgram::Desc &RtProgram::Desc::configureRayGenRootSignature(RootSignatureConfigurator c) { c(mRayGenRootSignatureConfig); return *this; }
RtProgram::Desc &RtProgram::Desc::configureHitGroupRootSignature(RootSignatureConfigurator c) { c(mHitGroupRootSignatureConfig); return *this; }
RtProgram::Desc &RtProgram::Desc::configureMissRootSignature(RootSignatureConfigurator c) { c(mMissRootSignatureConfig); return *this; }

RtProgram::SharedPtr RtProgram::create(RtContext::SharedPtr context, const Desc &desc, uint32_t, uint32_t) { return SharedPtr(new RtProgram(context, desc)); }

RtProgram::RtProgram(RtContext::SharedPtr context, const Desc &desc) : mDesc(desc), mContext(context) {
    ThrowIfFalse(desc.mLibrary >= 0, "RtProgram: no shader library");
    ThrowIfFalse(desc.mRayGen == "RayGen", "RtProgram: the ray generation shader must be 'RayGen'");
    // ray types 0 and 1 are the pipelines' own (primary, shadow); further hit groups (procedural geometry, other any-hit
    // behaviour) are reached through RtContext::traceRays
    ThrowIfFalse(desc.mHit.size() >= 2 && desc.mHit.size() <= 8 && desc.mMiss.size() == 2,
                 "RtProgram: the pipeline libraries define hit groups 0 (primary) and 1 (shadow) and 2 miss shaders");
    ThrowIfFalse(desc.mHit[0].closestHit == "PrimaryClosestHit" && desc.mMiss[0] == "PrimaryMiss" && desc.mHit[1].closestHit == "ShadowClosestHit" &&
                     desc.mMiss[1] == "ShadowMiss",
                 "RtProgram: ray type 0 must be the primary hit group/miss, ray type 1 the shadow one");
    mKind = static_cast<rt_program_kind>(desc.mLibrary);
    mRayGenProgram = std::make_shared<RtShader>(RtShader::Type::RayGeneration, desc.mRayGen);
    for (size_t i = 0; i < desc.mHit.size(); ++i) {
        HitGroup g;
        g.mClosestHit = std::make_shared<RtShader>(RtShader::Type::ClosestHit, desc.mHit[i].closestHit);
        if (!desc.mHit[i].anyHit.empty()) g.mAnyHit = std::make_shared<RtShader>(RtShader::Type::AnyHit, desc.mHit[i].anyHit);
        if (!desc.mHit[i].intersection.empty()) g.mIntersection = std::make_shared<RtShader>(RtShader::Type::Intersection, desc.mHit[i].intersection);
        g.mExportName = "HitGroup" + std::to_string(i);
        mHitPrograms.push_back(g);
    }
    for (const auto &m : desc.mMiss) mMissPrograms.push_back(std::make_shared<RtShader>(RtShader::Type::Miss, m));
    ThrowIfFailed(rt_program_create(context->getNative(), mKind, getHitProgramCount(), getMissProgramCount(), &mProgram), "rt_program_create");
}

RtProgram::~RtProgram() { rt_program_destroy(mProgram); }

rt_hit_group_programs RtProgram::getHitGroupPrograms(uint32_t rayIndex) const {
    const HitGroup &g = mHitPrograms.at(rayIndex);
    rt_hit_group_programs p{};
    p.any_hit = anyHitId(g.mAnyHit ? g.mAnyHit->getEntryPoint() : std::string());
    p.intersection = intersectionId(g.mIntersection ? g.mIntersection->getEntryPoint() : std::string());
    return p;
}

// ============================================================================================ RtParams / RtBindings
void RtParams::write(const void *src, UINT size, UINT alignment) {
    mRootOffset = (mRootOffset + alignment - 1) / alignment * alignment;
    const UINT at = mRootOffset - mInitialOffset;
    if (mData.size() < at + size) throw std::logic_error("RtParams: writing shader params out of bounds");
    std::memcpy(mData.data() + at, src, size);
    mRootOffset += size;
}
void RtParams::appendHeapRanges(UINT64 gpuHandle) { write(&gpuHandle, sizeof(UINT64), sizeof(UINT64)); }
void RtParams::append32BitConstants(const void *constants, UINT n) { write(constants, sizeof(uint32_t) * n, sizeof(uint32_t)); }
UINT RtParams::applyRootParams(uint8_t *record) {
    const UINT n = mRootOffset - mInitialOffset;
    std::memcpy(record, mData.data(), n);
    mRootOffset = mInitialOffset;
    return n;
}

RtBindings::RtBindings(RtContext::SharedPtr, RtProgram::SharedPtr program, RtScene::SharedPtr scene) : mProgram(program), mScene(scene) {
    mHitProgCount = program->getHitProgramCount();
    mMissProgCount = program->getMissProgramCount();
    mFirstHitVarEntry = 1 + mMissProgCount;
    const UINT maxRootSigSize = std::max<UINT>(80, std::max(program->getHitGroupArgumentBytes(), program->getMissArgumentBytes()));
    mRayGenParams = RtParams::create(kProgramIdentifierSize);
    mRayGenParams->allocateStorage(maxRootSigSize);
    const UINT instances = scene->getNumInstances();
    mHitParams.resize(mHitProgCount);
    for (UINT h = 0; h < mHitProgCount; ++h)
        for (UINT i = 0; i < instances; ++i) {
            mHitParams[h].push_back(RtParams::create(kProgramIdentifierSize));
            mHitParams[h].back()->allocateStorage(maxRootSigSize);
        }
    for (UINT m = 0; m < mMissProgCount; ++m) {
        mMissParams.push_back(RtParams::create(kProgramIdentifierSize));
        mMissParams.back()->allocateStorage(maxRootSigSize);
    }
    mRecordSize = (kProgramIdentifierSize + maxRootSigSize + 31u) & ~31u;  // D3D12_RAYTRACING_SHADER_RECORD_BYTE_ALIGNMENT
    mShaderTableData.assign(size_t(mRecordSize) * (1 + mMissProgCount + mHitProgCount * instances), 0);
}

void RtBindings::apply(RtContext::SharedPtr, RtState::SharedPtr state) {
    ThrowIfFalse(state && state->getProgram() == mProgram, "RtBindings::apply: state holds a different program");
    rt_program *prog = mProgram->getNative();
    // records carry the entry point name where the reference stores the 32-byte shader identifier
    auto stamp = [&](uint8_t *rec, const std::string &name) {
        std::memset(rec, 0, kProgramIdentifierSize);
        std::memcpy(rec, name.data(), std::min<size_t>(name.size(), kProgramIdentifierSize - 1));
    };
    stamp(recordPtr(0), mProgram->getRayGenProgram()->getEntryPoint());
    mRayGenParams->applyRootParams(recordPtr(0) + kProgramIdentifierSize);
    for (UINT h = 0; h < mHitProgCount; ++h) {
        for (UINT i = 0; i < mScene->getNumInstances(); ++i) {
            uint8_t *rec = recordPtr(mFirstHitVarEntry + mHitProgCount * i + h);
            stamp(rec, mProgram->getHitProgram(h).mClosestHit->getEntryPoint());
            const UINT n = mHitParams[h][i]->applyRootParams(rec + kProgramIdentifierSize);
            if (n == 0) continue;  // nothing appended this frame: the record keeps its previous arguments
            if (n < 16 + sizeof(rt_material_params)) throw std::logic_error("hit record needs {VB handle, IB handle, MaterialParams}");
            UINT64 vb, ib;
            rt_material_params mat;
            std::memcpy(&vb, rec + kProgramIdentifierSize, 8);
            std::memcpy(&ib, rec + kProgramIdentifierSize + 8, 8);
            std::memcpy(&mat, rec + kProgramIdentifierSize + 16, sizeof(mat));
            ThrowIfFailed(rt_bindings_set_hit_record(prog, h, i, reinterpret_cast<const void *>(vb), reinterpret_cast<const void *>(ib), &mat),
                          "rt_bindings_set_hit_record");
        }
    }
    for (UINT m = 0; m < mMissProgCount; ++m) {
        uint8_t *rec = recordPtr(1 + m);
        stamp(rec, mProgram->getMissProgram(m)->getEntryPoint());
        const UINT n = mMissParams[m]->applyRootParams(rec + kProgramIdentifierSize);
        if (n < 16) continue;
        UINT64 cube;
        std::memcpy(&cube, rec + kProgramIdentifierSize + 8, 8);  // {envMap t0, envCubemap t1}: only the cube is sampled
        const RtTexture *tex = reinterpret_cast<const RtTexture *>(cube);
        ThrowIfFailed(rt_bindings_set_miss_record(prog, m, tex && tex->texels ? static_cast<const float *>(tex->texels->ptr()) : nullptr, tex ? tex->size : 0),
                      "rt_bindings_set_miss_record");
    }
}

}  // namespace DXRFramework
