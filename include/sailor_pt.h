/*
 * sailor_pt.h — C-ABI of the B200 path tracer that replaces Sailor's CPU path tracer (Runtime/Raytracing).
 *
 * The reference has no FFI for this path: its only surface is the C++ class
 *     Sailor::Raytracing::PathTracer { struct Params; static ParseCommandLineArgs(...); void Run(const Params&); }
 * (reference Runtime/Raytracing/PathTracer.h:17-36).  This header follows the reference's existing C export
 * convention (reference Lib/DllMain.cpp:9-144: extern "C", POD arguments only, failures by return value, no
 * exceptions across the boundary) and keeps Params field-for-field (PathTracer.h:21-32).
 *
 * Two libraries export exactly this set:
 *   - sailor_b200/libsailor_pt_cuda.so : the product (CUDA, sm_100a).  No CPU fallback: every entry point that
 *     computes returns SAILOR_PT_ERR_NO_DEVICE when no CUDA device is usable.
 *   - oracle/_ref/libsailor_pt_ref.so  : the test oracle (the reference's own C++ compiled with g++), used only
 *     by tests/, smoke() and the bench's CPU-baseline legs.
 *
 * All buffers are caller-allocated host memory unless a name ends in `Device`.
 */
#ifndef SAILOR_PT_H
#define SAILOR_PT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define SAILOR_PT_API __declspec(dllexport)
#else
#define SAILOR_PT_API __attribute__((visibility("default")))
#endif

/* ---- error codes (negative = failure, like the reference's bool/count returns in Lib/DllMain.cpp:78-137) ---- */
enum {
	SAILOR_PT_OK = 0,
	SAILOR_PT_ERR_ARG = -1,        /* null / inconsistent argument */
	SAILOR_PT_ERR_IO = -2,         /* file missing / unreadable / unwritable */
	SAILOR_PT_ERR_FORMAT = -3,     /* glTF / PNG content not understood */
	SAILOR_PT_ERR_NO_DEVICE = -4,  /* product only: CUDA device or kernel image unavailable */
	SAILOR_PT_ERR_CUDA = -5,       /* product only: a CUDA call failed (message via SailorPt_LastError) */
	SAILOR_PT_ERR_LIMIT = -6,      /* > 256 materials / > 255 textures (reference u8 slots, MaterialUtils.h:157-174) */
	SAILOR_PT_ERR_UNSUPPORTED = -7
};

/* Mirrors PathTracer::Params (reference PathTracer.h:21-32).  Fields after `ambient` are extensions the
 * reference lacks (SURVEY.md F10/F11/H4); zero means "reference behaviour". */
typedef struct SailorPtParams {
	const char* pathToModel;      /* m_pathToModel */
	const char* output;           /* m_output (PNG); NULL/"" = do not write a file */
	const char* camera;           /* m_camera; NULL/"" = first camera */
	uint32_t height;              /* m_height */
	uint32_t numSamples;          /* m_numSamples        (S: importance samples at the first hit; <= 65535, else SAILOR_PT_ERR_LIMIT) */
	uint32_t numAmbientSamples;   /* m_numAmbientSamples (A: hemisphere samples at the first hit; <= 65535) */
	uint32_t maxBounces;          /* m_maxBounces (<= 64) */
	uint32_t msaa;                /* m_msaa (primary samples per pixel) */
	float ambient[3];             /* m_ambient */
	/* extensions */
	uint32_t widthOverride;       /* 0: width = uint(height * aspect) (PathTracer.cpp:137-142) */
	uint64_t seed;                /* RNG stream key; the reference uses unseeded rand() */
	uint32_t rowBegin, rowEnd;    /* render only image rows [rowBegin,rowEnd) of the task grid (multi-GPU shard); 0,0 = all */
	uint32_t msaaBegin, msaaEnd;  /* render only primary-sample indices [msaaBegin,msaaEnd); 0,0 = all */
	int32_t deviceCount;          /* SailorPt_Run / SailorPt_Render / SailorPt_RenderResident: CUDA devices to spread the frame over (SURVEY.md 8b), starting at the
	                                 scene's own device; clamped to the devices of the box; 0 or 1 = the scene's device only.  Row bands are handed out
	                                 dynamically, the frame is bit-identical to the single-device one (replaces the tile loop of PathTracer.cpp:418-487) */
	uint32_t flags;               /* SAILOR_PT_FLAG_*; 0 = default */
} SailorPtParams;

/* SailorPtParams::flags */
#define SAILOR_PT_FLAG_EXACT_TRAVERSAL 1u  /* trace every ray with the reference-visit-order kernel; default: secondary rays take the origin-local walk of the same tree and ambiguous ones are replayed exactly */
#define SAILOR_PT_FLAG_WIDE_TRAVERSAL 2u   /* secondary rays walk the 8-wide quantised layout instead (same results; built on demand) */

typedef struct SailorPtScene SailorPtScene; /* opaque */

/* One flattened triangle in the reference's Math::Triangle field order (reference Math/Bounds.h:12-25):
 * centroid(3) vertices(9) normals(9) tangent(9) bitangent(9) uvs(6) uvs2(6) = 51 floats, + material index. */
#define SAILOR_PT_TRI_FLOATS 51

/* The reference's BVH node (reference Raytracing/BVH.h:13-24), 32 bytes. */
typedef struct SailorPtBvhNode {
	float aabbMin[3];
	uint32_t leftFirst;
	float aabbMax[3];
	uint32_t triCount;
} SailorPtBvhNode;

/* One closest-hit result (the fields of Math::RaycastHit the integrator consumes, Bounds.h:59-71). */
typedef struct SailorPtHit {
	float t;          /* m_rayLenght; +inf when no hit */
	float baryU;      /* m_barycentricCoordinate.y */
	float baryV;      /* m_barycentricCoordinate.z */
	uint32_t triId;   /* m_triangleIndex (original, pre-BVH order); 0xFFFFFFFF when no hit */
} SailorPtHit;

typedef struct SailorPtStats {
	uint64_t rays;            /* closest-hit queries (BVH::IntersectBVH calls) of the last call */
	uint64_t primarySamples;  /* Raytrace() evaluations at depth 0 of the last call */
	uint64_t boxTests;        /* oracle (counting build) only: IntersectRayAABB calls */
	uint64_t triTests;        /* oracle (counting build) only: IntersectRayTriangle calls */
	double secondsTotal;      /* wall time of the last call (host clock) */
	double secondsFlatten;    /* SceneLoad: flatten kernel */
	double secondsBvhBuild;
	double secondsTraverse;   /* product: sum of traversal-kernel launches (CUDA events on the launch stream) */
	double secondsShade;
	double secondsOutput;
	uint32_t traverseLaunches;
	uint32_t kernelLaunches;  /* product: all kernel launches of the last call */
	uint32_t threads;         /* oracle: worker threads used */
	uint32_t batches;         /* product, render calls: batches of first hits the wavefront processed (one non-empty fan-out pass pair each) */
	uint64_t h2dBytes;        /* product: bytes copied host->device by the last call */
	uint64_t d2hBytes;        /* product: bytes copied device->host by the last call */
	/* product, render calls: device time per wavefront stage (CUDA events on the launch stream); secondsShade is their sum + the rest */
	double secondsExpand;     /* ExpandKernel: shade an activation, emit its few rays */
	double secondsFanOut;     /* FanOutKernel: hemisphere + importance samples of first hits */
	double secondsClassify;   /* ClassifyKernel + TraceSky continuation kernels */
	double secondsGather;     /* GatherKernel + resolve */
	uint64_t fanOutSamples;   /* rays emitted by FanOutKernel */
	double secondsCall;       /* product, RenderResident: the whole call between two CUDA events on the launch stream (BVH build + render + output stage) */
	uint64_t replayedRays;    /* product: rays of the last call that the fast secondary-ray walk handed to the exact (reference visit order) kernel */
	uint32_t devicesUsed;     /* product, render calls: CUDA devices the frame was spread over (SailorPtParams::deviceCount, clamped to what the box has) */
	uint32_t secondaryTraversal; /* product, render calls: kernel that traced the secondary rays: 1 origin-local walk, 2 exact top-down kernel (picked once per scene by a
	                                timed probe, same results either way), 0 the shared-memory kernel of small scenes / not applicable */
} SailorPtStats;

/* ---- the reference entry points (PathTracer.h:34-36) ---- */

/* PathTracer::ParseCommandLineArgs (PathTracer.cpp:30-73): --in --out --height --samples --bounces --camera
 * --ambient RRGGBB.  Strings stay owned by the library until the next call on the same thread. */
SAILOR_PT_API int32_t SailorPt_ParseCommandLineArgs(SailorPtParams* params, const char** args, int32_t num);

/* PathTracer::Run (PathTracer.cpp:75-575): glTF in, PNG out.  Blocking. */
SAILOR_PT_API int32_t SailorPt_Run(const SailorPtParams* params);

/* ---- staged entry points (the same pipeline, one stage per call; used by parity tests and the bench) ---- */

/* Load + flatten (PathTracer.cpp:84-162, MaterialUtils.cpp:64-198) + materials/textures/lights (:164-381).
 * Also expands EXT_mesh_gpu_instancing (not read by the reference): a node's mesh is drawn once per instance, in the triangle
 * order of the same scene with one child node per instance placed before the node's children.  A malformed instancing object
 * gives SAILOR_PT_ERR_FORMAT; more than 1,431,655,765 flattened triangles give SAILOR_PT_ERR_LIMIT before any device allocation.
 * TRIANGLES, TRIANGLE_STRIP and TRIANGLE_FAN primitives draw (strip and fan corners per glTF 2.0 3.7.2.1); sparse accessors are
 * applied (a malformed sparse block makes its accessor unreadable); quantized streams (KHR_mesh_quantization) are decoded on the
 * device.  A primitive above the triangle limit, or a scene above 1,073,741,823 vertices, gives SAILOR_PT_ERR_LIMIT before anything
 * is sized by that count. */
SAILOR_PT_API int32_t SailorPt_SceneLoad(const char* pathToModel, SailorPtScene** outScene);
SAILOR_PT_API void SailorPt_SceneFree(SailorPtScene* scene);
/* counts[0..5] = triangles, materials, textures, directional lights, cameras, BVH nodes used (0 before build) */
SAILOR_PT_API int32_t SailorPt_SceneCounts(const SailorPtScene* scene, uint32_t counts[6]);
/* triangles: numTriangles*SAILOR_PT_TRI_FLOATS floats; materialIndex: numTriangles bytes (either may be NULL). */
SAILOR_PT_API int32_t SailorPt_SceneGetTriangles(const SailorPtScene* scene, float* triangles, uint8_t* materialIndex);
/* Material import (PathTracer.cpp:164-360 -> Raytracing::Material, MaterialUtils.h:138-177): the fields the live integrator
 * reads, SAILOR_PT_MATERIAL_WORDS 32-bit words per material:
 *   [0..8]  m_uvTransform (glm::mat3, column-major)   [9..12] m_baseColorFactor   [13..15] m_emissiveFactor
 *   [16..18] m_attenuationColor   [19] m_metallicFactor   [20] m_roughnessFactor   [21] m_indexOfRefraction
 *   [22] m_transmissionFactor   [23] m_alphaCutoff   [24] m_thicknessFactor   [25] m_attenuationDistance
 *   then as uint32: [26] m_blendMode (0 opaque, 1 blend, 2 mask), [27] m_baseColorIndex, [28] m_normalIndex,
 *   [29] m_metallicRoughnessIndex, [30] m_emissiveIndex, [31] m_transmissionIndex (255 = no texture, the reference's u8(-1)). */
#define SAILOR_PT_MATERIAL_WORDS 32
SAILOR_PT_API int32_t SailorPt_SceneGetMaterials(const SailorPtScene* scene, uint32_t* words);
/* Directional lights (PathTracer.cpp:362-381 -> DirectionalLight, LightingModel.h:10-14): 6 floats per light,
 * m_direction then m_intensity (= color * intensity / 683). */
SAILOR_PT_API int32_t SailorPt_SceneGetLights(const SailorPtScene* scene, float* directionAndIntensity);

/* BVH::BuildBVH (BVH.cpp:280-338).  Idempotent. */
SAILOR_PT_API int32_t SailorPt_BuildBVH(SailorPtScene* scene);
/* nodes: 2N-1 reference-layout nodes (only counts[5] are meaningful); triIdxMapping: N entries (reordered->original). */
SAILOR_PT_API int32_t SailorPt_GetBVH(const SailorPtScene* scene, SailorPtBvhNode* nodes, uint32_t* triIdxMapping);

/* Camera + image size for params (PathTracer.cpp:102-153,390-403).
 * cam[0..2]=position, [3..5]=pixel00Dir, [6..8]=pixelDeltaU, [9..11]=pixelDeltaV. */
SAILOR_PT_API int32_t SailorPt_GetCamera(const SailorPtScene* scene, const SailorPtParams* params,
	uint32_t* width, uint32_t* height, float cam[12]);

/* BVH::IntersectBVH (BVH.cpp:122-191) for `count` rays: origin/dir 3 floats each, ignoreTri may be NULL. */
SAILOR_PT_API int32_t SailorPt_IntersectRays(SailorPtScene* scene, uint32_t count, const float* origins,
	const float* directions, const uint32_t* ignoreTri, SailorPtHit* hits);

/* The same query through the traversal variants the integrator uses for secondary rays.  flags: SAILOR_PT_RAYS_LOCAL = the
 * origin-local walk (starts at the leaf of ignoreTri), SAILOR_PT_RAYS_WIDE = the 8-wide quantised layout; both replay ambiguous
 * rays exactly, so the results equal SailorPt_IntersectRays.  SAILOR_PT_RAYS_ANY_HIT = hit-or-miss query: hits[i].triId !=
 * 0xFFFFFFFF iff BVH::IntersectBVH would return true (t, u, v, triId are those of SOME reachable hit, not necessarily the
 * closest).  The oracle ignores LOCAL / WIDE and answers ANY_HIT with its closest hit. */
#define SAILOR_PT_RAYS_WIDE 1u
#define SAILOR_PT_RAYS_ANY_HIT 2u
#define SAILOR_PT_RAYS_LOCAL 4u
SAILOR_PT_API int32_t SailorPt_IntersectRaysEx(SailorPtScene* scene, uint32_t count, const float* origins,
	const float* directions, const uint32_t* ignoreTri, uint32_t flags, SailorPtHit* hits);

/* Primary ray of sample 0 (offset .5,.5; PathTracer.cpp:458-466) for every pixel, in task order
 * (index = y*width + x with y the task row, i.e. before the row flip of :449). */
SAILOR_PT_API int32_t SailorPt_PrimaryHits(SailorPtScene* scene, const SailorPtParams* params, SailorPtHit* hits);

/* Tile loop + Raytrace (PathTracer.cpp:418-487, 622-879): linear accumulator, width*height*3 floats, rows as the
 * reference stores them (flipped, :449).  srgb8 (width*height*3 bytes, may be NULL) = output stage (:535-565). */
SAILOR_PT_API int32_t SailorPt_Render(SailorPtScene* scene, const SailorPtParams* params, float* linearRGB,
	uint8_t* srgb8);

/* Same as SailorPt_Render but the accumulator and the sRGB8 image stay resident with the scene (device memory in the
 * product): no host copies inside the call.  flags bit0: rebuild the BVH first (BuildBVH is part of the timed pass),
 * bit1: also run the output stage.  Used by bench.py for the device-resident number and by the multi-GPU path. */
SAILOR_PT_API int32_t SailorPt_RenderResident(SailorPtScene* scene, const SailorPtParams* params, uint32_t flags);
/* Read the resident results back to host buffers (either may be NULL). */
SAILOR_PT_API int32_t SailorPt_ReadResident(SailorPtScene* scene, float* linearRGB, uint8_t* srgb8);
/* Product only: copy the resident linear accumulator (width*height*3 floats) into a caller-owned DEVICE buffer
 * (e.g. a torch tensor handed to NCCL). */
SAILOR_PT_API int32_t SailorPt_CopyResidentToDevice(SailorPtScene* scene, void* dstDevice, uint64_t bytes);

/* Product only: run the output stage on the resident accumulator; when srcDevice != NULL that DEVICE buffer (width*height*3
 * floats, e.g. the NCCL-reduced frame) first replaces the resident accumulator.  The sRGB8 image stays resident. */
SAILOR_PT_API int32_t SailorPt_OutputStageResident(SailorPtScene* scene, const void* srcDevice, uint64_t bytes);

/* ---- the steps after the path (SURVEY.md section 8f ranks 3 and 4); product only, the oracle returns SAILOR_PT_ERR_UNSUPPORTED ---- */

/* Write a linear float image (width*height*3, rows as SailorPt_Render returns them) in the format the extension names:
 * .pfm (Portable Float Map: the accumulator's exact bits), .hdr (Radiance RGBE), anything else = the reference's own output,
 * i.e. output stage + sRGB8 PNG (PathTracer.cpp:535-565).  SailorPt_Run picks the format of params->output the same way. */
SAILOR_PT_API int32_t SailorPt_WriteImage(const char* path, uint32_t width, uint32_t height, const float* linearRGB);

/* Image difference report: metrics[0] mean relative error = mean|a-b| / mean|b| (the tolerance metric of the converged-image
 * tests), [1] RMSE, [2] max |a-b|, [3] PSNR in dB against peak 1.0 (1e30 when identical). */
SAILOR_PT_API int32_t SailorPt_CompareImages(uint32_t width, uint32_t height, const float* a, const float* b, double metrics[4]);

/* Progressive render with checkpoint / resume.  The primary samples [0, params->msaa) of the frame (PathTracer.cpp:457-469,
 * one Raytrace per pixel and sample, accumulator / msaa) are rendered in passes of `msaaPerPass` sample indices; the
 * un-normalised sum stays on the device and every pass continues the same chain of additions, so the finished frame has
 * the SAME BITS as SailorPt_Render.  maxPasses: stop after that many passes (0 = run to the end).  checkpointPath (may be
 * NULL): the running sum + the parameters it depends on, written when the call returns (and after every pass with flag 2).
 * flags: 1 = resume from checkpointPath when it exists (it must match scene, camera and parameters), 2 = checkpoint after
 * every pass, 4 = also write params->output after every pass (preview).  linearRGB / srgb8 (either may be NULL) receive
 * the estimate so far, normalised by the samples done; *msaaDone (may be NULL) the number of sample indices accumulated.
 * When the frame is complete and params->output is set, the image file is written as SailorPt_Run would. */
SAILOR_PT_API int32_t SailorPt_RenderProgressive(SailorPtScene* scene, const SailorPtParams* params, uint32_t msaaPerPass,
	uint32_t maxPasses, const char* checkpointPath, uint32_t flags, float* linearRGB, uint8_t* srgb8, uint32_t* msaaDone);

/* Product: page-lock a caller-owned HOST buffer (the result images a host reuses frame after frame) so that SailorPt_Render /
 * SailorPt_ReadResident DMA straight into it instead of staging through the library's own pinned chunks and a host memcpy.
 * The buffer must be unpinned before it is freed.  Results are identical either way.  The reference has no counterpart (its
 * image lives in host memory, PathTracer.cpp:449-469); the oracle accepts and ignores both calls. */
SAILOR_PT_API int32_t SailorPt_PinHostBuffer(void* hostBuffer, uint64_t bytes);
SAILOR_PT_API int32_t SailorPt_UnpinHostBuffer(void* hostBuffer);

/* Product: release the working memory the library keeps between frames (the wavefront arenas shared by every scene of the
 * process on the current device, up to 40 GiB, and the cached blocks of the stream-ordered pool).  Scenes stay valid; the next
 * frame allocates its working set again.  The oracle has nothing to release and returns SAILOR_PT_OK. */
SAILOR_PT_API int32_t SailorPt_TrimMemory(void);

/* Output stage alone (PathTracer.cpp:535-565 + Core/Utils.cpp:48-57). */
SAILOR_PT_API int32_t SailorPt_OutputStage(uint32_t width, uint32_t height, const float* linearRGB, uint8_t* srgb8);

/* CombinedSampler2D::Sample (MaterialUtils.h:75-124) on texture `textureIndex`: uv 2 floats per sample, out 4
 * floats per sample (vec3 textures leave .w = 0). */
SAILOR_PT_API int32_t SailorPt_SampleTexture(SailorPtScene* scene, uint32_t textureIndex, uint32_t count,
	const float* uv, float* out);

/* LightingModel function table (LightingModel.cpp:28-386) on `count` inputs; see tests/test_lighting.py for the
 * record layout (in: 24 floats, out: 28 floats). */
SAILOR_PT_API int32_t SailorPt_EvalLighting(uint32_t count, const float* in, float* out);

/* The image decoder of the glTF front end on a file held in memory: RGBA8, row 0 = top, i.e. what the reference's texture loader gets from
 * stbi_load_from_memory(..., STBI_rgb_alpha) (MaterialUtils.h:226-249).  PNG (all colour types and bit depths, interlaced too) and JPEG
 * (baseline and progressive, any subsampling, grey / YCbCr / RGB / CMYK / YCCK) decode byte-identically to stb_image; other formats return
 * SAILOR_PT_ERR_UNSUPPORTED.  rgba8 may be NULL to query the size; capacity is the size of rgba8 in bytes. */
SAILOR_PT_API int32_t SailorPt_DecodeImage(const uint8_t* data, uint64_t size, uint32_t* width, uint32_t* height, uint8_t* rgba8, uint64_t capacity);

/* The shading context the integrator builds at a hit, value for value (parity hook for rows a13/a15 of SURVEY.md 8):
 * PathTracer::Raytrace lines 636-661 (interpolated frame, face normal turned against the ray, uv through the material's
 * uvTransform, world normal, alpha-scaled sample counts) around PathTracer::GetMaterialData (PathTracer.cpp:881-927).
 * in:  triIds[count] (original triangle ids), baryUV[2*count] (SailorPtHit::baryU, baryV), rayDirs[3*count]
 * out: SAILOR_PT_SHADE_FLOATS per hit: baseColor(4) orm(3) emissive(3) sampled normal(3) transmission ior thickness opaque(0/1)
 *      worldNormal(3) faceNormal(3) uvTransformed(2) oppositeRay(0/1) numSamples numAmbientSamples (after the alpha rule, as floats) */
#define SAILOR_PT_SHADE_FLOATS 28
SAILOR_PT_API int32_t SailorPt_ShadeHits(SailorPtScene* scene, uint32_t count, const uint32_t* triIds, const float* baryUV, const float* rayDirs,
	uint32_t numSamples, uint32_t numAmbientSamples, float* out);

/* The product's counter-based sample generators (product only; the reference draws from unseeded rand(), SURVEY.md H4), for
 * distribution tests against glm::linearRand on rand() % 255 bytes (glm/gtc/random.inl:19-27,176-183) and the blue-noise table walk
 * (PathTracer.cpp:934-1077).  kind 0: `count` raw 32-bit draws (out = uint32 bit patterns); kind 1: `count` linearRand(0,1) floats;
 * kind 2: `count` draws of one NextVec2_BlueNoise walk, 4 floats each: x, y, table index of x, table index of y. */
SAILOR_PT_API int32_t SailorPt_SampleGenerators(uint64_t streamKey, uint32_t kind, uint32_t count, float* out);

SAILOR_PT_API int32_t SailorPt_GetStats(SailorPtStats* stats);
SAILOR_PT_API const char* SailorPt_LastError(void);
/* Product: make CUDA device `device` current for the calling thread (one process per GPU sets its LOCAL_RANK before
 * loading a scene; scenes stay on the device they were created on).  Oracle: accepts 0 only. */
SAILOR_PT_API int32_t SailorPt_SetDevice(int32_t device);
/* "cuda sm_100a" for the product, "reference-cpu" for the oracle. */
SAILOR_PT_API const char* SailorPt_Backend(void);

#ifdef __cplusplus
}
#endif
#endif
