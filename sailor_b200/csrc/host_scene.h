// host_scene.h — what the glTF front end hands to the device pipeline (host memory, product code).
//
// This is the input side of the hot path (SURVEY §8 rows a10/a11/a12/a14): raw vertex streams, once per source primitive,
// and a draw table of (source, world matrix, material) (flattened on the DEVICE by flatten.cuh), material factors, RGBA8
// texels (converted to float texels on the device), cameras and directional lights.  Loader contract: DESIGN.md "loader contract".
#pragma once
#include <stdint.h>
#include <string>
#include <vector>

namespace spt
{
	enum BlendMode : uint32_t { kOpaque = 0, kBlend = 1, kMask = 2 };          // reference MaterialUtils.h:131-136
	enum Clamping : uint32_t { kClamp = 0, kRepeat = 1 };                       // reference MaterialUtils.h:17-21
	constexpr uint32_t kNoTexture = 255;                                        // reference u8(-1), MaterialUtils.h:157-174

	// reference Material (MaterialUtils.h:138-177), the fields the live integrator reads. 36 words, 16-byte aligned.
	struct alignas(16) MaterialGpu
	{
		float uvTransform[12];   // glm::mat3 columns, each padded to 4 floats
		float baseColor[4];
		float emissive[3]; float metallic;
		float attenuationColor[3]; float roughness;
		float ior, transmission, alphaCutoff, thickness;
		float attenuationDistance; uint32_t blendMode; uint32_t texBase, texNormal;
		uint32_t texMetallicRoughness, texEmissive, texTransmission, pad;
	};
	static_assert(sizeof(MaterialGpu) == 144, "MaterialGpu layout");

	// One vertex stream as the file stores it (sparse substitution applied): one element per vertex of `comps` components of
	// `componentType`, tightly packed.  The device decodes it (DecodeComponent, hd.h) unless it already is the float32 stream
	// FlattenKernel reads.
	struct HostStream
	{
		std::vector<uint8_t> bytes;     // empty: the primitive has no such stream
		uint32_t componentType = 0, comps = 0;
		bool normalized = false;
		bool empty() const { return bytes.empty(); }
		bool IsFloat(uint32_t width) const { return componentType == 5126 && comps == width; }
	};

	// The streams of one glTF primitive, read once per document: every node that reaches a primitive with the same accessors
	// and mode, and every instance of EXT_mesh_gpu_instancing, draws these streams again without copying them.
	struct HostSource
	{
		uint64_t numVerts = 0;
		HostStream pos;             // decoded to 3 floats per vertex
		HostStream nrm;             // 3 or empty (-> flat face normals, aiProcess_GenNormals)
		HostStream uv0, uv1;        // 2 or empty
		HostStream tan;             // 4 (a VEC4 accessor) or empty
		uint32_t mode = 4;          // 4 TRIANGLES, 5 TRIANGLE_STRIP, 6 TRIANGLE_FAN
		uint32_t idxType = 0;       // component type of `idx`; 0: not indexed (the vertices in order)
		std::vector<uint8_t> idx;   // the index accessor's first components as stored, tightly packed; a u32 TRIANGLES list is clamped
		uint64_t faces = 0;         // TRIANGLES n / 3, strip and fan max(n - 2, 0); n = index count, or numVerts without indices
		// u32 triples that go to the device as they are (every other index form is assembled there by AssembleIndexKernel)
		bool DirectIdx() const { return mode == 4 && idxType == 5125; }
		bool FloatStreams() const
		{
			return pos.IsFloat(3) && (nrm.empty() || nrm.IsFloat(3)) && (uv0.empty() || uv0.IsFloat(2)) && (uv1.empty() || uv1.IsFloat(2)) && (tan.empty() || tan.IsFloat(4));
		}
	};

	// One placement of a source in the flattened scene.  Draws are in the scene's triangle order: the flattened triangles are
	// the triangles of each draw's source, draw after draw.
	struct HostDraw
	{
		uint32_t source = 0;        // into HostScene::sources
		uint32_t material = 0;      // already truncated to u8 like Triangle::m_materialIndex (Bounds.h:21)
		float world[16];            // reference convention: memory = row-major world matrix (glm m[c][r] = world[c*4+r])
	};

	// Most flattened triangles a scene may have.  The device pipeline indexes triangles with 32-bit integers, and the largest
	// product it forms from a triangle index is t * 3 + 2 (vertex slots of flatten, BVH build and every traversal layout);
	// node indices stay below 2 N and leaf references below 2^31 (traverse.cuh kLeafBit).  floor((2^32 - 1) / 3) keeps all of
	// them exact.  Device memory runs out long before this (about 232 B per flattened triangle plus the BVH).
	constexpr uint64_t kMaxTriangles = 0xFFFFFFFFull / 3u;
	// Most vertices all sources of a scene may have together: FlattenKernel forms vertex * 4 (tangents) in 32 bits.
	constexpr uint64_t kMaxVertices = 0xFFFFFFFFull / 4u;

	struct HostTexture
	{
		int32_t width = 0, height = 0;
		uint32_t channels = 3;      // 3 or 4 (CombinedSampler2D::m_channels)
		uint32_t clamping = kRepeat;
		bool srgb = false;          // bConvertToLinear
		bool normalMap = false;     // bNormalMap
		std::vector<uint8_t> rgba;  // width*height*4, stbi RGBA8 convention (row 0 = top)
		std::vector<float> rgbaF;   // Radiance .hdr images only: width*height*4 floats as stbi_loadf(..., STBI_rgb_alpha) returns them (rgba stays empty)
	};

	struct HostCamera
	{
		std::string name;
		float matrix[16];           // reference convention (see HostDraw::world)
		float aspect = 0.0f;
		float hFov = 0.0f;
	};

	struct HostLight { float direction[3]; float intensity[3]; };

	struct HostScene
	{
		std::vector<HostSource> sources;
		std::vector<HostDraw> draws;
		std::vector<MaterialGpu> materials;
		std::vector<HostTexture> textures;
		std::vector<HostCamera> cameras;
		std::vector<HostLight> lights;
		uint64_t numTriangles = 0;  // flattened (all draws), at most kMaxTriangles
		// which kernel traces this scene's secondary rays fastest (0 unknown; render.cuh decides it with a timed probe on the first frame): kept with the
		// parsed file so that reloads served by the scene cache and the per-device replicas of a multi-device render do not probe again
		mutable uint32_t traversalChoice = 0;
	};

	// returns SAILOR_PT_OK or a negative SAILOR_PT_ERR_*; err receives a message
	int LoadGltf(const char* path, HostScene& out, std::string& err);

	// PNG codec (png_codec.cpp).  Decode follows stb_image's conventions (RGBA8, 16-bit -> high byte, low bit depths
	// scaled, palette/tRNS expanded) because the reference decodes with stbi_load(..., STBI_rgb_alpha) (MaterialUtils.h:226-249).
	int DecodePngRgba8(const uint8_t* data, size_t size, int32_t& w, int32_t& h, std::vector<uint8_t>& rgba, std::string& err);
	// JPEG codec (jpeg_codec.cpp): baseline + progressive, byte-identical to stb_image's decoder
	bool IsJpeg(const uint8_t* data, size_t size);
	int DecodeJpegRgba8(const uint8_t* data, size_t size, int32_t& w, int32_t& h, std::vector<uint8_t>& rgba, std::string& err);
	// Radiance RGBE (.hdr) -> RGBA32F exactly as stbi_loadf_from_memory(..., STBI_rgb_alpha) (MaterialUtils.h:226-229)
	bool IsHdr(const uint8_t* data, size_t size);
	int DecodeHdrRgba32F(const uint8_t* data, size_t size, int32_t& w, int32_t& h, std::vector<float>& rgba, std::string& err);
	// any supported image file in memory -> RGBA8 (stbi_load_from_memory(..., STBI_rgb_alpha) convention)
	int DecodeImageRgba8(const uint8_t* data, size_t size, int32_t& w, int32_t& h, std::vector<uint8_t>& rgba, std::string& err);
	int EncodePngRgb8(const char* path, uint32_t w, uint32_t h, const uint8_t* rgb, std::string& err);

	// linear image dumps, comparison, progressive-render checkpoints (image_io.cpp)
	enum class ImageFormat { Png, Pfm, Hdr };
	ImageFormat ImageFormatOf(const char* path);                 // by extension; anything else is PNG (the reference's only format)
	int WritePfm(const char* path, uint32_t w, uint32_t h, const float* rgb, std::string& err);
	int WriteHdr(const char* path, uint32_t w, uint32_t h, const float* rgb, std::string& err);
	void CompareImages(size_t count, const float* a, const float* b, double out[4]);
	struct CheckpointHeader       // everything the running sum depends on; a resume must match all of it
	{
		uint32_t version, width, height, rowBegin, rowEnd, msaaTotal, msaaDone, numSamples, numAmbientSamples, maxBounces, numTriangles, pad;
		uint64_t seed; float ambient[3]; float camera[12]; uint32_t pad2;
	};
	int WriteCheckpoint(const char* path, const CheckpointHeader& hd, const float* runningSum, std::string& err);
	int ReadCheckpoint(const char* path, CheckpointHeader& hd, std::vector<float>& runningSum, std::string& err);

	struct CameraSetup { uint32_t width, height; float pos[3], pixel00Dir[3], deltaU[3], deltaV[3]; };
	struct SailorPtParamsView { const char* camera; uint32_t height; uint32_t widthOverride; };
	// PathTracer.cpp:102-153 + 390-403 (host, glibc tan/atan like the reference)
	CameraSetup SetupCamera(const HostScene& scene, const SailorPtParamsView& p);
}
