// flatten.cuh — scene flattening on the device: glTF primitives -> SoA triangle buffers (SURVEY §8 row a10).
//
// One thread per output triangle.  Restates, operation for operation, what the reference's (commented-out)
// ProcessMesh_Assimp does per face (reference MaterialUtils.cpp:64-163): world-transform of positions (divide by
// w), normals / tangents / bitangents as vec4(v,0)*M without renormalisation, centroid = sum * 0.333f, per-face
// tangent generation (MaterialUtils.cpp:33-62) when the primitive has no TANGENT stream.  `vec4 * mat4` follows
// glm's order m[j][0]*v0 + m[j][1]*v1 + m[j][2]*v2 + m[j][3]*v3 (glm/detail/type_mat4x4.inl:586-595).
//
// Input: the vertex streams of each source primitive once (SourceDesc), and the draws in triangle order (DrawDesc: source,
// world matrix, material; drawStart: first output triangle of each draw).  A mesh placed by many nodes or instanced by
// EXT_mesh_gpu_instancing is many draws of one source.  Output triangle t belongs to the last draw whose drawStart <= t.
// FlattenBlockKernel finds that draw once for the first triangle of every kFlattenSpan, so a thread searches only the draws
// its own span touches: none for a few large draws, a handful when 10^5 draws of small meshes share the scene.
//
// HBM layout produced (all 16-byte aligned for LDG.128):
//   vtx      float4[3N]  (v0|v1|v2).xyz per triangle           -> BVH build input, 48 B / triangle
//   centroid float4[N]   centroid.xyz, w = material index bits -> BVH build input, 16 B / triangle
//   shade    float4[9N]  n0,uv0.x | n1,uv0.y | n2,uv1.x | t0,uv1.y | t1,uv2.x | t2,uv2.y | b0,mat | b1,0 | b2,0
//                                                               -> shading stage, 144 B / shaded hit
//   uv2      float2[3N]  second UV set (only read back by SailorPt_SceneGetTriangles; the integrator never uses it)
#pragma once
#include "backend.h"

namespace spt
{
	struct SourceDesc
	{
		uint32_t vtxOffset;    // into pos (x3), nrm (x3), uv0/uv1 (x2), tan (x4): element = vertex
		uint32_t idxOffset;    // into idx
		uint32_t hasNrm, hasUv0, hasUv1, hasTan;
		uint32_t pad[2];
	};

	struct DrawDesc
	{
		float world[16];
		uint32_t source;       // into the SourceDesc table
		uint32_t material;
		uint32_t pad[2];
	};

	constexpr uint32_t kFlattenSpan = 256;     // output triangles per entry of the block table (= threads per launch_for block)

	// last draw d in [lo, hi) with drawStart[d] <= t (drawStart[lo] <= t)
	SPT_HD uint32_t FindDraw(const uint32_t* drawStart, uint32_t lo, uint32_t hi, uint32_t t)
	{
		while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (drawStart[mid] <= t) lo = mid; else hi = mid; }
		return lo;
	}

	// blockDraw[b] = the draw of output triangle min(b * kFlattenSpan, numTris - 1), for b in [0, ceil(numTris / kFlattenSpan)]
	struct FlattenBlockKernel
	{
		const uint32_t* drawStart; uint32_t numDraws, numTris; uint32_t* blockDraw;
		SPT_KERNEL_BODY void operator()(uint32_t b) const
		{
			const uint32_t t = b < (numTris - 1u) / kFlattenSpan + 1u ? b * kFlattenSpan : numTris - 1u;
			blockDraw[b] = FindDraw(drawStart, 0u, numDraws, t);
		}
	};

	// ---- stored streams -> the float streams and u32 triples FlattenKernel reads (before it, in the same stream) ----
	// Sources whose streams are not float32 of FlattenKernel's width, and whose indices are not a u32 TRIANGLES list, are uploaded
	// as the file stores them (each piece starting at a multiple of 4 bytes) and expanded here: one launch per stream kind across
	// all such sources, each thread finding its source in a prefix table (FindDraw) as FlattenKernel finds its draw.

	struct StreamDecodeDesc
	{
		uint64_t srcByte;      // into the staged bytes of this stream kind
		uint32_t dstVertex;    // SourceDesc::vtxOffset
		uint32_t componentType, comps, normalized;
		uint32_t pad[2];
	};

	// vertex i of the decoded sources of one stream kind -> `width` floats; components beyond the stored ones read 0
	struct DecodeStreamKernel
	{
		const uint32_t* start; const StreamDecodeDesc* desc; uint32_t numDesc, width; const uint8_t* src; float* dst;
		SPT_KERNEL_BODY void operator()(uint32_t i) const
		{
			const uint32_t j = FindDraw(start, 0u, numDesc, i);
			const StreamDecodeDesc& D = desc[j];
			const uint32_t v = i - start[j];
			const uint32_t elemBytes = D.comps * (D.componentType == 5126 || D.componentType == 5125 ? 4u : (D.componentType == 5122 || D.componentType == 5123 ? 2u : 1u));
			const uint8_t* e = src + D.srcByte + (size_t)v * elemBytes;
			float* o = dst + ((size_t)D.dstVertex + v) * width;
			for (uint32_t c = 0; c < width; c++) o[c] = c < D.comps ? DecodeComponent(e, D.componentType, D.normalized != 0, c) : 0.0f;
		}
	};

	struct IndexAssemblyDesc
	{
		uint64_t srcByte;      // into the staged index bytes (unused when idxType is 0)
		uint32_t dstIndex;     // SourceDesc::idxOffset
		uint32_t idxType;      // 0: not indexed, corner k is vertex k
		uint32_t mode;         // 4 TRIANGLES, 5 TRIANGLE_STRIP, 6 TRIANGLE_FAN
		uint32_t numVerts;     // an index at or above it reads vertex 0
		uint32_t pad[2];
	};

	// face f of the assembled sources -> its three vertex indices, corners as glTF 2.0 §3.7.2.1 orders them:
	// list (3f, 3f+1, 3f+2), strip (f, f+1+f%2, f+2-f%2), fan (f+1, f+2, 0)
	struct AssembleIndexKernel
	{
		const uint32_t* start; const IndexAssemblyDesc* desc; uint32_t numDesc; const uint8_t* src; uint32_t* idx;
		SPT_KERNEL_BODY void operator()(uint32_t t) const
		{
			const uint32_t j = FindDraw(start, 0u, numDesc, t);
			const IndexAssemblyDesc& D = desc[j];
			const uint32_t f = t - start[j];
			uint32_t corner[3];
			if (D.mode == 5) { corner[0] = f; corner[1] = f + 1u + (f & 1u); corner[2] = f + 2u - (f & 1u); }
			else if (D.mode == 6) { corner[0] = f + 1u; corner[1] = f + 2u; corner[2] = 0u; }
			else { corner[0] = f * 3u; corner[1] = f * 3u + 1u; corner[2] = f * 3u + 2u; }
			const uint8_t* s = src + D.srcByte;
			for (int k = 0; k < 3; k++)
			{
				const uint32_t v = D.idxType ? IndexAt(s, D.idxType, corner[k]) : corner[k];
				idx[(size_t)D.dstIndex + (size_t)f * 3 + k] = v < D.numVerts ? v : 0u;
			}
		}
	};

	SPT_HD V3 RowMul3(const float* M, V3 v, float w)
	{
		return v3(M[0] * v.x + M[1] * v.y + M[2] * v.z + M[3] * w,
			M[4] * v.x + M[5] * v.y + M[6] * v.z + M[7] * w,
			M[8] * v.x + M[9] * v.y + M[10] * v.z + M[11] * w);
	}
	SPT_HD float RowMulW(const float* M, V3 v, float w) { return M[12] * v.x + M[13] * v.y + M[14] * v.z + M[15] * w; }

	struct FlattenKernel
	{
		const DrawDesc* draws; const uint32_t* drawStart; const uint32_t* blockDraw; const SourceDesc* sources;
		const float* pos; const float* nrm; const float* uv0; const float* uv1; const float* tan; const uint32_t* idx;
		V4* vtx; V4* centroid; V4* shade; V2* uv2;

		SPT_KERNEL_BODY void operator()(uint32_t t) const
		{
			const uint32_t b = t / kFlattenSpan;
			const uint32_t d = FindDraw(drawStart, blockDraw[b], blockDraw[b + 1] + 1u, t);
			const DrawDesc& D = draws[d];
			const SourceDesc& P = sources[D.source];
			const uint32_t f = t - drawStart[d];
			const float* M = D.world;
			uint32_t vi[3];
			V3 lp[3], ln[3], wv[3], wn[3], wt[3], wb[3];
			V2 uvA[3], uvB[3];
			for (int k = 0; k < 3; k++)
			{
				vi[k] = idx[P.idxOffset + f * 3 + k] + P.vtxOffset;
				lp[k] = v3(pos[vi[k] * 3], pos[vi[k] * 3 + 1], pos[vi[k] * 3 + 2]);
			}
			if (P.hasNrm) { for (int k = 0; k < 3; k++) ln[k] = v3(nrm[vi[k] * 3], nrm[vi[k] * 3 + 1], nrm[vi[k] * 3 + 2]); }
			else { const V3 fn = normalize(cross(lp[1] - lp[0], lp[2] - lp[0])); ln[0] = ln[1] = ln[2] = fn; }
			for (int k = 0; k < 3; k++)
			{
				wn[k] = RowMul3(M, ln[k], 0.0f);
				const V3 xyz = RowMul3(M, lp[k], 1.0f);
				const float w = RowMulW(M, lp[k], 1.0f);
				wv[k] = xyz / w;
				uvA[k] = P.hasUv0 ? v2(uv0[vi[k] * 2], uv0[vi[k] * 2 + 1]) : v2(0.0f, 0.0f);
				uvB[k] = P.hasUv1 ? v2(uv1[vi[k] * 2], uv1[vi[k] * 2 + 1]) : v2(0.0f, 0.0f);
			}
			const V3 c = (wv[0] + wv[1] + wv[2]) * 0.333f;
			if (P.hasTan)
			{
				for (int k = 0; k < 3; k++)
				{
					const V3 tg = v3(tan[vi[k] * 4], tan[vi[k] * 4 + 1], tan[vi[k] * 4 + 2]);
					const float w = tan[vi[k] * 4 + 3];
					const V3 bt = cross(ln[k], tg) * w;
					wt[k] = RowMul3(M, tg, 0.0f);
					wb[k] = RowMul3(M, bt, 0.0f);
				}
			}
			else
			{
				// GenerateTangentBitangent (MaterialUtils.cpp:33-62) on the WORLD-space vertices
				V3 tg = v3(0.0f), bt = v3(0.0f);
				const V3 e1 = wv[1] - wv[0], e2 = wv[2] - wv[0];
				const V2 d1 = uvA[1] - uvA[0], d2 = uvA[2] - uvA[0];
				const float den = d1.x * d2.y - d2.x * d1.y;
				if (!(fabsf(den) < 1e-6f))
				{
					const float fI = 1.0f / den;
					tg = v3(fI * (d2.y * e1.x - d1.y * e2.x), fI * (d2.y * e1.y - d1.y * e2.y), fI * (d2.y * e1.z - d1.y * e2.z));
					const V3 nn = cross(e1, e2);
					bt = normalize(cross(nn, tg));
					tg = normalize(tg);
				}
				wt[0] = wt[1] = wt[2] = tg;
				wb[0] = wb[1] = wb[2] = bt;
			}
			for (int k = 0; k < 3; k++) vtx[t * 3 + k] = v4(wv[k].x, wv[k].y, wv[k].z, 0.0f);
			centroid[t] = v4(c.x, c.y, c.z, u2f(D.material));
			V4* s = shade + (size_t)t * 9;
			s[0] = v4(wn[0].x, wn[0].y, wn[0].z, uvA[0].x);
			s[1] = v4(wn[1].x, wn[1].y, wn[1].z, uvA[0].y);
			s[2] = v4(wn[2].x, wn[2].y, wn[2].z, uvA[1].x);
			s[3] = v4(wt[0].x, wt[0].y, wt[0].z, uvA[1].y);
			s[4] = v4(wt[1].x, wt[1].y, wt[1].z, uvA[2].x);
			s[5] = v4(wt[2].x, wt[2].y, wt[2].z, uvA[2].y);
			s[6] = v4(wb[0].x, wb[0].y, wb[0].z, u2f(D.material));
			s[7] = v4(wb[1].x, wb[1].y, wb[1].z, 0.0f);
			s[8] = v4(wb[2].x, wb[2].y, wb[2].z, 0.0f);
			for (int k = 0; k < 3; k++) uv2[t * 3 + k] = uvB[k];
		}
	};
}
