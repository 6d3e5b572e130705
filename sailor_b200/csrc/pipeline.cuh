// pipeline.cuh — the device-resident scene and the stage drivers behind the C-ABI (product).
//
// Stages (SURVEY §8): upload + flatten (a10) -> BVH build (a6) -> traversal layout pack -> trace (a7-a9) ->
// integrator (a15/a16, integrator.cuh) -> output stage (a18, output.cuh).  Everything after the glTF parse runs on
// the device; host code only sequences launches and reads back the per-level node counts of the BVH build.
#pragma once
#include "backend.h"
#include "host_scene.h"
#include "flatten.cuh"
#include "bvh_build.cuh"
#include "trace_kernels.cuh"
#include "trace_wide.cuh"
#include "bvh_build_small.cuh"
#include "../../include/sailor_pt.h"

#include <chrono>
#include <memory>

namespace spt
{
	inline double HostNow() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

	// offset: into the texel pool (RGBA8 texels); mode: how CombinedSampler2D::Initialize turns a byte into a float (MaterialUtils.h:42-65)
	enum TexelMode : uint32_t { kTexelLinear = 0, kTexelSrgb = 1, kTexelNormal = 2, kTexelFloat = 3 };      // kTexelFloat: offset is into the float4 pool of .hdr images
	struct DeviceTexture { uint32_t width, height, channels, clamping; uint64_t offset; uint32_t mode, pad; };

	struct SceneDevice
	{
		Ctx ctx;
		int device = 0;                       // CUDA device this replica of the scene lives on
		std::shared_ptr<const HostScene> hostPtr;     // the parsed file: shared by the scene cache (capi.cu) and by the per-device replicas of a multi-device render
		const HostScene& Host() const { return *hostPtr; }
		uint32_t numTris = 0;

		// flattened triangles
		DevBuf<V4> vtx, centroid, shade;
		DevBuf<V2> uv2;
		DevBuf<MaterialGpu> materials;
		DevBuf<uint32_t> texels;              // all textures as the file's RGBA8 texels (4 bytes each); converted to float at fetch time (textures.cuh)
		DevBuf<V4> texelsF;                   // .hdr images only: float4 texels, converted on the host with the reference's expressions (Initialize<T, vec4>)
		DevBuf<float> srgbLut;                // 256 floats: Utils::SRGBToLinear(byte / 255) evaluated with the host's powf (bit-identical to the reference's)
		DevBuf<DeviceTexture> textures;
		std::vector<DeviceTexture> hostTextures;
		DevBuf<V4> lights;                    // 2 float4 per light: direction, intensity

		// BVH: reference layout (parity / C-ABI) and traversal layout
		bool built = false;
		uint32_t nodesUsed = 0, numInternal = 0, numLevels = 0;
		DevBuf<SailorPtBvhNode> refNodes;
		DevBuf<uint32_t> mapping;
		DevBuf<TNode> tnodes;
		DevBuf<TTri> ttris;
		uint32_t rootRef = 0;
		// origin-local traversal layout (trace_fast.cuh): built with every BVH the shared-memory kernel does not take
		bool hasFast = false;
		// which kernel traces the secondary rays of this scene: 0 not decided yet, 1 origin-local walk, 2 exact (top-down) kernel.  Decided once per
		// geometry by a timed probe on the first level of the first frame (render.cuh); the results are identical either way.
		uint32_t traceChoice = 0, traceChoiceTris = 0; float probeMs[2] = { 0.0f, 0.0f };
		DevBuf<FNode> fnodes; DevBuf<FNode> fclimb; DevBuf<FTri> ftris; DevBuf<FStart> fstart; DevBuf<FHeader> fheader; DevBuf<uint32_t> nodeUp;
		// wide layout (wide_bvh.cuh): an alternative traversal layout, built on demand (SAILOR_PT_FLAG_WIDE_TRAVERSAL / SAILOR_PT_RAYS_WIDE)
		bool hasWide = false;
		bool wantWide = false;                // the caller renders through the wide layout: BuildBvh builds it (inside its timed region)
		uint32_t numWideNodes = 0, numWideLevels = 0;
		DevBuf<WNode> wnodes; DevBuf<TTri> wtris; DevBuf<V4> wleafBox; DevBuf<WDesc> wdesc; DevBuf<WideCounters> wcounters;
		DevBuf<uint32_t> replayList;          // IntersectRays / sky queues; the wavefront levels use an arena of the frame

		// results of the last RenderResident (stay on the device until read back or handed to NCCL)
		DevBuf<float> residentLin; DevBuf<uint8_t> residentSrgb; uint32_t residentW = 0, residentH = 0;

		SpanTimer traceTimer, stageTimer[4];      // stageTimer: expand, fan-out, classify (+sky), gather
		// BVH build scratch, kept across builds
		DevBuf<uint32_t> buildU32[24];
		DevBuf<float> buildF32[4];

		DevBuf<uint32_t> counter;             // persistent-kernel work counters
		SailorPtStats stats{};

		BvhView View() const { BvhView v; v.nodes = tnodes.p; v.tris = ttris.p; v.rootRef = rootRef; v.numNodes = numInternal; v.numTris = numTris; return v; }
		WideView Wide() const { WideView w; w.nodes = wnodes.p; w.tris = wtris.p; w.leafBox = wleafBox.p; w.numNodes = numWideNodes; return w; }
		FastView Fast() const { FastView w; w.nodes = fnodes.p; w.tris = ftris.p; w.start = fstart.p; w.header = fheader.p; w.climb = fclimb.p; w.numNodes = numInternal; w.numTris = numTris; return w; }
		// [12] wide work counter, [13] replay count, [14] replay work counter, [15] rays replayed since the last reset
		ReplayBuffers Replay(uint32_t* list, uint32_t cap) { ReplayBuffers b; b.counters = counter.p + 12; b.replayList = list; b.replayCap = cap; return b; }

		// true when the frame's secondary rays go to the shared-memory kernel (the exact layout, whole scene on chip), which needs
		// neither the origin-local layout nor the wide one (SAILOR_PT_FORCE_WIDE / SAILOR_PT_FORCE_LOCAL: tests build and use them anyway)
		bool TakesSmallKernel() const
		{
			size_t smallBytes;
			return SmallScene(View(), smallBytes) && !getenv("SAILOR_PT_FORCE_WIDE") && !getenv("SAILOR_PT_FORCE_LOCAL");
		}

		// The origin-local traversal layout.  The arguments are the build scratch of the tree just built.
		int BuildFast(const uint32_t* left, const uint32_t* count, const float* aabb, const uint32_t* rank, const uint32_t* refIdx, const uint32_t* leafOffsetByRef)
		{
			hasFast = false;
			if (TakesSmallKernel() || !numInternal || getenv("SAILOR_PT_NO_FAST")) return SAILOR_PT_OK;
			fnodes.Ensure(ctx, numInternal); fclimb.Ensure(ctx, (size_t)numInternal * 2); ftris.Ensure(ctx, numTris); fstart.Ensure(ctx, numTris); fheader.Ensure(ctx, 1); nodeUp.Ensure(ctx, numInternal);
			if (!ctx.ok) return CudaStatus();
			launch_for(ctx, 1, FastHeaderKernel{ aabb, fheader.p });
			launch_for(ctx, nodesUsed, FastLinkKernel{ left, rank, nodeUp.p });
			launch_for(ctx, nodesUsed, FastPackKernel{ left, count, rank, refIdx, leafOffsetByRef, mapping.p, aabb, vtx.p, nodeUp.p, fheader.p, fnodes.p, ftris.p, fstart.p });
			launch_for(ctx, numInternal, FastClimbKernel{ fnodes.p, nodeUp.p, fclimb.p });
			launch_for(ctx, numTris, FastReachKernel{ fnodes.p, ftris.p, fstart.p, fheader.p, numTris });
			hasFast = ctx.ok;
			return CudaStatus();
		}

		// Collapse the binary tree into the wide layout, on demand (the build scratch of the last BuildBvh is still in place).
		const uint32_t* scratchLeft = nullptr; const uint32_t* scratchCount = nullptr; const float* scratchAabb = nullptr;
		const uint32_t* scratchRefIdx = nullptr; const uint32_t* scratchLeafOffset = nullptr;
		int EnsureWide()
		{
			if (hasWide || !built || !scratchLeft) return SAILOR_PT_OK;
			return BuildWide(scratchLeft, scratchCount, scratchAabb, scratchRefIdx, scratchLeafOffset);
		}
		int BuildWide(const uint32_t* left, const uint32_t* count, const float* aabb, const uint32_t* refIdx, const uint32_t* leafOffsetByRef)
		{
			hasWide = false;
			if (TakesSmallKernel()) return SAILOR_PT_OK;
			const uint32_t N = numTris;
			const uint32_t nodeCap = numInternal + N / kWideLeafMax + 2u;
			wnodes.Ensure(ctx, nodeCap); wtris.Ensure(ctx, N); wleafBox.Ensure(ctx, (size_t)N * 2); wdesc.Ensure(ctx, nodeCap); wcounters.Ensure(ctx, 1);
			if (!ctx.ok) return CudaStatus();
			WideBuildArgs a;
			a.left = left; a.count = count; a.aabb = aabb; a.refIdx = refIdx; a.leafOffsetByRef = leafOffsetByRef; a.ttris = ttris.p;
			a.nodes = wnodes.p; a.wtris = wtris.p; a.leafBox = wleafBox.p; a.desc = wdesc.p; a.c = wcounters.p; a.nodeCap = nodeCap; a.numTris = N;
			launch_for(ctx, 1, WideInitKernel{ a });
			uint32_t levels = 0;
			WideCounters c{};
			for (;;)
			{
				// a wide level consumes at least one binary level: numLevels launches finish every tree without chunked leaves; the
				// counters say whether anything is left
				const uint32_t rounds = levels == 0 ? (numLevels < 6u ? numLevels + 1u : numLevels / 2u + 2u) : 4u;
				for (uint32_t r = 0; r < rounds; r++)
				{
					launch_for_range(ctx, &wcounters.p->lvlBegin, &wcounters.p->lvlEnd, nodeCap, nodeCap, WideLevelKernel{ a });
					launch_for(ctx, 1, WideAdvanceKernel{ wcounters.p, nodeCap });
				}
				levels += rounds;
				DevDownload(ctx, &c, wcounters.p, sizeof(c));
				if (!ctx.ok) return CudaStatus();
				if (c.overflow) { ctx.error = "wide BVH: node arena overflow"; return SAILOR_PT_ERR_LIMIT; }
				if (c.lvlBegin >= c.lvlEnd) break;
				if (levels > 4096u) { ctx.error = "wide BVH: collapse did not terminate"; return SAILOR_PT_ERR_LIMIT; }
			}
			if (c.triCount != N) { ctx.error = "wide BVH: triangle count mismatch"; return SAILOR_PT_ERR_LIMIT; }
			numWideNodes = c.nodeCount; numWideLevels = levels;
			hasWide = true;
			return SAILOR_PT_OK;
		}

		int Fail(int code) { return code; }
		int CudaStatus() { return ctx.ok ? SAILOR_PT_OK : SAILOR_PT_ERR_CUDA; }

		// ---------------------------------------------------------------------------------------------- load
		int Upload()
		{
			const double t0 = HostNow();
			const HostScene& H = Host();
			if (H.numTriangles > kMaxTriangles) { ctx.error = "the scene has more than " + std::to_string(kMaxTriangles) + " triangles"; return SAILOR_PT_ERR_LIMIT; }
			numTris = (uint32_t)H.numTriangles;
			counter.Alloc(ctx, 16); counter.Zero(ctx);
			if (numTris == 0) return CudaStatus();
			// Each source primitive's streams go to the device once, however many draws place it.  A float32 stream of the width
			// FlattenKernel reads and a u32 TRIANGLES list go straight into FlattenKernel's buffers.  Every other stream is uploaded as
			// the file stores it and decoded in place by DecodeStreamKernel; every other index form (u8 / u16 indices of quantized
			// sources, strips, fans, no indices) is turned into u32 triples by AssembleIndexKernel.  A stream a source lacks is never
			// read (FlattenKernel looks at SourceDesc::has*), so its part of the device buffer stays uninitialised.
			constexpr int kKinds = 5;                                     // pos, nrm, uv0, uv1, tan
			const uint32_t width[kKinds] = { 3, 3, 2, 2, 4 };
			auto streamOf = [](const HostSource& hs, int k) -> const HostStream& { return k == 0 ? hs.pos : k == 1 ? hs.nrm : k == 2 ? hs.uv0 : k == 3 ? hs.uv1 : hs.tan; };
			auto align4 = [](uint64_t b) { return (b + 3u) & ~(uint64_t)3u; };
			std::vector<SourceDesc> srcs(H.sources.size());
			std::vector<StreamDecodeDesc> dec[kKinds]; std::vector<uint32_t> decStart[kKinds];
			std::vector<IndexAssemblyDesc> asmb; std::vector<uint32_t> asmStart;
			uint64_t vtxTotal = 0, idxTotal = 0, decVerts[kKinds] = {}, staged[kKinds + 1] = {}, asmFaces = 0;     // staged[kKinds]: indices
			bool any[kKinds] = {};
			for (size_t i = 0; i < H.sources.size(); i++)
			{
				const HostSource& hs = H.sources[i];
				SourceDesc& d = srcs[i];
				memset(&d, 0, sizeof(d));
				d.vtxOffset = (uint32_t)vtxTotal; d.idxOffset = (uint32_t)idxTotal;
				uint32_t* has[kKinds] = { nullptr, &d.hasNrm, &d.hasUv0, &d.hasUv1, &d.hasTan };
				for (int k = 0; k < kKinds; k++)
				{
					const HostStream& st = streamOf(hs, k);
					if (st.empty()) continue;
					if (has[k]) *has[k] = 1;
					any[k] = true;
					if (st.IsFloat(width[k])) continue;
					decStart[k].push_back((uint32_t)decVerts[k]);
					dec[k].push_back(StreamDecodeDesc{ staged[k], (uint32_t)vtxTotal, st.componentType, st.comps, st.normalized ? 1u : 0u, { 0, 0 } });
					decVerts[k] += hs.numVerts; staged[k] += align4(st.bytes.size());
				}
				if (!hs.DirectIdx() && hs.faces)
				{
					asmStart.push_back((uint32_t)asmFaces);
					asmb.push_back(IndexAssemblyDesc{ staged[kKinds], (uint32_t)idxTotal, hs.idxType, hs.mode, (uint32_t)hs.numVerts, { 0, 0 } });
					asmFaces += hs.faces; staged[kKinds] += align4(hs.idx.size());
				}
				vtxTotal += hs.numVerts; idxTotal += hs.faces * 3;
			}
			// FlattenKernel forms vertex * 4 (tangents) and index offsets in 32 bits
			if (vtxTotal > kMaxVertices || idxTotal > 0xFFFFFFFFull) { ctx.error = "the scene's vertex streams are too large for 32-bit offsets"; return SAILOR_PT_ERR_LIMIT; }
			const uint32_t vtxOffset = (uint32_t)vtxTotal, idxOffset = (uint32_t)idxTotal;
			std::vector<DrawDesc> draws(H.draws.size());
			std::vector<uint32_t> drawStart(H.draws.size() + 1);
			uint64_t triStart = 0;
			for (size_t i = 0; i < H.draws.size(); i++)
			{
				const HostDraw& hd = H.draws[i];
				DrawDesc& d = draws[i];
				memset(&d, 0, sizeof(d));
				memcpy(d.world, hd.world, sizeof(d.world));
				d.source = hd.source; d.material = hd.material;
				drawStart[i] = (uint32_t)triStart;
				triStart += H.sources[hd.source].faces;
			}
			drawStart[H.draws.size()] = (uint32_t)triStart;
			if (triStart != numTris) { ctx.error = "draw table does not cover the scene's triangles"; return SAILOR_PT_ERR_FORMAT; }

			DevBuf<SourceDesc> dSrcs; DevBuf<DrawDesc> dDraws; DevBuf<uint32_t> dDrawStart, dBlockDraw;
			DevBuf<float> dStream[kKinds]; DevBuf<uint32_t> dIdx;
			// staging of the stored forms and their tables: freed when Upload returns, behind the flatten pass on the stream
			DevBuf<uint8_t> dStaged[kKinds + 1]; DevBuf<StreamDecodeDesc> dDec[kKinds]; DevBuf<uint32_t> dDecStart[kKinds], dAsmStart; DevBuf<IndexAssemblyDesc> dAsm;
			dSrcs.Upload(ctx, srcs); dDraws.Upload(ctx, draws); dDrawStart.Upload(ctx, drawStart);
			const uint32_t numBlocks = (numTris - 1u) / kFlattenSpan + 1u;
			dBlockDraw.Alloc(ctx, (size_t)numBlocks + 1);
			dIdx.Alloc(ctx, (size_t)idxOffset + 1);
			for (int k = 0; k < kKinds; k++)
			{
				dStream[k].Alloc(ctx, k == 0 ? (size_t)vtxOffset * 3 + 1 : (any[k] ? (size_t)vtxOffset * width[k] : 1));
				if (staged[k]) { dStaged[k].Alloc(ctx, staged[k]); dDec[k].Upload(ctx, dec[k]); dDecStart[k].Upload(ctx, decStart[k]); }
			}
			if (staged[kKinds]) dStaged[kKinds].Alloc(ctx, staged[kKinds]);
			if (!asmb.empty()) { dAsm.Upload(ctx, asmb); dAsmStart.Upload(ctx, asmStart); }
			if (!ctx.ok) return CudaStatus();
			{
				// With few sources the pieces are copied one by one, straight from the importer's vectors (no host-side concatenation:
				// at 10 M triangles that was hundreds of MB of extra copies); with many, one copy per buffer of a host-side concatenation
				// beats thousands of tiny transfers.
				const bool concat = H.sources.size() > 32;
				struct Pieces
				{
					uint8_t* dev; bool concat; std::vector<uint8_t> host; size_t lo = ~(size_t)0, hi = 0;
					void Put(Ctx& ctx, size_t off, const void* src, size_t bytes)
					{
						if (!bytes) return;
						if (!concat) { DevUpload(ctx, dev + off, src, bytes); return; }
						if (host.size() < off + bytes) host.resize(off + bytes);
						memcpy(host.data() + off, src, bytes);
						lo = off < lo ? off : lo; hi = off + bytes > hi ? off + bytes : hi;
					}
					void Flush(Ctx& ctx) { if (hi > lo) DevUpload(ctx, dev + lo, host.data() + lo, hi - lo); }
				};
				std::vector<Pieces> direct, stage;
				for (int k = 0; k < kKinds; k++) direct.push_back(Pieces{ (uint8_t*)dStream[k].p, concat }), stage.push_back(Pieces{ dStaged[k].p, concat });
				direct.push_back(Pieces{ (uint8_t*)dIdx.p, concat }); stage.push_back(Pieces{ dStaged[kKinds].p, concat });
				uint64_t off[kKinds + 1] = {};
				for (size_t i = 0; i < H.sources.size(); i++)
				{
					const HostSource& hs = H.sources[i];
					const SourceDesc& d = srcs[i];
					for (int k = 0; k < kKinds; k++)
					{
						const HostStream& st = streamOf(hs, k);
						if (st.empty()) continue;
						if (st.IsFloat(width[k])) direct[k].Put(ctx, (size_t)d.vtxOffset * width[k] * sizeof(float), st.bytes.data(), st.bytes.size());
						else { stage[k].Put(ctx, off[k], st.bytes.data(), st.bytes.size()); off[k] += align4(st.bytes.size()); }
					}
					if (hs.DirectIdx()) direct[kKinds].Put(ctx, (size_t)d.idxOffset * sizeof(uint32_t), hs.idx.data(), (size_t)hs.faces * 3 * sizeof(uint32_t));
					else if (hs.faces) { stage[kKinds].Put(ctx, off[kKinds], hs.idx.data(), hs.idx.size()); off[kKinds] += align4(hs.idx.size()); }
				}
				for (int k = 0; k <= kKinds; k++) { direct[k].Flush(ctx); stage[k].Flush(ctx); }
				if (concat) ctx.Sync();                       // the staging vectors die at the end of this block
			}
			vtx.Alloc(ctx, (size_t)numTris * 3); centroid.Alloc(ctx, numTris); shade.Alloc(ctx, (size_t)numTris * 9); uv2.Alloc(ctx, (size_t)numTris * 3);
			if (!ctx.ok) return CudaStatus();

			// secondsFlatten: the decode and assembly passes (none for files of float32 streams and u32 lists) and the flatten pass
			ctx.TimerStart();
			for (int k = 0; k < kKinds; k++)
				if (decVerts[k]) launch_for(ctx, (uint32_t)decVerts[k], DecodeStreamKernel{ dDecStart[k].p, dDec[k].p, (uint32_t)dec[k].size(), width[k], dStaged[k].p, dStream[k].p });
			if (asmFaces) launch_for(ctx, (uint32_t)asmFaces, AssembleIndexKernel{ dAsmStart.p, dAsm.p, (uint32_t)asmb.size(), dStaged[kKinds].p, dIdx.p });
			launch_for(ctx, numBlocks + 1u, FlattenBlockKernel{ dDrawStart.p, (uint32_t)draws.size(), numTris, dBlockDraw.p });
			FlattenKernel fk;
			fk.draws = dDraws.p; fk.drawStart = dDrawStart.p; fk.blockDraw = dBlockDraw.p; fk.sources = dSrcs.p;
			fk.pos = dStream[0].p; fk.nrm = dStream[1].p; fk.uv0 = dStream[2].p; fk.uv1 = dStream[3].p; fk.tan = dStream[4].p; fk.idx = dIdx.p;
			fk.vtx = vtx.p; fk.centroid = centroid.p; fk.shade = shade.p; fk.uv2 = uv2.p;
			launch_for(ctx, numTris, fk);
			stats.secondsFlatten = ctx.TimerStop();

			materials.Upload(ctx, Host().materials);
			std::vector<V4> lightData;
			for (const auto& l : Host().lights) { lightData.push_back(v4(l.direction[0], l.direction[1], l.direction[2], 0.0f)); lightData.push_back(v4(l.intensity[0], l.intensity[1], l.intensity[2], 0.0f)); }
			lights.Upload(ctx, lightData);
			const int rc = UploadTextures();
			ctx.Sync();
			stats.secondsTotal = HostNow() - t0;
			return rc != SAILOR_PT_OK ? rc : CudaStatus();
		}

		int UploadTextures();   // textures.cuh

		// ---------------------------------------------------------------------------------------------- BVH
		int BuildBvh()
		{
			if (built) return SAILOR_PT_OK;
			if (numTris == 0) { ctx.error = "scene has no triangles"; return SAILOR_PT_ERR_FORMAT; }
			const uint32_t N = numTris, maxNodes = 2 * N - 1;
			const double t0 = HostNow();
			// scratch lives with the scene (Ensure only grows): a rebuild allocates nothing
			DevBuf<uint32_t>& idxA = buildU32[0]; DevBuf<uint32_t>& idxB = buildU32[1]; DevBuf<uint32_t>& nodeOfA = buildU32[2]; DevBuf<uint32_t>& nodeOfB = buildU32[3];
			DevBuf<uint32_t>& flags = buildU32[4]; DevBuf<uint32_t>& scan = buildU32[5]; DevBuf<uint32_t>& holes = buildU32[6]; DevBuf<uint32_t>& srcs = buildU32[7];
			DevBuf<uint32_t>& first = buildU32[8]; DevBuf<uint32_t>& count = buildU32[9]; DevBuf<uint32_t>& left = buildU32[10]; DevBuf<uint32_t>& keys = buildU32[11];
			DevBuf<uint32_t>& state = buildU32[12]; DevBuf<uint32_t>& splitAxis = buildU32[13]; DevBuf<uint32_t>& nL = buildU32[14]; DevBuf<uint32_t>& bins = buildU32[15];
			DevBuf<uint32_t>& splitFlag = buildU32[16]; DevBuf<uint32_t>& splitScan = buildU32[17]; DevBuf<uint32_t>& scanScratch = buildU32[18];
			DevBuf<float>& aabb = buildF32[0]; DevBuf<float>& splitPos = buildF32[1]; DevBuf<float>& binScale = buildF32[2];
			idxA.Ensure(ctx, N); idxB.Ensure(ctx, N); nodeOfA.Ensure(ctx, N); nodeOfB.Ensure(ctx, N); flags.Ensure(ctx, N); scan.Ensure(ctx, (size_t)N + 1);
			holes.Ensure(ctx, N); srcs.Ensure(ctx, N);
			first.Ensure(ctx, maxNodes); count.Ensure(ctx, maxNodes); left.Ensure(ctx, maxNodes); keys.Ensure(ctx, (size_t)maxNodes * 12);
			aabb.Ensure(ctx, (size_t)maxNodes * 6); state.Ensure(ctx, maxNodes); splitPos.Ensure(ctx, maxNodes); splitAxis.Ensure(ctx, maxNodes); nL.Ensure(ctx, maxNodes);
			binScale.Ensure(ctx, (size_t)maxNodes * 6);
			// a node is binned only when it holds > 4 triangles, so one level never bins more than N/5 nodes
			const size_t maxBinned = (size_t)N / 5 + 1;
			bins.Ensure(ctx, maxBinned * kNodeBinWords); splitFlag.Ensure(ctx, (size_t)N + 1); splitScan.Ensure(ctx, (size_t)N + 2);
			DevBuf<uint32_t>& binSlot = buildU32[19]; DevBuf<uint32_t>& binCounter = buildU32[20];
			binSlot.Ensure(ctx, maxNodes); binCounter.Ensure(ctx, 4);
			if (!ctx.ok) return CudaStatus();

			BuildState s;
			s.vtx = vtx.p; s.centroid = centroid.p; s.idxA = idxA.p; s.idxB = idxB.p; s.nodeOfA = nodeOfA.p; s.nodeOfB = nodeOfB.p;
			s.flags = flags.p; s.scan = scan.p; s.holes = holes.p; s.srcs = srcs.p;
			s.first = first.p; s.count = count.p; s.left = left.p; s.keys = keys.p; s.aabb = aabb.p; s.state = state.p;
			s.splitPos = splitPos.p; s.splitAxis = splitAxis.p; s.nL = nL.p; s.binScale = binScale.p; s.bins = nullptr;
			s.bins = bins.p; s.splitFlag = splitFlag.p; s.splitScan = splitScan.p; s.binSlot = binSlot.p; s.binCounter = binCounter.p; s.n = N;

			ctx.TimerStart();
#if !defined(SPT_EMU)
			if (N <= kSmallBuildMax && !getenv("SAILOR_PT_NO_SMALL_BUILD"))
			{
				// small scene: the whole build in one launch of one CTA (bvh_build_small.cuh), same functors, same bits
				DevBuf<uint32_t>& internalCount = buildU32[21]; DevBuf<uint32_t>& refIdx = buildU32[22]; DevBuf<uint32_t>& rank = buildU32[23];
				internalCount.Ensure(ctx, maxNodes); refIdx.Ensure(ctx, maxNodes); rank.Ensure(ctx, maxNodes);
				flags.Ensure(ctx, maxNodes); scan.Ensure(ctx, (size_t)maxNodes + 1); buildF32[3].Ensure(ctx, N);
				refNodes.Ensure(ctx, maxNodes); mapping.Ensure(ctx, N); tnodes.Ensure(ctx, N); ttris.Ensure(ctx, N);
				if (!ctx.ok) return CudaStatus();
				s.flags = flags.p; s.scan = scan.p;
				SmallBuildOut o;
				o.internalCount = internalCount.p; o.refIdx = refIdx.p; o.rank = rank.p; o.leafCountByRef = flags.p; o.leafOffsetByRef = scan.p; o.leafCountAtSlot = holes.p;
				o.areaScratch = buildF32[3].p; o.refNodes = refNodes.p; o.mapping = mapping.p; o.tnodes = tnodes.p; o.ttris = ttris.p;
				o.result = counter.p + 8; o.maxNodes = maxNodes;
				k_build_small<<<1, kSmallBuildBlock, 0, ctx.stream>>>(s, o);
				ctx.kernelLaunches++;
				SPT_CUDA_CHECK(ctx, cudaGetLastError());
				uint32_t res[4] = { 0u, 0u, 0u, 1u };
				DevDownload(ctx, res, o.result, sizeof(res));
				if (ctx.ok && res[3] == 0u)
				{
					nodesUsed = res[0]; numInternal = res[1]; numLevels = res[2];
					rootRef = numInternal ? 0u : kLeafBit;
					hasWide = false;
					scratchLeft = s.left; scratchCount = s.count; scratchAabb = s.aabb; scratchRefIdx = refIdx.p; scratchLeafOffset = scan.p;
					int rcw = BuildFast(s.left, s.count, s.aabb, rank.p, refIdx.p, scan.p);
					if (rcw == SAILOR_PT_OK && wantWide) rcw = BuildWide(s.left, s.count, s.aabb, refIdx.p, scan.p);
					if (rcw != SAILOR_PT_OK) { ctx.TimerStop(); return rcw; }
					stats.secondsBvhBuild = ctx.TimerStop();
					stats.secondsTotal = HostNow() - t0;
					built = ctx.ok;
					return CudaStatus();
				}
				if (!ctx.ok) return CudaStatus();
				// deeper than kSmallBuildLevels (degenerate input): redo it with the multi-launch build below
			}
#endif
			launch_for(ctx, N, InitSlotsKernel{ s });
			const uint32_t rootInit[2] = { 0u, N };
			DevUpload(ctx, first.p, &rootInit[0], 4); DevUpload(ctx, count.p, &rootInit[1], 4);   // BVH.cpp:291-293

			std::vector<uint32_t> levelStart; std::vector<uint32_t> levelCount;
			uint32_t start = 0, cnt = 1;
			while (cnt && ctx.ok)
			{
				levelStart.push_back(start); levelCount.push_back(cnt);
				DevMemset(ctx, binCounter.p, 0, sizeof(uint32_t));
				launch_for(ctx, cnt, InitNodesKernel{ s, start });
				LaunchBuildBounds(ctx, s, start);
				launch_for(ctx, cnt, PrepareKernel{ s, start });
				{
					const uint64_t words = (uint64_t)(cnt < maxBinned ? cnt : maxBinned) * kNodeBinWords;
					for (uint64_t base = 0; base < words; base += 1ull << 30) launch_for(ctx, (uint32_t)(words - base < (1ull << 30) ? words - base : (1ull << 30)), BinInitKernel{ s, base });
				}
				LaunchBuildBin(ctx, s, start);
				launch_for(ctx, cnt, SplitKernel{ s, start });
				launch_for(ctx, N, FlagKernel{ s, start });
				ExclusiveScanU32(ctx, flags.p, scan.p, N, scanScratch);
				launch_for(ctx, cnt, CountKernel{ s, start });
				ExclusiveScanU32(ctx, splitFlag.p, splitScan.p, cnt, scanScratch);
				launch_for(ctx, cnt, AllocKernel{ s, start, start + cnt });
				launch_for(ctx, N, HoleKernel{ s, start });
				launch_for(ctx, N, ScatterKernel{ s, start });
				uint32_t numSplit = 0;
				DevDownload(ctx, &numSplit, splitScan.p + cnt, 4);
				{ uint32_t* t = s.idxA; s.idxA = s.idxB; s.idxB = t; t = s.nodeOfA; s.nodeOfA = s.nodeOfB; s.nodeOfB = t; }
				start += cnt; cnt = 2 * numSplit;
			}
			nodesUsed = start;
			numLevels = (uint32_t)levelStart.size();

			// renumber into the reference's allocation order and emit both layouts
			DevBuf<uint32_t>& internalCount = buildU32[21]; DevBuf<uint32_t>& refIdx = buildU32[22]; DevBuf<uint32_t>& rank = buildU32[23];
			DevBuf<uint32_t>& leafCountByRef = flags; DevBuf<uint32_t>& leafOffsetByRef = scan; DevBuf<uint32_t>& leafCountAtSlot = holes;   // partition scratch is free now
			DevBuf<float>& areaScratch = buildF32[3];
			internalCount.Ensure(ctx, maxNodes); refIdx.Ensure(ctx, maxNodes); rank.Ensure(ctx, maxNodes);
			leafCountByRef.Ensure(ctx, maxNodes); leafOffsetByRef.Ensure(ctx, (size_t)maxNodes + 1); areaScratch.Ensure(ctx, N);
			refNodes.Ensure(ctx, maxNodes); mapping.Ensure(ctx, N);
			if (!ctx.ok) return CudaStatus();
			refNodes.Zero(ctx, maxNodes); refIdx.Zero(ctx, nodesUsed); rank.Zero(ctx, nodesUsed); leafCountAtSlot.Zero(ctx, N);
			for (size_t l = levelStart.size(); l-- > 0;) launch_for(ctx, levelCount[l], SubtreeKernel{ s, levelStart[l], internalCount.p });
			for (size_t l = 0; l < levelStart.size(); l++) launch_for(ctx, levelCount[l], RenumberKernel{ s, levelStart[l], internalCount.p, refIdx.p, rank.p });
			launch_for(ctx, nodesUsed, LeafCountKernel{ s, refIdx.p, leafCountByRef.p });
			ExclusiveScanU32(ctx, leafCountByRef.p, leafOffsetByRef.p, nodesUsed, scanScratch);
			launch_for(ctx, nodesUsed, EmitKernel{ s, refIdx.p, leafOffsetByRef.p, s.idxA, refNodes.p, mapping.p, areaScratch.p });
			DevDownload(ctx, &numInternal, internalCount.p, 4);

			tnodes.Ensure(ctx, numInternal ? numInternal : 1); ttris.Ensure(ctx, N);
			if (!ctx.ok) return CudaStatus();
			launch_for(ctx, nodesUsed, LeafCountAtSlotKernel{ s.left, s.count, refIdx.p, leafOffsetByRef.p, leafCountAtSlot.p });
			launch_for(ctx, nodesUsed, PackNodesKernel{ s.left, rank.p, refIdx.p, leafOffsetByRef.p, s.aabb, tnodes.p });
			launch_for(ctx, N, PackTrisKernel{ vtx.p, mapping.p, leafCountAtSlot.p, ttris.p, N });
			rootRef = numInternal ? 0u : kLeafBit;      // a root that never split is one leaf at slot 0
			{
				hasWide = false;
				scratchLeft = s.left; scratchCount = s.count; scratchAabb = s.aabb; scratchRefIdx = refIdx.p; scratchLeafOffset = leafOffsetByRef.p;
				int rcw = BuildFast(s.left, s.count, s.aabb, rank.p, refIdx.p, leafOffsetByRef.p);
				if (rcw == SAILOR_PT_OK && wantWide) rcw = BuildWide(s.left, s.count, s.aabb, refIdx.p, leafOffsetByRef.p);
				if (rcw != SAILOR_PT_OK) { ctx.TimerStop(); return rcw; }
			}
			stats.secondsBvhBuild = ctx.TimerStop();
			stats.secondsTotal = HostNow() - t0;
			built = ctx.ok;
			return CudaStatus();
		}
	};
}
