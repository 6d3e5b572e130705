// gltf_loader.cpp — product glTF 2.0 / GLB front end (host C++; no third-party parser).
//
// Replaces the Assimp import of the reference's PathTracer::Run (reference PathTracer.cpp:84-98,102-153,164-381;
// MaterialUtils.cpp:64-198 for which mesh fields are consumed).  It only PARSES: vertex streams are handed to the
// device untransformed (flatten.cuh does the per-triangle arithmetic), texels stay RGBA8 (texture_convert kernel).
// Loader contract (shared with the oracle's restated driver, DESIGN.md): default scene, depth-first node order,
// world = node * parent in the reference's transposed-matrix convention, TRIANGLES primitives only (the oracle's side), u8 material
// index, texture slots deduplicated by (image, clamping, channels) in the order base / normal / metallicRoughness /
// emissive / transmission, directional KHR_lights_punctual only (intensity = color * intensity / 683).
// EXT_mesh_gpu_instancing (which the oracle does not read) draws a node's mesh once per instance, exactly as if the node had one
// child node per instance, placed before its own children.  TRIANGLE_STRIP / TRIANGLE_FAN primitives and sparse accessors (which the
// oracle does not read either) are imported as their float32 TRIANGLES-list twin: streams stay in their stored form and are decoded
// and assembled on the device (flatten.cuh).
#include "host_scene.h"
#include "hd.h"
#if defined(__unix__)
#include <sys/mman.h>
#include <sys/stat.h>
#include <fcntl.h>
#include <unistd.h>
#endif
#include "../../include/sailor_pt.h"

#include <array>
#include <atomic>
#include <cmath>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <memory>
#include <new>
#include <stdexcept>

namespace spt
{
	namespace
	{
		// ------------------------------------------------------------------------------------------ JSON
		struct Json
		{
			enum Type { Null, Bool, Number, String, Array, Object } type = Null;
			bool b = false;
			double num = 0.0;
			std::string str;
			std::vector<Json> arr;
			std::vector<std::pair<std::string, Json>> obj;

			const Json* find(const char* key) const
			{
				if (type != Object) return nullptr;
				for (const auto& kv : obj) if (kv.first == key) return &kv.second;
				return nullptr;
			}
			const Json& at(const char* key) const { static const Json none; const Json* j = find(key); return j ? *j : none; }
			const Json& at(size_t i) const { static const Json none; return (type == Array && i < arr.size()) ? arr[i] : none; }
			bool isNumber() const { return type == Number; }
			size_t size() const { return type == Array ? arr.size() : 0; }
			double number(double def) const { return type == Number ? num : def; }
			int integer(int def) const { return type == Number ? (int)num : def; }
		};

		struct JsonParser
		{
			const char* p; const char* end; std::string err;
			void ws() { while (p < end && (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r')) p++; }
			bool fail(const char* m) { if (err.empty()) err = m; return false; }
			bool value(Json& out, int depth)
			{
				if (depth > 256) return fail("json nesting too deep");
				ws();
				if (p >= end) return fail("unexpected end of json");
				const char c = *p;
				if (c == '{')
				{
					out.type = Json::Object; p++; ws();
					if (p < end && *p == '}') { p++; return true; }
					for (;;)
					{
						ws();
						Json key;
						if (p >= end || *p != '"' || !string(key.str)) return fail("object key expected");
						ws();
						if (p >= end || *p != ':') return fail("':' expected");
						p++;
						out.obj.emplace_back(std::move(key.str), Json());
						if (!value(out.obj.back().second, depth + 1)) return false;
						ws();
						if (p < end && *p == ',') { p++; continue; }
						if (p < end && *p == '}') { p++; return true; }
						return fail("',' or '}' expected");
					}
				}
				if (c == '[')
				{
					out.type = Json::Array; p++; ws();
					if (p < end && *p == ']') { p++; return true; }
					for (;;)
					{
						out.arr.emplace_back();
						if (!value(out.arr.back(), depth + 1)) return false;
						ws();
						if (p < end && *p == ',') { p++; continue; }
						if (p < end && *p == ']') { p++; return true; }
						return fail("',' or ']' expected");
					}
				}
				if (c == '"') { out.type = Json::String; return string(out.str); }
				if (end - p >= 4 && !strncmp(p, "true", 4)) { out.type = Json::Bool; out.b = true; p += 4; return true; }
				if (end - p >= 5 && !strncmp(p, "false", 5)) { out.type = Json::Bool; out.b = false; p += 5; return true; }
				if (end - p >= 4 && !strncmp(p, "null", 4)) { out.type = Json::Null; p += 4; return true; }
				// number: strtod on a bounded copy (same correctly-rounded double the reference's json parser produces)
				const char* s = p;
				while (p < end && (strchr("+-.eE", *p) || (*p >= '0' && *p <= '9'))) p++;
				if (s == p) return fail("unexpected character in json");
				const std::string tok(s, p);
				char* e = nullptr;
				out.num = strtod(tok.c_str(), &e);
				if (!e || *e) return fail("bad number");
				out.type = Json::Number;
				return true;
			}
			static void utf8(std::string& o, uint32_t cp)
			{
				if (cp < 0x80) o += (char)cp;
				else if (cp < 0x800) { o += (char)(0xC0 | (cp >> 6)); o += (char)(0x80 | (cp & 63)); }
				else if (cp < 0x10000) { o += (char)(0xE0 | (cp >> 12)); o += (char)(0x80 | ((cp >> 6) & 63)); o += (char)(0x80 | (cp & 63)); }
				else { o += (char)(0xF0 | (cp >> 18)); o += (char)(0x80 | ((cp >> 12) & 63)); o += (char)(0x80 | ((cp >> 6) & 63)); o += (char)(0x80 | (cp & 63)); }
			}
			bool hex4(uint32_t& v)
			{
				if (end - p < 4) return false;
				v = 0;
				for (int i = 0; i < 4; i++)
				{
					const char h = *p++;
					v <<= 4;
					if (h >= '0' && h <= '9') v |= h - '0'; else if (h >= 'a' && h <= 'f') v |= h - 'a' + 10; else if (h >= 'A' && h <= 'F') v |= h - 'A' + 10; else return false;
				}
				return true;
			}
			bool string(std::string& out)
			{
				p++; // opening quote
				while (p < end)
				{
					const char c = *p++;
					if (c == '"') return true;
					if (c != '\\') { out += c; continue; }
					if (p >= end) break;
					const char e = *p++;
					switch (e)
					{
					case 'n': out += '\n'; break; case 't': out += '\t'; break; case 'r': out += '\r'; break;
					case 'b': out += '\b'; break; case 'f': out += '\f'; break;
					case 'u':
					{
						uint32_t cp;
						if (!hex4(cp)) return fail("bad \\u escape");
						if (cp >= 0xD800 && cp < 0xDC00 && end - p >= 6 && p[0] == '\\' && p[1] == 'u')
						{
							p += 2; uint32_t lo;
							if (!hex4(lo)) return fail("bad \\u escape");
							cp = 0x10000 + ((cp - 0xD800) << 10) + (lo - 0xDC00);
						}
						utf8(out, cp);
						break;
					}
					default: out += e; break;
					}
				}
				return fail("unterminated string");
			}
		};

		// ------------------------------------------------------------------------------------------ helpers
		bool ReadFile(const std::string& path, std::vector<uint8_t>& out)
		{
			FILE* f = fopen(path.c_str(), "rb");
			if (!f) return false;
			fseek(f, 0, SEEK_END);
			const long n = ftell(f);
			fseek(f, 0, SEEK_SET);
			out.resize(n > 0 ? (size_t)n : 0);
			const size_t got = out.empty() ? 0 : fread(out.data(), 1, out.size(), f);
			fclose(f);
			return got == out.size();
		}

		bool Base64(const char* s, size_t n, std::vector<uint8_t>& out)
		{
			static int8_t T[256]; static bool init = false;
			if (!init)
			{
				memset(T, -1, sizeof(T));
				const char* A = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
				for (int i = 0; i < 64; i++) T[(uint8_t)A[i]] = (int8_t)i;
				init = true;
			}
			uint32_t acc = 0; int bits = 0;
			out.reserve(n * 3 / 4);
			for (size_t i = 0; i < n; i++)
			{
				const int8_t v = T[(uint8_t)s[i]];
				if (v < 0) { if (s[i] == '=' || s[i] == '\n' || s[i] == '\r') continue; return false; }
				acc = (acc << 6) | (uint32_t)v; bits += 6;
				if (bits >= 8) { bits -= 8; out.push_back((uint8_t)(acc >> bits)); }
			}
			return true;
		}

		std::string UriDecode(const std::string& s)
		{
			std::string o;
			for (size_t i = 0; i < s.size(); i++)
			{
				if (s[i] == '%' && i + 2 < s.size() + 0 && isxdigit((unsigned char)s[i + 1]) && isxdigit((unsigned char)s[i + 2]))
				{
					o += (char)strtol(s.substr(i + 1, 2).c_str(), nullptr, 16); i += 2;
				}
				else o += s[i];
			}
			return o;
		}

		bool LoadUri(const std::string& uri, const std::string& baseDir, std::vector<uint8_t>& out)
		{
			if (uri.compare(0, 5, "data:") == 0)
			{
				const size_t comma = uri.find(',');
				if (comma == std::string::npos) return false;
				return Base64(uri.c_str() + comma + 1, uri.size() - comma - 1, out);
			}
			return ReadFile(baseDir + UriDecode(uri), out);
		}

		// mat4 product in glm's operation order (glm/detail/type_mat4x4.inl:630-648): R[c] = A0*B[c][0] + A1*B[c][1] + A2*B[c][2] + A3*B[c][3]
		void Mat4Mul(const float* A, const float* B, float* R)
		{
			float tmp[16];
			for (int c = 0; c < 4; c++)
				for (int r = 0; r < 4; r++)
					tmp[c * 4 + r] = A[0 * 4 + r] * B[c * 4 + 0] + A[1 * 4 + r] * B[c * 4 + 1] + A[2 * 4 + r] * B[c * 4 + 2] + A[3 * 4 + r] * B[c * 4 + 3];
			memcpy(R, tmp, sizeof(tmp));
		}

		// A readable accessor: `count` elements of `elem` bytes at base + i * stride (base null: zeros), then element sparseAt[k]
		// replaced by the k-th element of sparseValues for k < sparseCount (sparseAt strictly increasing).  Nothing is copied here:
		// whatever is sized by `count` is allocated by the caller, after the count has passed the caller's limit.
		struct Accessor
		{
			const uint8_t* base = nullptr;
			size_t stride = 0, count = 0, elem = 0;
			int componentType = 0, comps = 0;
			bool normalized = false, valid = false;
			const uint8_t* sparseAt = nullptr; const uint8_t* sparseValues = nullptr;
			size_t sparseCount = 0; int sparseType = 0;
		};

		int CompsOf(const std::string& t)
		{
			if (t == "SCALAR") return 1; if (t == "VEC2") return 2; if (t == "VEC3") return 3; if (t == "VEC4") return 4;
			if (t == "MAT2") return 4; if (t == "MAT3") return 9; if (t == "MAT4") return 16;
			return 0;
		}
		int CompSize(int ct)
		{
			switch (ct) { case 5120: case 5121: return 1; case 5122: case 5123: return 2; case 5125: case 5126: return 4; default: return 0; }
		}

		struct Gltf
		{
			Json root;
			struct Buffer       // bytes of one glTF buffer: a view into the mapped GLB (BIN chunk) or owned storage (uri / data: buffers)
			{
				std::vector<uint8_t> own; const uint8_t* p = nullptr; size_t n = 0;
				const uint8_t* data() const { return p; }
				size_t size() const { return n; }
				const uint8_t* begin() const { return p; }
			};
			std::vector<Buffer> buffers;
			std::string baseDir;

			// An accessor with a bufferView reads it; one without reads zeros, and only when it has a sparse block.  A malformed sparse
			// block makes the accessor unreadable.
			Accessor accessor(int index) const
			{
				Accessor a;
				const Json& accs = root.at("accessors");
				if (index < 0 || (size_t)index >= accs.size()) return a;
				const Json& acc = accs.at(index);
				const Json* sparse = acc.find("sparse");
				const bool hasView = acc.find("bufferView") || !sparse;
				const int bv = acc.at("bufferView").integer(-1);
				const Json& views = root.at("bufferViews");
				if (hasView && (bv < 0 || (size_t)bv >= views.size())) return a;
				static const Json none;
				const Json& view = hasView ? views.at(bv) : none;
				const int bi = view.at("buffer").integer(-1);
				if (hasView && (bi < 0 || (size_t)bi >= buffers.size())) return a;
				a.comps = CompsOf(acc.at("type").str);
				a.componentType = acc.at("componentType").integer(0);
				a.elem = (size_t)CompSize(a.componentType) * a.comps;
				// sizes and offsets come from the file: negative or absurd numbers are rejected before any size_t arithmetic, and the
				// range check is written so that it cannot wrap
				const double dbs = view.at("byteStride").number(0), dvo = view.at("byteOffset").number(0), dao = acc.at("byteOffset").number(0), dcount = acc.at("count").number(0);
				if (!(dbs >= 0 && dbs <= 65536.0 && dvo >= 0 && dvo < kLim && dao >= 0 && dao < kLim && dcount >= 0 && dcount < kLim)) return a;
				const size_t bs = (size_t)dbs;
				a.stride = bs ? bs : a.elem;
				const size_t off = (size_t)dvo + (size_t)dao;
				a.count = (size_t)dcount;
				a.normalized = acc.at("normalized").type == Json::Bool && acc.at("normalized").b;
				if (!a.elem || !a.count) return a;
				if (hasView)
				{
					const size_t size = buffers[bi].size();
					if (off > size || a.elem > size - off || a.stride == 0 || (a.count - 1) > (size - off - a.elem) / a.stride) return a;
					a.base = buffers[bi].data() + off;
				}
				if (sparse && !Sparse(*sparse, a)) return a;
				a.valid = true;
				return a;
			}

			static constexpr double kLim = 1e15;

			// `bytes` bytes at o.byteOffset inside the bufferView o.bufferView, or null when they are not all inside it and its buffer
			const uint8_t* ViewBytes(const Json& o, size_t bytes) const
			{
				const Json& views = root.at("bufferViews");
				const int bv = o.at("bufferView").integer(-1);
				if (bv < 0 || (size_t)bv >= views.size()) return nullptr;
				const Json& view = views.at(bv);
				const int bi = view.at("buffer").integer(-1);
				if (bi < 0 || (size_t)bi >= buffers.size()) return nullptr;
				const double dvo = view.at("byteOffset").number(0), dlen = view.at("byteLength").number(0), doo = o.at("byteOffset").number(0);
				if (!(dvo >= 0 && dvo < kLim && dlen >= 0 && dlen < kLim && doo >= 0 && doo < kLim)) return nullptr;
				const size_t vo = (size_t)dvo, len = (size_t)dlen, oo = (size_t)doo, size = buffers[bi].size();
				if (vo > size || len > size - vo || oo > len || bytes > len - oo) return nullptr;
				return buffers[bi].data() + vo + oo;
			}

			// accessor.sparse: count in [1, accessor count], u8 / u16 / u32 indices strictly increasing and below the accessor count,
			// indices and values (tightly packed, the accessor's element type) inside their views
			bool Sparse(const Json& s, Accessor& a) const
			{
				const double dk = s.at("count").number(0);
				if (!(dk >= 1.0 && dk <= (double)a.count) || dk != (double)(uint64_t)dk) return false;
				const size_t k = (size_t)dk;
				const Json& si = s.at("indices");
				const int it = si.at("componentType").integer(0);
				if (it != 5121 && it != 5123 && it != 5125) return false;
				const uint8_t* at = ViewBytes(si, k * (size_t)CompSize(it));
				const uint8_t* values = ViewBytes(s.at("values"), k * a.elem);
				if (!at || !values) return false;
				for (size_t i = 0; i < k; i++)
				{
					const uint32_t v = IndexAt(at, (uint32_t)it, i);
					if (v >= a.count || (i && v <= IndexAt(at, (uint32_t)it, i - 1))) return false;
				}
				a.sparseAt = at; a.sparseValues = values; a.sparseCount = k; a.sparseType = it;
				return true;
			}
		};

		// the bytes of element i (elem of them): a sparse value, the base view's element, or zeros
		const uint8_t* Element(const Accessor& a, size_t i)
		{
			static const uint8_t zeros[64] = {};            // the largest element, MAT4 of float
			size_t lo = 0, hi = a.sparseCount;
			while (lo < hi)
			{
				const size_t mid = (lo + hi) / 2;
				const uint32_t at = IndexAt(a.sparseAt, (uint32_t)a.sparseType, mid);
				if (at == i) return a.sparseValues + mid * a.elem;
				if (at < i) lo = mid + 1; else hi = mid;
			}
			return a.base ? a.base + a.stride * i : zeros;
		}

		// the first `keep` bytes of every element, tightly packed (the stored form the device reads)
		void Gather(const Accessor& a, size_t keep, std::vector<uint8_t>& out)
		{
			out.assign(a.count * keep, 0);
			if (a.base && a.stride == keep) memcpy(out.data(), a.base, out.size());
			else if (a.base) for (size_t i = 0; i < a.count; i++) memcpy(out.data() + i * keep, a.base + a.stride * i, keep);
			for (size_t k = 0; k < a.sparseCount; k++) memcpy(out.data() + (size_t)IndexAt(a.sparseAt, (uint32_t)a.sparseType, k) * keep, a.sparseValues + k * a.elem, keep);
		}

		float ReadFloat(const Accessor& a, size_t i, int c) { return DecodeComponent(Element(a, i), (uint32_t)a.componentType, a.normalized, (uint32_t)c); }

		// an accessor's elements in their stored form, for a vertex stream of the device
		HostStream Stream(const Accessor& a)
		{
			HostStream s;
			Gather(a, a.elem, s.bytes);
			s.componentType = (uint32_t)a.componentType; s.comps = (uint32_t)a.comps; s.normalized = a.normalized;
			return s;
		}

		float ExtNumber(const Json& o, const char* key, float def) { const Json* j = o.find(key); return (j && j->isNumber()) ? (float)j->num : def; }

		struct Builder
		{
			const Gltf& g;
			HostScene& scene;
			std::vector<int> cameraSeen, lightSeen;
			std::vector<std::vector<float>> lightMatrix;
			bool needDefault = false;              // some primitive uses the default material

			int rc = SAILOR_PT_OK;                 // the first refusal (ERR_FORMAT / ERR_LIMIT) stops the traversal
			std::string err;
			// source index by the accessors a primitive reads (POSITION, NORMAL, TANGENT, TEXCOORD_0, TEXCOORD_1, indices) and its mode:
			// -1 when the primitive draws nothing
			std::map<std::array<int, 7>, int> sourceOf;
			uint64_t numVertices = 0;              // of all sources so far, at most kMaxVertices

			bool Refuse(int code, int node, const std::string& what)
			{
				if (rc == SAILOR_PT_OK) { rc = code; err = "node[" + std::to_string(node) + "]: " + what; }
				return false;
			}

			// node local matrix, reference convention = transpose of the mathematical matrix (MaterialUtils.cpp:186-191)
			void LocalMatrix(const Json& n, float* out) const
			{
				const Json& jm = n.at("matrix");
				if (jm.size() == 16)
				{
					float m[16];
					for (int i = 0; i < 16; i++) m[i] = (float)jm.at(i).num;
					for (int c = 0; c < 4; c++) for (int r = 0; r < 4; r++) out[c * 4 + r] = m[r * 4 + c]; // transpose
					return;
				}
				float t[3] = { 0, 0, 0 }, s[3] = { 1, 1, 1 }, q[4] = { 0, 0, 0, 1 };
				if (n.at("translation").size() == 3) for (int i = 0; i < 3; i++) t[i] = (float)n.at("translation").at(i).num;
				if (n.at("scale").size() == 3) for (int i = 0; i < 3; i++) s[i] = (float)n.at("scale").at(i).num;
				if (n.at("rotation").size() == 4) for (int i = 0; i < 4; i++) q[i] = (float)n.at("rotation").at(i).num;
				TrsMatrix(t, q, s, out);
			}

			// translation, rotation quaternion (x, y, z, w), scale -> matrix in the reference convention.  Node TRS and the
			// instances of EXT_mesh_gpu_instancing both go through here, so an instance has the bits of a child node with its TRS.
			static void TrsMatrix(const float* t, const float* q, const float* s, float* out)
			{
				float m[16];
				const float x = q[0], y = q[1], z = q[2], w = q[3];
				const float R[3][3] = {
					{ 1.0f - 2.0f * (y * y + z * z), 2.0f * (x * y - w * z), 2.0f * (x * z + w * y) },
					{ 2.0f * (x * y + w * z), 1.0f - 2.0f * (x * x + z * z), 2.0f * (y * z - w * x) },
					{ 2.0f * (x * z - w * y), 2.0f * (y * z + w * x), 1.0f - 2.0f * (x * x + y * y) } };
				for (int c = 0; c < 3; c++) { for (int r = 0; r < 3; r++) m[c * 4 + r] = R[r][c] * s[c]; m[c * 4 + 3] = 0.0f; }
				m[12] = t[0]; m[13] = t[1]; m[14] = t[2]; m[15] = 1.0f;
				for (int c = 0; c < 4; c++) for (int r = 0; r < 4; r++) out[c * 4 + r] = m[r * 4 + c]; // transpose
			}

			// the streams of a primitive, read on its first use; -1 when it draws nothing (a mode other than TRIANGLES, TRIANGLE_STRIP
			// and TRIANGLE_FAN, POSITION unreadable) or when it is refused (rc set: more vertices or faces than a scene may have)
			int Source(const Json& prim, int node)
			{
				const int mode = prim.at("mode").integer(4);
				if (mode != 4 && mode != 5 && mode != 6) return -1;
				const Json& attrs = prim.at("attributes");
				const std::array<int, 7> key = { attrs.at("POSITION").integer(-1), attrs.at("NORMAL").integer(-1), attrs.at("TANGENT").integer(-1),
					attrs.at("TEXCOORD_0").integer(-1), attrs.at("TEXCOORD_1").integer(-1), prim.at("indices").integer(-1), mode };
				const auto found = sourceOf.find(key);
				if (found != sourceOf.end()) return found->second;
				int& slot = sourceOf[key];
				slot = -1;
				const Accessor pos = g.accessor(key[0]);
				if (!pos.valid) return -1;
				const Accessor idx = g.accessor(key[5]);
				// the counts come from the file (a sparse accessor without a bufferView is not bounded by the file's size): each passes
				// the limit of its consumer before anything is sized by it
				const uint64_t n = idx.valid ? idx.count : pos.count;
				const uint64_t faces = mode == 4 ? n / 3 : (n > 2 ? n - 2 : 0);
				if (pos.count > kMaxVertices - numVertices) { Refuse(SAILOR_PT_ERR_LIMIT, node, "the scene has more than " + std::to_string(kMaxVertices) + " vertices"); return -1; }
				if (faces > kMaxTriangles) { Refuse(SAILOR_PT_ERR_LIMIT, node, "a primitive has more than " + std::to_string(kMaxTriangles) + " triangles"); return -1; }
				numVertices += pos.count;
				scene.sources.emplace_back();
				HostSource& hp = scene.sources.back();
				slot = (int)scene.sources.size() - 1;
				hp.numVerts = pos.count; hp.mode = (uint32_t)mode; hp.faces = faces;
				hp.pos = Stream(pos);
				// an attribute stream whose element count differs from POSITION's is malformed: it is ignored (the device buffers are
				// sized by the position count, and FlattenKernel indexes every stream with position indices)
				auto attr = [&](int k) { Accessor a = g.accessor(key[k]); if (a.valid && a.count != pos.count) a.valid = false; return a; };
				const Accessor nrm = attr(1);
				if (nrm.valid) hp.nrm = Stream(nrm);
				const Accessor tan = attr(2);
				if (tan.valid && tan.comps == 4) hp.tan = Stream(tan);
				const Accessor uv0 = attr(3);
				if (uv0.valid) hp.uv0 = Stream(uv0);
				const Accessor uv1 = attr(4);
				if (uv1.valid) hp.uv1 = Stream(uv1);
				if (!idx.valid) return slot;                     // not indexed: AssembleIndexKernel numbers the vertices
				hp.idxType = (uint32_t)idx.componentType;
				const size_t cs = (size_t)CompSize(idx.componentType);
				const bool packed = idx.base && idx.stride == cs && !idx.sparseCount;       // what exporters write: read in place
				const bool typed = hp.idxType == 5121 || hp.idxType == 5123 || hp.idxType == 5125;
				const bool list = mode == 4 && typed && (hp.idxType == 5125 || hp.FloatStreams());
				if (!packed) Gather(idx, cs, hp.idx);
				else if (!list) hp.idx.assign(idx.base, idx.base + idx.count * cs);
				if (!list) return slot;
				// A TRIANGLES list of u32 indices, or of u8 / u16 indices in a source of float32 streams, goes to the device as u32
				// triples that FlattenKernel reads in place (so files of float32 streams upload what they always did).  Out-of-range
				// indices read vertex 0 (no crash on bad files), as AssembleIndexKernel does for every other index form.  Typed loops:
				// the compiler vectorises them (a per-element switch cost ~10 ms per million triangles).
				const uint8_t* stored = packed ? idx.base : hp.idx.data();
				const size_t n3 = (size_t)faces * 3;
				std::vector<uint8_t> u32(n3 * 4);
				const uint32_t limit = (uint32_t)(pos.count < 0xFFFFFFFFull ? pos.count : 0xFFFFFFFFull);
				auto widen = [&](auto zero)
					{
						using T = decltype(zero);
						for (size_t i = 0; i < n3; i++)
						{
							T v; memcpy(&v, stored + sizeof(T) * i, sizeof(T));
							const uint32_t c = (uint32_t)v < limit ? (uint32_t)v : 0u;
							memcpy(u32.data() + 4 * i, &c, 4);
						}
					};
				if (hp.idxType == 5121) widen(uint8_t(0)); else if (hp.idxType == 5123) widen(uint16_t(0)); else widen(uint32_t(0));
				hp.idx.swap(u32);
				hp.idxType = 5125;
				return slot;
			}

			// a primitive without a material (or with an index outside the array) gets the DEFAULT material, which Assimp's glTF2
			// importer appends after the file's own materials (index = their count); LoadGltf appends it when `needDefault` is set
			uint32_t Material(const Json& prim)
			{
				const int mat = prim.at("material").integer(-1);
				const size_t nm = g.root.at("materials").size();
				const bool own = mat >= 0 && (size_t)mat < nm;
				if (!own) needDefault = true;
				return (uint32_t)(own ? (size_t)mat : nm);
			}

			// draws every primitive of a mesh once per world matrix (one matrix: an ordinary node; K: the node's instances), instance-major
			void DrawMesh(const Json& prims, const std::vector<int>& src, const float* worlds, size_t count)
			{
				for (size_t k = 0; k < count; k++)
					for (size_t i = 0; i < prims.size(); i++)
					{
						if (src[i] < 0) continue;
						const uint32_t material = Material(prims.at(i));
						const uint64_t faces = scene.sources[(size_t)src[i]].faces;
						if (!faces) continue;
						scene.draws.emplace_back();
						HostDraw& d = scene.draws.back();
						d.source = (uint32_t)src[i]; d.material = material;
						memcpy(d.world, worlds + k * 16, sizeof(d.world));
						scene.numTriangles += faces;
					}
			}

			// EXT_mesh_gpu_instancing: the world matrix of every instance, TRS_i * nodeWorld (a child node with that TRS)
			bool InstanceMatrices(const Json& attrs, int node, const float* world, uint64_t meshFaces, std::vector<float>& out)
			{
				struct Attr { const char* name; int comps; Accessor a; bool present; } A[3] = { { "TRANSLATION", 3, {}, false }, { "ROTATION", 4, {}, false }, { "SCALE", 3, {}, false } };
				size_t count = 0; bool any = false;
				for (Attr& at : A)
				{
					const Json* j = attrs.find(at.name);
					if (!j) continue;
					at.present = true;
					at.a = g.accessor(j->isNumber() ? j->integer(-1) : -1);
					if (!at.a.valid) return Refuse(SAILOR_PT_ERR_FORMAT, node, std::string("EXT_mesh_gpu_instancing: the ") + at.name + " accessor is missing or unreadable");
					if (at.a.comps != at.comps) return Refuse(SAILOR_PT_ERR_FORMAT, node, std::string("EXT_mesh_gpu_instancing: ") + at.name + (at.comps == 3 ? " is not VEC3" : " is not VEC4"));
					if (any && at.a.count != count) return Refuse(SAILOR_PT_ERR_FORMAT, node, "EXT_mesh_gpu_instancing: the attributes have different counts");
					count = at.a.count; any = true;
				}
				// names starting with '_' are application-specific and ignored (the extension's specification); nothing else is defined
				if (!any) return Refuse(SAILOR_PT_ERR_FORMAT, node, "EXT_mesh_gpu_instancing: no TRANSLATION, ROTATION or SCALE attribute");
				// the expanded triangle count in 64 bits, before any per-instance data exists
				if (meshFaces && (uint64_t)count > (kMaxTriangles - scene.numTriangles) / meshFaces)
					return Refuse(SAILOR_PT_ERR_LIMIT, node, "EXT_mesh_gpu_instancing: " + std::to_string(count) + " instances of " + std::to_string(meshFaces) +
						" triangles exceed the " + std::to_string(kMaxTriangles) + " triangles a scene may have");
				// a mesh that draws nothing gets no per-instance data: its count has passed no bound (a sparse accessor without a
				// bufferView can claim any count below 1e15)
				if (!meshFaces) return true;
				out.resize(count * 16);
				for (size_t i = 0; i < count; i++)
				{
					float t[3] = { 0, 0, 0 }, q[4] = { 0, 0, 0, 1 }, s[3] = { 1, 1, 1 }, local[16];
					if (A[0].present) for (int c = 0; c < 3; c++) t[c] = ReadFloat(A[0].a, i, c);
					if (A[1].present) for (int c = 0; c < 4; c++) q[c] = ReadFloat(A[1].a, i, c);
					if (A[2].present) for (int c = 0; c < 3; c++) s[c] = ReadFloat(A[2].a, i, c);
					TrsMatrix(t, q, s, local);
					Mat4Mul(local, world, out.data() + i * 16);
				}
				return true;
			}

			void Node(int index, const float* parent, int depth)
			{
				const Json& nodes = g.root.at("nodes");
				if (rc != SAILOR_PT_OK || index < 0 || (size_t)index >= nodes.size() || depth > 512) return;
				const Json& n = nodes.at(index);
				float local[16], world[16];
				LocalMatrix(n, local);
				Mat4Mul(local, parent, world);                    // nodeMatrix * parentMatrix (MaterialUtils.cpp:191-197)
				const int mesh = n.at("mesh").integer(-1);
				if (mesh >= 0 && (size_t)mesh < g.root.at("meshes").size())
				{
					const Json& prims = g.root.at("meshes").at(mesh).at("primitives");
					std::vector<int> src(prims.size());
					uint64_t faces = 0;
					for (size_t i = 0; i < prims.size(); i++) { src[i] = Source(prims.at(i), index); if (src[i] >= 0) faces += scene.sources[(size_t)src[i]].faces; }
					if (rc != SAILOR_PT_OK) return;
					const Json* inst = n.at("extensions").find("EXT_mesh_gpu_instancing");
					if (inst && inst->find("attributes"))
					{
						std::vector<float> worlds;
						if (!InstanceMatrices(inst->at("attributes"), index, world, faces, worlds)) return;
						DrawMesh(prims, src, worlds.data(), worlds.size() / 16);
					}
					else
					{
						if (faces > kMaxTriangles - scene.numTriangles) { Refuse(SAILOR_PT_ERR_LIMIT, index, "the scene has more than " + std::to_string(kMaxTriangles) + " triangles"); return; }
						DrawMesh(prims, src, world, 1);
					}
				}
				const int cam = n.at("camera").integer(-1);
				if (cam >= 0 && (size_t)cam < scene.cameras.size() && !cameraSeen[cam])
				{
					cameraSeen[cam] = 1;
					memcpy(scene.cameras[cam].matrix, world, sizeof(world));
					const std::string& nodeName = n.at("name").str;
					if (!nodeName.empty()) scene.cameras[cam].name = nodeName;
				}
				const Json* kl = n.at("extensions").find("KHR_lights_punctual");
				if (kl && kl->at("light").isNumber())
				{
					const int li = kl->at("light").integer(-1);
					if (li >= 0 && (size_t)li < lightSeen.size() && !lightSeen[li]) { lightSeen[li] = 1; lightMatrix[li].assign(world, world + 16); }
				}
				const Json& ch = n.at("children");
				for (size_t i = 0; i < ch.size(); i++) Node(ch.at(i).integer(-1), world, depth + 1);
			}
		};
	}

	namespace
	{
		// The scene file is mapped, not read: a 10 M-triangle GLB is hundreds of MB, and read-into-a-vector costs a zero fill, a copy
		// out of the page cache and a page fault per 4 KB of it.  Falls back to ReadFile where mmap is not available.
		struct MappedFile
		{
			const uint8_t* p = nullptr; size_t n = 0; bool mapped = false; std::vector<uint8_t> own;
			const uint8_t* data() const { return p; }
			size_t size() const { return n; }
			bool Open(const std::string& path)
			{
#if defined(__unix__)
				const int fd = open(path.c_str(), O_RDONLY);
				if (fd >= 0)
				{
					struct stat st;
					if (fstat(fd, &st) == 0 && st.st_size > 0)
					{
						void* m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
						if (m != MAP_FAILED) { p = (const uint8_t*)m; n = (size_t)st.st_size; mapped = true; }
					}
					close(fd);
					if (mapped) return true;
				}
#endif
				if (!ReadFile(path, own)) return false;
				p = own.data(); n = own.size();
				return true;
			}
			~MappedFile()
			{
#if defined(__unix__)
				if (mapped) munmap(const_cast<uint8_t*>(p), n);
#endif
			}
		};
	}

	static int LoadGltfFile(const char* path, HostScene& scene, std::string& err);

	// Every count that sizes an allocation is bounded first, but a bounded scene can still need more host memory than there is: that is
	// an error code, not an exception crossing the C ABI.
	int LoadGltf(const char* path, HostScene& scene, std::string& err)
	{
		try { return LoadGltfFile(path, scene, err); }
		catch (const std::bad_alloc&) { scene = HostScene(); err = "the scene needs more host memory than is available"; return SAILOR_PT_ERR_LIMIT; }
		catch (const std::length_error&) { scene = HostScene(); err = "the scene needs more host memory than is available"; return SAILOR_PT_ERR_LIMIT; }
	}

	static int LoadGltfFile(const char* path, HostScene& scene, std::string& err)
	{
		MappedFile file;
		const std::string p = path;
		if (!file.Open(p)) { err = "cannot open " + p; return SAILOR_PT_ERR_IO; }
		Gltf g;
		const size_t slash = p.find_last_of("/\\");
		g.baseDir = slash == std::string::npos ? "" : p.substr(0, slash + 1);

		const uint8_t* json = file.data(); size_t jsonLen = file.size();
		const uint8_t* bin = nullptr; size_t binLen = 0;
		if (file.size() >= 12 && !memcmp(file.data(), "glTF", 4))
		{
			uint32_t version, total; memcpy(&version, file.data() + 4, 4); memcpy(&total, file.data() + 8, 4);
			if (version != 2 || total > file.size()) { err = "unsupported GLB container"; return SAILOR_PT_ERR_FORMAT; }
			size_t off = 12; json = nullptr;
			while (off + 8 <= total)
			{
				uint32_t len, type; memcpy(&len, file.data() + off, 4); memcpy(&type, file.data() + off + 4, 4);
				if (off + 8 + len > total) break;
				if (type == 0x4E4F534Au && !json) { json = file.data() + off + 8; jsonLen = len; }
				else if (type == 0x004E4942u && !bin) { bin = file.data() + off + 8; binLen = len; }
				off += 8 + ((len + 3) & ~3u);
			}
			if (!json) { err = "GLB without JSON chunk"; return SAILOR_PT_ERR_FORMAT; }
		}
		JsonParser jp{ (const char*)json, (const char*)json + jsonLen, {} };
		if (!jp.value(g.root, 0) || g.root.type != Json::Object) { err = "json: " + (jp.err.empty() ? std::string("not an object") : jp.err); return SAILOR_PT_ERR_FORMAT; }

		const Json& jbufs = g.root.at("buffers");
		g.buffers.resize(jbufs.size());
		for (size_t i = 0; i < jbufs.size(); i++)
		{
			const Json* uri = jbufs.at(i).find("uri");
			if (uri && uri->type == Json::String)
			{
				if (!LoadUri(uri->str, g.baseDir, g.buffers[i].own)) { err = "cannot load buffer " + std::to_string(i); return SAILOR_PT_ERR_IO; }
				g.buffers[i].p = g.buffers[i].own.data(); g.buffers[i].n = g.buffers[i].own.size();
			}
			else if (i == 0 && bin) { g.buffers[i].p = bin; g.buffers[i].n = binLen; }       // no copy: the file stays mapped while the scene is imported
			else { err = "buffer without data"; return SAILOR_PT_ERR_FORMAT; }
		}

		// Structural checks the reference's importer makes on the whole document, whether or not a scene node reaches the object
		// (tinygltf's parse rejects these files outright; External/tinygltf/models/BoundsChecking/*.gltf are its regression inputs):
		// a bufferView's byteLength is a positive integer; a primitive's index accessor, that accessor's bufferView and an image's bufferView
		// (and that view's buffer) exist.
		{
			const Json& views = g.root.at("bufferViews"); const Json& accs = g.root.at("accessors"); const Json& imgs = g.root.at("images");
			for (size_t i = 0; i < views.size(); i++)
			{
				const Json* len = views.at(i).find("byteLength");
				if (!len || len->type != Json::Number || !(len->num >= 1.0) || !(len->num <= 9007199254740992.0) || len->num != (double)(uint64_t)len->num)
				{ err = "bufferView[" + std::to_string(i) + "]: 'byteLength' is not a positive integer"; return SAILOR_PT_ERR_FORMAT; }
			}
			const Json& meshes = g.root.at("meshes");
			for (size_t m = 0; m < meshes.size(); m++)
			{
				const Json& prims = meshes.at(m).at("primitives");
				for (size_t k = 0; k < prims.size(); k++)
				{
					const Json* idx = prims.at(k).find("indices");
					if (idx && (idx->type != Json::Number || idx->num < 0.0 || idx->num >= (double)accs.size())) { err = "mesh[" + std::to_string(m) + "]: primitive indices accessor out of bounds"; return SAILOR_PT_ERR_FORMAT; }
					// ... and that accessor's bufferView must exist (attribute accessors are NOT checked by the reference's importer: a primitive
					// whose POSITION cannot be read is dropped by the flattener instead)
					if (idx)
					{
						const Json* bv = accs.at((size_t)idx->num).find("bufferView");
						if (bv && bv->type == Json::Number && bv->num >= (double)views.size()) { err = "accessor[" + std::to_string((size_t)idx->num) + "]: invalid bufferView"; return SAILOR_PT_ERR_FORMAT; }
					}
				}
			}
			for (size_t i = 0; i < imgs.size(); i++)
			{
				const Json* bv = imgs.at(i).find("bufferView");
				if (!bv) continue;
				if (bv->type != Json::Number || bv->num < 0.0 || bv->num >= (double)views.size()) { err = "image[" + std::to_string(i) + "]: invalid bufferView"; return SAILOR_PT_ERR_FORMAT; }
				const double bi = views.at((size_t)bv->num).at("buffer").number(-1.0);
				if (bi < 0.0 || bi >= (double)g.buffers.size()) { err = "image[" + std::to_string(i) + "]: buffer not found"; return SAILOR_PT_ERR_FORMAT; }
			}
		}

		const Json& jmats = g.root.at("materials");
		if (jmats.size() > 256) { err = "more than 256 materials"; return SAILOR_PT_ERR_LIMIT; }

		// cameras (PathTracer.cpp:111-148; Assimp: hFov = 2 atan(tan(yfov/2) * aspect))
		const Json& jcams = g.root.at("cameras");
		scene.cameras.resize(jcams.size());
		for (size_t i = 0; i < jcams.size(); i++)
		{
			HostCamera& c = scene.cameras[i];
			c.name = jcams.at(i).at("name").str;
			for (int k = 0; k < 16; k++) c.matrix[k] = (k % 5 == 0) ? 1.0f : 0.0f;
			if (jcams.at(i).at("type").str == "perspective")
			{
				const Json& pj = jcams.at(i).at("perspective");
				c.aspect = (float)pj.at("aspectRatio").number(0.0);
				const float yfov = (float)pj.at("yfov").number(0.0);
				c.hFov = 2.0f * std::atan(std::tan(yfov * 0.5f) * ((c.aspect == 0.0f) ? 1.0f : c.aspect));
			}
		}

		const Json* klights = g.root.at("extensions").find("KHR_lights_punctual");
		const Json& jlights = klights ? klights->at("lights") : Json();
		const size_t numLights = jlights.size();

		Builder b{ g, scene };
		b.cameraSeen.assign(scene.cameras.size(), 0);
		b.lightSeen.assign(numLights, 0);
		b.lightMatrix.assign(numLights, std::vector<float>{ 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1 });
		const float identity[16] = { 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1 };
		const int sceneIndex = g.root.at("scene").integer(0);
		const Json& roots = g.root.at("scenes").at(sceneIndex >= 0 ? sceneIndex : 0).at("nodes");
		for (size_t i = 0; i < roots.size(); i++) b.Node(roots.at(i).integer(-1), identity, 0);
		if (b.rc != SAILOR_PT_OK) { err = b.err; return b.rc; }
		for (size_t i = 0; i < scene.cameras.size(); i++) if (!b.cameraSeen[i]) scene.cameras[i].name.clear();

		// images are decoded lazily, once per texture slot
		const Json& jtex = g.root.at("textures");
		const Json& jimg = g.root.at("images");
		const Json& jsamp = g.root.at("samplers");
		auto clampingOf = [&](int tex) -> uint32_t
			{
				const int s = jtex.at(tex).at("sampler").integer(-1);
				if (s < 0 || (size_t)s >= jsamp.size()) return kRepeat;
				return jsamp.at(s).at("wrapS").integer(10497) == 10497 ? kRepeat : kClamp;
			};
		auto decodeImage = [&](int image, HostTexture& t) -> bool
			{
				if (image < 0 || (size_t)image >= jimg.size()) return false;
				const Json& im = jimg.at(image);
				std::vector<uint8_t> bytes;
				const int bv = im.at("bufferView").integer(-1);
				if (bv >= 0)
				{
					const Json& view = g.root.at("bufferViews").at(bv);
					const int bi = view.at("buffer").integer(-1);
					const size_t off = (size_t)view.at("byteOffset").number(0), len = (size_t)view.at("byteLength").number(0);
					if (bi < 0 || (size_t)bi >= g.buffers.size() || off + len > g.buffers[bi].size()) return false;
					bytes.assign(g.buffers[bi].begin() + off, g.buffers[bi].begin() + off + len);
				}
				else if (im.at("uri").type == Json::String) { if (!LoadUri(im.at("uri").str, g.baseDir, bytes)) return false; }
				else return false;
				std::string perr;
				if (IsHdr(bytes.data(), bytes.size())) return DecodeHdrRgba32F(bytes.data(), bytes.size(), t.width, t.height, t.rgbaF, perr) == SAILOR_PT_OK;   // stbi_is_hdr_from_memory branch (MaterialUtils.h:224-229)
				return DecodeImageRgba8(bytes.data(), bytes.size(), t.width, t.height, t.rgba, perr) == SAILOR_PT_OK;
			};

		// materials + textures (PathTracer.cpp:164-360)
		struct PendingImage { int image; uint32_t slot; };
		std::vector<PendingImage> pendingImages;
		struct Key { uint32_t slot; };
		std::map<int, uint32_t> textureMapping; // "file" (= image index) -> slot, overwritten like m_textureMapping[file] = ...
		// the glTF default material (an empty material object: baseColor 1, metallic 1, roughness 1, opaque) follows the file's own
		const size_t numMaterials = jmats.size() + (b.needDefault ? 1u : 0u);
		if (numMaterials > 256) { err = "more than 256 materials (with the default material)"; return SAILOR_PT_ERR_LIMIT; }
		const Json defaultMaterial;
		scene.materials.resize(numMaterials);
		bool limit = false, badImage = false;
		for (size_t i = 0; i < numMaterials; i++)
		{
			const Json& jm = i < jmats.size() ? jmats.at(i) : defaultMaterial;
			MaterialGpu& m = scene.materials[i];
			memset(&m, 0, sizeof(m));
			m.uvTransform[0] = 1; m.uvTransform[5] = 1; m.uvTransform[10] = 1;       // mat3(1)
			m.texBase = m.texNormal = m.texMetallicRoughness = m.texEmissive = m.texTransmission = kNoTexture;
			const std::string& alphaMode = jm.at("alphaMode").str;
			m.blendMode = alphaMode == "BLEND" ? kBlend : (alphaMode == "MASK" ? kMask : kOpaque);
			m.alphaCutoff = (float)jm.at("alphaCutoff").number(0.5);
			const Json& ext = jm.at("extensions");
			m.ior = 1.5f;
			if (const Json* e = ext.find("KHR_materials_ior")) m.ior = ExtNumber(*e, "ior", 1.5f);

			auto bind = [&](const Json& texInfo, uint32_t channels, uint32_t& slotOut, bool srgb, bool normalMap, bool checkKey)
				{
					const int ti = texInfo.at("index").integer(-1);
					if (ti < 0 || (size_t)ti >= jtex.size()) return;
					const int image = jtex.at(ti).at("source").integer(-1);
					const uint32_t clamping = clampingOf(ti);
					auto it = textureMapping.find(image);
					if (it != textureMapping.end() && (!checkKey || (scene.textures[it->second].clamping == clamping && scene.textures[it->second].channels == channels)))
					{
						slotOut = it->second;
						return;
					}
					if (scene.textures.size() >= 255) { limit = true; return; }
					HostTexture t;
					t.channels = channels; t.clamping = clamping; t.srgb = srgb; t.normalMap = normalMap;
					slotOut = (uint32_t)scene.textures.size();
					pendingImages.push_back(PendingImage{ image, slotOut });      // decoded after the material loop, on several threads
					textureMapping[image] = slotOut;
					scene.textures.push_back(std::move(t));
				};
			const Json& pbr = jm.at("pbrMetallicRoughness");
			bind(pbr.at("baseColorTexture"), 4, m.texBase, true, false, true);
			bind(jm.at("normalTexture"), 3, m.texNormal, false, true, true);
			bind(pbr.at("metallicRoughnessTexture"), 3, m.texMetallicRoughness, false, false, true);
			bind(jm.at("emissiveTexture"), 3, m.texEmissive, true, false, true);
			if (const Json* e = ext.find("KHR_materials_transmission"))
			{
				m.transmission = ExtNumber(*e, "transmissionFactor", 0.0f);
				if (e->find("transmissionTexture")) bind(e->at("transmissionTexture"), 3, m.texTransmission, false, false, false);
			}
			const Json& ef = jm.at("emissiveFactor");
			float strength = 1.0f;
			if (const Json* e = ext.find("KHR_materials_emissive_strength")) strength = ExtNumber(*e, "emissiveStrength", 1.0f);
			for (int k = 0; k < 3; k++) m.emissive[k] = (ef.size() == 3 ? (float)ef.at(k).num : 0.0f) * strength;
			const Json& bc = pbr.at("baseColorFactor");
			for (int k = 0; k < 4; k++) m.baseColor[k] = bc.size() == 4 ? (float)bc.at(k).num : 1.0f;
			m.roughness = (float)pbr.at("roughnessFactor").number(1.0);
			m.metallic = (float)pbr.at("metallicFactor").number(1.0);
			m.thickness = 0.0f; m.attenuationDistance = std::numeric_limits<float>::max();
			m.attenuationColor[0] = m.attenuationColor[1] = m.attenuationColor[2] = 1.0f;
			if (const Json* e = ext.find("KHR_materials_volume"))
			{
				m.thickness = ExtNumber(*e, "thicknessFactor", 0.0f);
				m.attenuationDistance = ExtNumber(*e, "attenuationDistance", std::numeric_limits<float>::max());
				const Json& ac = e->at("attenuationColor");
				if (ac.size() == 3) for (int k = 0; k < 3; k++) m.attenuationColor[k] = (float)ac.at(k).num;
			}
			if (const Json* e = pbr.at("baseColorTexture").at("extensions").find("KHR_texture_transform"))
			{
				float offX = 0, offY = 0, scX = 1, scY = 1;
				const float rot = ExtNumber(*e, "rotation", 0.0f);
				if (e->at("offset").size() == 2) { offX = (float)e->at("offset").at((size_t)0).num; offY = (float)e->at("offset").at((size_t)1).num; }
				if (e->at("scale").size() == 2) { scX = (float)e->at("scale").at((size_t)0).num; scY = (float)e->at("scale").at((size_t)1).num; }
				// translation * rotation * scale with glm's mat3 product order (type_mat3x3.inl:486-520), columns of 3
				const float S[9] = { scX, 0, 0, 0, scY, 0, 0, 0, 1 };
				const float Tm[9] = { 1, 0, 0, 0, 1, 0, offX, offY, 1 };
				const float c = std::cos(rot), s = std::sin(rot);
				const float Rm[9] = { c, -s, 0, s, c, 0, 0, 0, 1 };
				auto mul3 = [](const float* A, const float* B, float* R)
					{
						float tmp[9];
						for (int col = 0; col < 3; col++) for (int r = 0; r < 3; r++)
							tmp[col * 3 + r] = A[0 * 3 + r] * B[col * 3 + 0] + A[1 * 3 + r] * B[col * 3 + 1] + A[2 * 3 + r] * B[col * 3 + 2];
						memcpy(R, tmp, sizeof(tmp));
					};
				float TR[9], TRS[9];
				mul3(Tm, Rm, TR); mul3(TR, S, TRS);
				for (int col = 0; col < 3; col++) for (int r = 0; r < 3; r++) m.uvTransform[col * 4 + r] = TRS[col * 3 + r];
			}
		}
		if (limit) { err = "more than 255 textures"; return SAILOR_PT_ERR_LIMIT; }
		// Decode the images on several host threads: inflating a 1024x1024 PNG takes ~30 ms, and a scene like BASELINE's C4 binds 224 of
		// them (6.7 s one after the other).  The reference loads its textures as parallel tasks too (LoadTexture_Task, MaterialUtils.h:189-269).
		if (!pendingImages.empty())
		{
			std::atomic<size_t> next{ 0 };
			std::atomic<bool> failed{ false };
			auto worker = [&]()
				{
					for (;;)
					{
						const size_t k = next.fetch_add(1);
						if (k >= pendingImages.size()) break;
						if (!decodeImage(pendingImages[k].image, scene.textures[pendingImages[k].slot])) failed = true;
					}
				};
			unsigned hw = std::thread::hardware_concurrency(); if (hw == 0) hw = 4; if (hw > 32) hw = 32;
			const size_t nThreads = pendingImages.size() < hw ? pendingImages.size() : hw;
			std::vector<std::thread> pool;
			for (size_t t = 1; t < nThreads; t++) pool.emplace_back(worker);
			worker();
			for (auto& t : pool) t.join();
			if (failed) badImage = true;
		}
		if (badImage) { err = "an image could not be decoded (PNG and JPEG are supported)"; return SAILOR_PT_ERR_FORMAT; }

		// directional lights (PathTracer.cpp:362-381)
		for (size_t i = 0; i < numLights; i++)
		{
			const Json& L = jlights.at(i);
			if (L.at("type").str != "directional") continue;
			HostLight hl;
			float color[3] = { 1, 1, 1 };
			if (L.at("color").size() == 3) for (int k = 0; k < 3; k++) color[k] = (float)L.at("color").at(k).num;
			const float intensity = (float)L.at("intensity").number(1.0);
			const float* M = b.lightMatrix[i].data();
			// vec3(vec4(0,0,-1,0) * M): component j = M[j][0]*0 + M[j][1]*0 + M[j][2]*(-1) + M[j][3]*0 (type_mat4x4.inl:586-595)
			float d[3];
			for (int j = 0; j < 3; j++) d[j] = M[j * 4 + 0] * 0.0f + M[j * 4 + 1] * 0.0f + M[j * 4 + 2] * -1.0f + M[j * 4 + 3] * 0.0f;
			const float inv = 1.0f / std::sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
			for (int j = 0; j < 3; j++) { hl.direction[j] = d[j] * inv; hl.intensity[j] = (color[j] * intensity) / 683.0f; }
			scene.lights.push_back(hl);
		}
		return SAILOR_PT_OK;
	}

	// ---------------------------------------------------------------------------------------------- camera
	namespace
	{
		struct F3 { float x, y, z; };
		F3 f3(float x, float y, float z) { return F3{ x, y, z }; }
		F3 add(F3 a, F3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
		F3 sub(F3 a, F3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
		F3 mul(F3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
		F3 smul(float s, F3 a) { return f3(s * a.x, s * a.y, s * a.z); }
		F3 divs(F3 a, float s) { return f3(a.x / s, a.y / s, a.z / s); }
		F3 neg(F3 a) { return f3(-a.x, -a.y, -a.z); }
		float dot3(F3 a, F3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
		F3 cross3(F3 x, F3 y) { return f3(x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y); }
		F3 norm3(F3 v) { return mul(v, 1.0f / std::sqrt(dot3(v, v))); }
		// vec3(vec4(v, w) * M) in glm's order (type_mat4x4.inl:586-595)
		void rowMul(const float* M, float x, float y, float z, float w, float out[4])
		{
			for (int j = 0; j < 4; j++) out[j] = M[j * 4 + 0] * x + M[j * 4 + 1] * y + M[j * 4 + 2] * z + M[j * 4 + 3] * w;
		}
	}

	CameraSetup SetupCamera(const HostScene& scene, const SailorPtParamsView& p)
	{
		F3 cameraPos = f3(0, 0.75f, 5.0f);                                         // PathTracer.cpp:102-109
		F3 cameraUp = norm3(f3(0, 1, 0));
		F3 cameraForward = norm3(neg(cameraPos));
		const F3 axis = norm3(cross3(cameraForward, cameraUp));
		cameraUp = norm3(cross3(axis, cameraForward));

		const bool hasCameras = !scene.cameras.empty();
		size_t cameraIndex = 0;
		if (hasCameras)                                                            // :111-135
		{
			const char* want = p.camera ? p.camera : "";
			for (size_t i = 0; i < scene.cameras.size(); i++) if (scene.cameras[i].name == want) { cameraIndex = i; break; }
			const float* M = scene.cameras[cameraIndex].matrix;
			float t[4], u[4], f[4];
			rowMul(M, 0.0f, 0.0f, 0.0f, 1.0f, t);
			cameraPos = divs(f3(t[0], t[1], t[2]), t[3]);
			rowMul(M, 0.0f, 1.0f, 0.0f, 0.0f, u);
			cameraUp = norm3(f3(u[0], u[1], u[2]));
			rowMul(M, 0.0f, 0.0f, -1.0f, 0.0f, f);
			cameraForward = norm3(f3(f[0], f[1], f[2]));
		}
		float aspectRatio = (hasCameras && scene.cameras[cameraIndex].aspect > 0.0f) ? scene.cameras[cameraIndex].aspect : (4.0f / 3.0f);
		const uint32_t height = p.height;
		uint32_t width = static_cast<uint32_t>(height * aspectRatio);              // :141-142
		if (p.widthOverride) { width = p.widthOverride; aspectRatio = (float)width / (float)height; }
		const float hFov = (hasCameras && scene.cameras[cameraIndex].hFov > 0.0f) ? scene.cameras[cameraIndex].hFov : (60.0f * 0.01745329251994329576923690768489f);
		const float vFov = 2.0f * std::atan(std::tan(hFov * 0.5f) * (1.0f / aspectRatio)); // :148

		const float h = std::tan(vFov / 2);                                        // :390-403
		const float viewportHeight = 2.0f * h;
		const float viewportWidth = aspectRatio * viewportHeight;
		const F3 _u = norm3(cross3(cameraUp, neg(cameraForward)));
		const F3 _v = cross3(neg(cameraForward), _u);
		const F3 viewportU = smul(viewportWidth, _u);
		const F3 viewportV = smul(viewportHeight, _v);
		const F3 pivot = add(sub(cameraPos, mul(add(viewportU, viewportV), 0.5f)), cameraForward);
		const F3 dU = divs(viewportU, (float)width);
		const F3 dV = divs(viewportV, (float)height);
		const F3 p00 = sub(add(pivot, smul(0.5f, add(dU, dV))), cameraPos);

		CameraSetup c;
		c.width = width; c.height = height;
		c.pos[0] = cameraPos.x; c.pos[1] = cameraPos.y; c.pos[2] = cameraPos.z;
		c.pixel00Dir[0] = p00.x; c.pixel00Dir[1] = p00.y; c.pixel00Dir[2] = p00.z;
		c.deltaU[0] = dU.x; c.deltaU[1] = dU.y; c.deltaU[2] = dU.z;
		c.deltaV[0] = dV.x; c.deltaV[1] = dV.y; c.deltaV[2] = dV.z;
		return c;
	}
}
