// Packed-weight cache (SURVEY.md §8(f)4): the one-time conversion of a voice's generator.onnx into the engine's
// GEMM-ready fp32 slab + 16-bit tensor-core operand slab, written once and re-read on later loads.
//
// Reference side: the file this replaces the parsing of is `voice_dir/"generator.onnx"` (mimic3_tts/voice.py:273),
// loaded once per path per process under _SHARED_MODELS_LOCK (voice.py:277-299); the voice registry
// mimic3_tts/voices.json (read by _resources.py:35-51) lists a sha256_sum for it, which download.py:108-117 compares
// with the file on disk.  The blob records that digest at conversion time, so the manifest check costs a string
// compare on every later load instead of a pass over the 76 MB file.
//
// Blob = [CacheHeader 512 B][meta: serialised DeviceVoice, pointers as slab offsets][fp32 slab][16-bit slab];
// a 64-bit checksum over everything after the header; any mismatch (magic, layout version, pack switches, size /
// mtime of generator.onnx, digest of config.json, checksum, out-of-range offset) means "miss", never an error.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "engine.h"

namespace m3 {

constexpr uint32_t kCacheLayoutVersion = 10;  // bump whenever pack_voice's output or a *W struct changes

struct CacheKey {
  std::string onnx_path, config_path;  // resolved
  uint64_t onnx_size = 0;
  int64_t onnx_mtime_ns = 0;
  std::string config_sha256;  // config.json is small: hashed on every load
  std::string pack_flags;
  std::string file_name() const;  // "<32 hex>.m3w"
};

struct CacheImage {  // a validated blob, still on the host
  std::vector<uint8_t> bytes;
  size_t meta_off = 0, meta_bytes = 0, meta_len = 0, f32_off = 0, f32_count = 0, h16_off = 0, h16_count = 0;
  std::string onnx_sha256;
};

// voice directory or generator.onnx -> the two files a voice is made of (same rule as load_host_voice)
void resolve_voice_paths(const std::string& path, std::string* onnx, std::string* config);
CacheKey make_cache_key(const std::string& path);  // throws "cannot open ..." like the loader
std::string sha256_file(const std::string& path);  // throws "cannot open ..."

// pointers of `dv` must be resolved against `base` (host or device); appends to `out`
void serialize_voice(const DeviceVoice& dv, const float* base, std::vector<uint8_t>& out);
// false on any inconsistency; pointers come out as base + offset, offsets checked against the slab sizes
bool deserialize_voice(DeviceVoice& dv, const float* base, size_t n_f32, size_t n_h16, const uint8_t* p, size_t n);

// Writes atomically (temp file + rename).  `pv.fix` is applied against pv.f32.data() first.
void write_cache_file(const std::string& file, const CacheKey& key, const std::string& onnx_sha256, PackedVoice& pv);
// Empty pointer = miss (absent, stale or damaged); `why` says which.
std::unique_ptr<CacheImage> read_cache_file(const std::string& file, const CacheKey* key, std::string* why);
std::unique_ptr<DeviceVoice> upload_cached(const CacheImage& img, int device);

}  // namespace m3
