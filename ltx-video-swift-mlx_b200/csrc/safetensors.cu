// Checkpoint ingestion: reads a .safetensors file and feeds the tensors of the hot path to the context under the
// reference's post-mapping key names, so a real LTX-2 checkpoint loads straight into libltxcuda.
//
// Restates (does not share code with) the reference loader:
//   LTXWeightLoader.loadTransformerWeights   Utils/ModelDownloader.swift:605-639  (prefix filter, audio / connector skip)
//   mapTransformerKey                        Utils/ModelDownloader.swift:756-803
//   loadVAEWeights + mapVAEWeights           Utils/ModelDownloader.swift:649-659, 808-899
// File format (safetensors): u64 little-endian header length, a flat JSON object {name: {"dtype", "shape", "data_offsets"}}
// (+ "__metadata__"), then the raw little-endian tensor bytes.  The file is mmap'ed; each selected tensor goes through
// load_tensor_host (H2D copy + the fp32 -> bf16 cast of :1005-1012 on the device).
//
// Scaled-FP8 transformer files (the convention the reference's ".weight_scale" / ".input_scale" filter implies, :617-629; no
// such file was at hand, so anything else is refused rather than guessed at): a Linear weight "X.weight" in F8_E4M3 (e4m3fn)
// of shape [N, K] with "X.weight_scale" beside it, F32 or BF16 of shape [] / [1] (per tensor) or [N] / [N, 1] (per output
// channel), finite and > 0: w[n][k] = e4m3(code) * scale.  "X.input_scale" is ignored: FP8 mode quantises the activation rows
// at run time.  Those go through load_tensor_e4m3_host.
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cmath>
#include <cstring>

#include "ctx.h"

namespace ltx {

namespace {

bool starts_with(const std::string& s, const char* p) { return s.compare(0, strlen(p), p) == 0; }
bool ends_with(const std::string& s, const char* p) {
  const size_t n = strlen(p);
  return s.size() >= n && s.compare(s.size() - n, n, p) == 0;
}
bool contains(const std::string& s, const char* p) { return s.find(p) != std::string::npos; }
void replace_all(std::string& s, const std::string& from, const std::string& to) {
  size_t pos = 0;
  while ((pos = s.find(from, pos)) != std::string::npos) {
    s.replace(pos, from.size(), to);
    pos += to.size();
  }
}

// ---------------------------------------------------------------- minimal JSON reader for the safetensors header
struct TensorInfo {
  std::string dtype;
  std::vector<int64_t> shape;
  uint64_t begin = 0, end = 0;
};

struct Json {
  const char* p;
  const char* e;
  void ws() { while (p < e && (*p == ' ' || *p == '\n' || *p == '\t' || *p == '\r')) ++p; }
  void expect(char c) {
    ws();
    LTX_CHECK(p < e && *p == c, LTX_ERR_WEIGHTS, std::string("safetensors header: expected '") + c + "'");
    ++p;
  }
  bool peek(char c) { ws(); return p < e && *p == c; }
  std::string str() {
    expect('"');
    std::string out;
    while (p < e && *p != '"') {
      if (*p == '\\' && p + 1 < e) {
        ++p;
        switch (*p) {
          case 'n': out += '\n'; break;
          case 't': out += '\t'; break;
          case 'r': out += '\r'; break;
          case 'b': out += '\b'; break;
          case 'f': out += '\f'; break;
          case 'u': {  // \uXXXX: keep ASCII, replace the rest (tensor names are ASCII)
            LTX_CHECK(p + 4 < e, LTX_ERR_WEIGHTS, "safetensors header: bad \\u escape");
            unsigned v = 0;
            for (int i = 1; i <= 4; ++i) {
              const char ch = p[i];
              v = v * 16 + (ch >= '0' && ch <= '9' ? ch - '0' : (ch | 32) >= 'a' && (ch | 32) <= 'f' ? (ch | 32) - 'a' + 10 : 0);
            }
            out += v < 128 ? static_cast<char>(v) : '?';
            p += 4;
            break;
          }
          default: out += *p;
        }
        ++p;
      } else {
        out += *p++;
      }
    }
    LTX_CHECK(p < e, LTX_ERR_WEIGHTS, "safetensors header: unterminated string");
    ++p;
    return out;
  }
  int64_t integer() {
    ws();
    bool neg = false;
    if (p < e && *p == '-') { neg = true; ++p; }
    LTX_CHECK(p < e && *p >= '0' && *p <= '9', LTX_ERR_WEIGHTS, "safetensors header: expected an integer");
    int64_t v = 0;
    while (p < e && *p >= '0' && *p <= '9') v = v * 10 + (*p++ - '0');
    return neg ? -v : v;
  }
  void skip_value() {   // strings / numbers / nested containers of "__metadata__"
    ws();
    LTX_CHECK(p < e, LTX_ERR_WEIGHTS, "safetensors header: truncated");
    if (*p == '"') { str(); return; }
    if (*p == '{' || *p == '[') {
      const char open = *p, close = open == '{' ? '}' : ']';
      ++p;
      if (peek(close)) { ++p; return; }
      for (;;) {
        if (open == '{') { str(); expect(':'); }
        skip_value();
        if (peek(',')) { ++p; continue; }
        expect(close);
        return;
      }
    }
    while (p < e && *p != ',' && *p != '}' && *p != ']') ++p;   // number / true / false / null
  }
};

std::map<std::string, TensorInfo> parse_header(const char* json, size_t n) {
  std::map<std::string, TensorInfo> out;
  Json j{json, json + n};
  j.expect('{');
  if (j.peek('}')) return out;
  for (;;) {
    const std::string name = j.str();
    j.expect(':');
    if (name == "__metadata__") {
      j.skip_value();
    } else {
      TensorInfo t;
      j.expect('{');
      for (;;) {
        const std::string k = j.str();
        j.expect(':');
        if (k == "dtype") {
          t.dtype = j.str();
        } else if (k == "shape") {
          j.expect('[');
          if (!j.peek(']'))
            for (;;) { t.shape.push_back(j.integer()); if (j.peek(',')) { ++j.p; continue; } break; }
          j.expect(']');
        } else if (k == "data_offsets") {
          j.expect('[');
          { const int64_t v = j.integer(); LTX_CHECK(v >= 0, LTX_ERR_WEIGHTS, "safetensors header: negative data offset"); t.begin = static_cast<uint64_t>(v); }
          j.expect(',');
          { const int64_t v = j.integer(); LTX_CHECK(v >= 0, LTX_ERR_WEIGHTS, "safetensors header: negative data offset"); t.end = static_cast<uint64_t>(v); }
          j.expect(']');
        } else {
          j.skip_value();
        }
        if (j.peek(',')) { ++j.p; continue; }
        break;
      }
      j.expect('}');
      out[name] = t;
    }
    if (j.peek(',')) { ++j.p; continue; }
    break;
  }
  j.expect('}');
  return out;
}

struct MappedFile {
  int fd = -1;
  const uint8_t* base = nullptr;
  size_t size = 0;
  explicit MappedFile(const char* path) {
    fd = open(path, O_RDONLY);
    LTX_CHECK(fd >= 0, LTX_ERR_WEIGHTS, std::string("cannot open '") + path + "'");
    struct stat st;
    LTX_CHECK(fstat(fd, &st) == 0 && st.st_size >= 8, LTX_ERR_WEIGHTS, std::string("'") + path + "' is not a safetensors file");
    size = static_cast<size_t>(st.st_size);
    void* m = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
    LTX_CHECK(m != MAP_FAILED, LTX_ERR_WEIGHTS, std::string("mmap failed for '") + path + "'");
    base = static_cast<const uint8_t*>(m);
  }
  ~MappedFile() {
    if (base) munmap(const_cast<uint8_t*>(base), size);
    if (fd >= 0) close(fd);
  }
};

// The header is untrusted input: bound the rank, reject negative dims and an element count that overflows, and only then
// compare the byte count with the data offsets.  Returns the element count.
uint64_t checked_numel(const std::string& key, const TensorInfo& t, size_t esz, uint64_t data_size) {
  LTX_CHECK(t.shape.size() <= 8, LTX_ERR_WEIGHTS, "tensor '" + key + "': more than 8 dimensions");
  LTX_CHECK(t.begin <= t.end && t.end <= data_size, LTX_ERR_WEIGHTS, "tensor '" + key + "': data_offsets outside the file");
  const uint64_t span = t.end - t.begin;
  uint64_t n_u = 1;
  for (int64_t d : t.shape) {
    LTX_CHECK(d >= 0, LTX_ERR_WEIGHTS, "tensor '" + key + "': negative dimension");
    LTX_CHECK(d == 0 || n_u <= UINT64_MAX / static_cast<uint64_t>(d), LTX_ERR_WEIGHTS, "tensor '" + key + "': element count overflows");
    n_u *= static_cast<uint64_t>(d);
  }
  LTX_CHECK(n_u <= span / esz && n_u * esz == span, LTX_ERR_WEIGHTS, "tensor '" + key + "': data_offsets do not match its shape");
  return n_u;
}

}  // namespace

// Transformer key of the checkpoint -> name the context expects, or "" when the tensor is not part of the video-only DiT.
// `key` is the name inside the file (with or without the "model.diffusion_model." prefix of the unified checkpoint).
std::string map_transformer_key(const std::string& file_key, bool include_audio) {
  std::string key = file_key;
  // loadTransformerWeights (:617-629): quantisation side tensors, audio / vocoder / cross-modal tensors, connectors
  if (ends_with(key, ".weight_scale") || ends_with(key, ".input_scale")) return "";
  if (!include_audio && (contains(key, "audio") || starts_with(key, "vocoder") || contains(key, "av_ca_"))) return "";
  if (include_audio && starts_with(key, "vocoder")) return "";   // not under model.diffusion_model. (:624)
  static const char* kPrefix = "model.diffusion_model.";
  if (starts_with(key, kPrefix)) key = key.substr(strlen(kPrefix));
  if (starts_with(key, "video_embeddings_connector.") || starts_with(key, "audio_embeddings_connector.")) return "";
  // mapTransformerKey (:760-771): audio / cross-modal tensors of the dual model
  if (!include_audio && (starts_with(key, "audio_") || contains(key, ".audio_") || starts_with(key, "av_cross_attn_") ||
      contains(key, "video_to_audio") || contains(key, "video_a2v") || contains(key, "a2v_ca") ||
      contains(key, "scale_shift_table_a2v")))
    return "";
  std::string k = key;
  if (starts_with(k, "proj_in.")) k = "patchify_proj." + k.substr(strlen("proj_in."));                       // :776-778
  if (starts_with(k, "time_embed.emb.timestep_embedder."))                                                    // :781-787
    k = "adaln_single.emb." + k.substr(strlen("time_embed.emb.timestep_embedder."));
  else if (starts_with(k, "time_embed.linear."))
    k = "adaln_single." + k.substr(strlen("time_embed."));
  else if (starts_with(k, "adaln_single.emb.timestep_embedder."))
    k = "adaln_single.emb." + k.substr(strlen("adaln_single.emb.timestep_embedder."));
  replace_all(k, ".emb.timestep_embedder.", ".emb.");                                                         // :791
  replace_all(k, ".norm_q.", ".q_norm.");                                                                     // :794-795
  replace_all(k, ".norm_k.", ".k_norm.");
  replace_all(k, ".to_out.0.", ".to_out.");                                                                   // :798
  replace_all(k, "ff.net.0.proj.", "ff.project_in.proj.");                                                    // :802-803
  replace_all(k, "ff.net.2.", "ff.project_out.");
  return k;
}

// VAE key of the checkpoint -> context name ("vae." + Swift module path), or "" for encoder tensors.
std::string map_vae_key(const std::string& file_key) {
  std::string key = file_key;
  if (starts_with(key, "vae.")) key = key.substr(4);                      // unified checkpoint
  if (starts_with(key, "encoder.")) return "";                            // :818
  if (contains(key, "per_channel_statistics")) {                          // :821-829
    const std::string base = key.substr(key.rfind('.') + 1);
    if (base == "mean-of-means") return "vae.mean_of_means";
    if (base == "std-of-means") return "vae.std_of_means";
    return "";
  }
  if (key == "latents_mean") return "vae.mean_of_means";                  // :832-839 (squeezed by the caller)
  if (key == "latents_std") return "vae.std_of_means";
  std::string k = key;
  if (starts_with(k, "decoder.")) k = k.substr(strlen("decoder."));      // :844-846
  if (starts_with(k, "mid_block.")) {                                     // :858-860
    k = "up_blocks_0." + k.substr(strlen("mid_block."));
  } else {
    for (int i = 0; i <= 2; ++i) {                                        // :863-876
      const std::string up = "up_blocks." + std::to_string(i) + ".upsamplers.0.";
      const std::string rn = "up_blocks." + std::to_string(i) + ".resnets.";
      if (starts_with(k, up.c_str())) { k = "up_blocks_" + std::to_string(2 * i + 1) + "." + k.substr(up.size()); break; }
      if (starts_with(k, rn.c_str())) { k = "up_blocks_" + std::to_string(2 * i + 2) + ".resnets." + k.substr(rn.size()); break; }
    }
  }
  for (int i = 0; i <= 6; ++i) {                                          // :879-885 legacy "up_blocks.{i}."
    const std::string src = "up_blocks." + std::to_string(i) + ".";
    if (starts_with(k, src.c_str())) { k = "up_blocks_" + std::to_string(i) + "." + k.substr(src.size()); break; }
  }
  replace_all(k, ".resnets.", ".res_blocks.");                            // :888
  return "vae." + k;
}

// VAE-encoder key of the checkpoint -> "vae_encoder." + Swift module path (mapVAEEncoderWeights, U/ModelDownloader.swift:1224-1280),
// or "" for everything that is not an "encoder." tensor.
std::string map_vae_encoder_key(const std::string& file_key) {
  std::string key = file_key;
  if (starts_with(key, "vae.")) key = key.substr(4);
  if (!starts_with(key, "encoder.")) return "";                           // :1233
  std::string k = key.substr(strlen("encoder."));
  for (int i = 0; i <= 3; ++i) {                                          // :1238-1244
    const std::string src = "down_blocks." + std::to_string(i) + ".";
    if (starts_with(k, src.c_str())) { k = "down_blocks_" + std::to_string(i) + "." + k.substr(src.size()); break; }
  }
  for (int i = 0; i <= 3; ++i) {                                          // :1253-1263: EncoderDownBlock.resnets -> group .resnets
    const std::string rp = "down_blocks_" + std::to_string(i) + ".resnets.";
    if (starts_with(k, rp.c_str())) {
      const std::string suffix = k.substr(rp.size());
      if (!starts_with(suffix, "resnets.")) k = rp + "resnets." + suffix;
      break;
    }
  }
  for (int i = 0; i <= 3; ++i) {                                          // :1266-1273
    const std::string dp = "down_blocks_" + std::to_string(i) + ".downsamplers.0.";
    if (starts_with(k, dp.c_str())) { k = "down_blocks_" + std::to_string(i) + ".downsamplers." + k.substr(dp.size()); break; }
  }
  return "vae_encoder." + k;
}

// Upscaler checkpoint key -> "upscaler." + key; the fixed blur kernel is skipped (loadSpatialUpscaler,
// Models/Upscaler/SpatialUpscaler.swift:262-300).  Conv kernels stay in the checkpoint (PyTorch) layout, repacked at finalize.
std::string map_upscaler_key(const std::string& file_key) {
  if (contains(file_key, "blur_down")) return "";
  return "upscaler." + file_key;
}

// LoRAKeyMapper.loraKeyToModelKey (LoRA/LoRALoader.swift:209-243): LoRA layer key (ComfyUI / Diffusers naming) -> the model weight
// it patches, in the context's post-mapping names.
std::string map_lora_key(const std::string& lora_key) {
  std::string k = lora_key;
  if (starts_with(k, "diffusion_model.")) k = k.substr(strlen("diffusion_model."));
  replace_all(k, ".emb.timestep_embedder.", ".emb.");
  replace_all(k, ".to_out.0", ".to_out");
  replace_all(k, ".ff.net.0.proj", ".ff.project_in.proj");
  replace_all(k, ".ff.net.2", ".ff.project_out");
  return k + ".weight";
}

// which: 1 = transformer tensors (mapTransformerKey), 2 = VAE decoder tensors (mapVAEWeights), 3 = VAE encoder tensors
// (mapVAEEncoderWeights), 4 = latent upscaler file.  Returns how many were loaded.
int load_safetensors(ltx_ctx* c, const char* path, int which) {
  LTX_CHECK(path != nullptr && which >= 1 && which <= 5, LTX_ERR_INVALID_ARGUMENT, "load_safetensors: bad arguments");
  MappedFile f(path);
  uint64_t hlen = 0;
  memcpy(&hlen, f.base, 8);
  LTX_CHECK(hlen > 0 && hlen <= f.size - 8, LTX_ERR_WEIGHTS, std::string("'") + path + "': bad safetensors header length");
  const auto header = parse_header(reinterpret_cast<const char*>(f.base + 8), static_cast<size_t>(hlen));
  const uint8_t* data = f.base + 8 + hlen;
  const uint64_t data_size = f.size - 8 - hlen;
  // A unified checkpoint holds every sub-model: there the transformer tensors are exactly the "model.diffusion_model."
  // keys (:624) and the VAE tensors the "vae." keys; a stand-alone file carries no such prefix and is taken whole.
  const char* want = (which == 1 || which == 5) ? "model.diffusion_model." : "vae.";
  bool unified = false;
  if (which != 4)
    for (const auto& kv : header) unified = unified || starts_with(kv.first, want);
  const bool transformer = which == 1 || which == 5;
  // Pass 1 validates every tensor the call takes (and pairs each e4m3 weight with its scale) before anything is uploaded, so a
  // refused file loads nothing.
  struct Item {
    std::string name;
    const uint8_t* bytes;
    int dtype;                   // an ltx_dtype, or DT_E4M3: codes of a scaled-FP8 Linear
    std::vector<int64_t> shape;
    std::vector<float> scales;   // DT_E4M3: 1 (per tensor) or shape[0] (per output channel) values, finite and > 0
  };
  std::vector<Item> items;
  for (const auto& kv : header) {
    if (unified && !starts_with(kv.first, want)) continue;
    const std::string name = which == 1   ? map_transformer_key(kv.first)
                             : which == 2 ? map_vae_key(kv.first)
                             : which == 3 ? map_vae_encoder_key(kv.first)
                             : which == 4 ? map_upscaler_key(kv.first)
                                          : map_transformer_key(kv.first, true);
    if (name.empty()) continue;
    const TensorInfo& t = kv.second;
    Item it;
    it.name = name;
    it.dtype = DT_E4M3;
    size_t esz = 1;
    if (t.dtype == "F32") { it.dtype = LTX_F32; esz = 4; }
    else if (t.dtype == "BF16") { it.dtype = LTX_BF16; esz = 2; }
    else if (t.dtype == "F16") { it.dtype = LTX_F16; esz = 2; }
    else LTX_CHECK(t.dtype == "F8_E4M3", LTX_ERR_WEIGHTS, "tensor '" + kv.first + "' has unsupported dtype " + t.dtype);
    const uint64_t n_u = checked_numel(kv.first, t, esz, data_size);
    if (it.dtype == DT_E4M3) {
      // scaled FP8: only the 2-D weight of a transformer Linear, with its weight_scale beside it
      LTX_CHECK(transformer && ends_with(kv.first, ".weight") && t.shape.size() == 2 && n_u > 0, LTX_ERR_WEIGHTS,
                "tensor '" + kv.first + "': F8_E4M3 is only accepted for the 2-D weight of a transformer Linear");
      const std::string skey = kv.first + "_scale";
      const auto s = header.find(skey);
      LTX_CHECK(s != header.end(), LTX_ERR_WEIGHTS, "tensor '" + kv.first + "': F8_E4M3 without '" + skey + "'");
      const TensorInfo& st = s->second;
      LTX_CHECK(st.dtype == "F32" || st.dtype == "BF16", LTX_ERR_WEIGHTS, "'" + skey + "': scale dtype must be F32 or BF16");
      const int64_t N = t.shape[0];
      const std::vector<int64_t>& ss = st.shape;
      const bool per_tensor = ss.empty() || (ss.size() == 1 && ss[0] == 1);
      const bool per_row = (ss.size() == 1 && ss[0] == N) || (ss.size() == 2 && ss[0] == N && ss[1] == 1);
      LTX_CHECK(per_tensor || per_row, LTX_ERR_WEIGHTS, "'" + skey + "': scale shape must be [], [1], [N] or [N, 1]");
      const size_t sesz = st.dtype == "F32" ? 4 : 2;
      const uint64_t ns = checked_numel(skey, st, sesz, data_size);
      const uint8_t* sp = data + st.begin;
      for (uint64_t i = 0; i < ns; ++i) {
        uint32_t u = 0;
        if (sesz == 4) memcpy(&u, sp + 4 * i, 4);
        else { uint16_t h; memcpy(&h, sp + 2 * i, 2); u = static_cast<uint32_t>(h) << 16; }
        float v;
        memcpy(&v, &u, 4);
        LTX_CHECK(std::isfinite(v) && v > 0.f, LTX_ERR_WEIGHTS, "'" + skey + "': every scale must be finite and > 0");
        it.scales.push_back(v);
      }
    }
    if (n_u == 0) continue;   // empty tensor: nothing to load
    const int64_t n = static_cast<int64_t>(n_u);
    it.bytes = data + t.begin;
    it.shape = t.shape;
    if (name == "vae.mean_of_means" || name == "vae.std_of_means") it.shape.assign(1, n);   // .squeezed() (:833, :837)
    if (it.shape.empty()) it.shape.assign(1, 1);                                              // scalars (timestep_scale_multiplier)
    items.push_back(std::move(it));
  }
  // Pass 2 uploads.  The NaN check of e4m3 codes runs on the device during the upload; when it (or anything else) fails, every
  // tensor this call loaded is removed again.
  std::vector<std::string> done;
  try {
    for (const Item& it : items) {
      if (it.dtype == DT_E4M3)
        // the dual audio/video model has no FP8 mode: its tensors are always decoded
        load_tensor_e4m3_host(c, it.name, it.bytes, it.scales.data(), static_cast<int64_t>(it.scales.size()), it.shape.data(),
                              which == 1);
      else
        load_tensor_host(c, it.name, it.bytes, it.dtype, it.shape.data(), static_cast<int>(it.shape.size()));
      done.push_back(it.name);
    }
  } catch (...) {
    cudaStreamSynchronize(c->stream);
    for (const std::string& k : done) {
      auto t = c->tensors.find(k);
      if (t == c->tensors.end()) continue;
      t->second.free_storage();
      c->tensors.erase(t);
    }
    throw;
  }
  return static_cast<int>(items.size());
}

}  // namespace ltx
