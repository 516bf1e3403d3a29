// extern "C" surface of libltxcuda.so (include/ltxcuda.h).  Every entry point catches C++ exceptions and maps
// them to the integer status + ltx_last_error() contract.
#include <cstring>

#include "ctx.h"

using namespace ltx;

namespace {

thread_local std::string g_create_error;

template <typename Fn>
int guarded(ltx_ctx* c, Fn&& fn) {
  if (!c) return LTX_ERR_INVALID_ARGUMENT;
  try {
    LTX_CUDA(cudaSetDevice(c->device));
    fn();
    return LTX_OK;
  } catch (const LtxError& e) {
    c->last_error = e.what();
    return e.code;
  } catch (const std::exception& e) {
    c->last_error = e.what();
    return LTX_ERR_CUDA;
  }
}

size_t dsize(int dt) { return dt == LTX_F32 ? 4 : 2; }

void h2d(ltx_ctx* c, DevBuf& buf, const void* host, size_t bytes) {
  buf.reserve(bytes);
  LTX_CUDA(cudaMemcpyAsync(buf.ptr, host, bytes, cudaMemcpyHostToDevice, c->stream));
}

// A context_key promises "same text as last time under this key".  The host-buffer entry points can check that promise
// cheaply: a sampled 64-bit hash of the embedding (512 strided 8-byte words + both ends) and of the whole mask is recorded
// with the cache entry; a later call whose buffers hash differently under the same key rebuilds the entry instead of silently
// reusing another prompt's K / V (the device-pointer entry points cannot look at their inputs and trust the key).
uint64_t fnv1a(uint64_t h, const void* data, size_t n) {
  const uint8_t* p = static_cast<const uint8_t*>(data);
  for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 1099511628211ull; }
  return h;
}
uint64_t host_text_fingerprint(const void* ctx, size_t bytes, const int32_t* mask, size_t mask_n) {
  uint64_t h = 1469598103934665603ull;
  h = fnv1a(h, &bytes, sizeof bytes);
  const uint8_t* p = static_cast<const uint8_t*>(ctx);
  if (bytes <= 8192) {
    h = fnv1a(h, p, bytes);
  } else {
    h = fnv1a(h, p, 64);
    h = fnv1a(h, p + bytes - 64, 64);
    const size_t words = bytes / 8, step = words / 512;
    for (size_t i = 0; i < 512; ++i) h = fnv1a(h, p + (i * step) * 8, 8);
  }
  if (mask) h = fnv1a(h, mask, mask_n * 4);
  else h = fnv1a(h, &mask_n, 1);
  return h ? h : 1;
}
// drop the entry cached under `key` if it was built from different host buffers
void text_cache_guard(TextCache* slots, uint64_t key, uint64_t fp) {
  if (key == 0) return;
  for (int i = 0; i < 2; ++i)
    if (slots[i].key == key && slots[i].fingerprint != 0 && slots[i].fingerprint != fp) { slots[i].key = 0; slots[i].fingerprint = 0; }
}
void text_cache_stamp(TextCache* slots, uint64_t key, uint64_t fp) {
  if (key == 0) return;
  for (int i = 0; i < 2; ++i)
    if (slots[i].key == key) slots[i].fingerprint = fp;
}

// ---------------------------------------------------------------- captured step graphs
// A denoise step is ~600 kernel launches whose sequence depends only on shapes, flags and buffer addresses.  run_graphed
// runs `body` -- code that only ENQUEUES work on c->stream -- eagerly the first time a key is seen (so every grow-only
// workspace reaches its final size), captures it into a CUDA graph the second time, and replays the graph from then on: no
// per-launch host work (tensor-map encoding, argument marshalling), and launch gaps handled by the graph executor.  A graph
// is dropped when any workspace was (re)allocated since its capture; anything that cannot be captured falls back to eager.
struct KeyBuilder {
  std::string s;
  template <typename T>
  KeyBuilder& add(const T& v) {
    s.append(reinterpret_cast<const char*>(&v), sizeof v);
    return *this;
  }
};

void graph_destroy(StepGraph& g) {
  if (g.exec) cudaGraphExecDestroy(g.exec);
  g.exec = nullptr;
}

template <typename Fn>
void run_graphed(ltx_ctx* c, const std::string& key, bool eligible, Fn&& body) {
  static const bool env_on = [] { const char* e = getenv("LTX_GRAPH"); return e ? atoi(e) != 0 : true; }();
  if (!eligible || !env_on || !c->graphs_enabled || c->prof_on) { body(); return; }
  auto it = c->graphs.find(key);
  if (it != c->graphs.end() && it->second.state == 1 && it->second.generation != devbuf_generation().load()) {
    graph_destroy(it->second);   // a workspace moved since the capture
    c->graphs.erase(it);
    it = c->graphs.end();
  }
  if (it == c->graphs.end()) {   // first sighting: eager, so that every workspace reaches its final size
    if (c->graphs.size() >= 8) {
      auto lru = c->graphs.begin();
      for (auto j = c->graphs.begin(); j != c->graphs.end(); ++j)
        if (j->second.last_use < lru->second.last_use) lru = j;
      graph_destroy(lru->second);
      c->graphs.erase(lru);
    }
    StepGraph g;
    g.last_use = ++c->graph_clock;
    c->graphs[key] = g;
    body();
    return;
  }
  StepGraph& g = it->second;
  g.last_use = ++c->graph_clock;
  if (g.state < 0) { body(); return; }   // capture failed before: stay eager
  if (g.state == 0) {
    const uint64_t gen = devbuf_generation().load();
    const uint64_t l0 = c->launches;
    cudaGraph_t graph = nullptr;
    bool ok = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed) == cudaSuccess;
    if (ok) {
      try {
        body();
      } catch (...) {
        cudaStreamEndCapture(c->stream, &graph);
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        g.state = -1;
        throw;
      }
      ok = cudaStreamEndCapture(c->stream, &graph) == cudaSuccess && graph != nullptr;
    }
    const uint64_t n_launch = c->launches - l0;
    if (ok && devbuf_generation().load() == gen) ok = cudaGraphInstantiate(&g.exec, graph, 0) == cudaSuccess;
    else ok = false;
    if (graph) cudaGraphDestroy(graph);
    if (!ok) {   // nothing has run yet: do the step eagerly and do not try again for this key
      cudaGetLastError();
      graph_destroy(g);
      g.state = -1;
      c->launches = l0;
      body();
      return;
    }
    g.state = 1;
    g.generation = gen;
    g.launches = n_launch;
    c->graph_captures++;
    LTX_CUDA(cudaGraphLaunch(g.exec, c->stream));
    return;
  }
  c->launches += g.launches;
  c->graph_replays++;
  LTX_CUDA(cudaGraphLaunch(g.exec, c->stream));
}

const TextCache* find_text(const TextCache* slots, uint64_t key, int B, int S) {
  if (key == 0) return nullptr;
  for (int i = 0; i < 2; ++i)
    if (slots[i].key == key && slots[i].B == B && slots[i].S == S) return &slots[i];
  return nullptr;
}

}  // namespace

namespace ltx {
void graphs_clear(ltx_ctx* c) {
  for (auto& kv : c->graphs) graph_destroy(kv.second);
  c->graphs.clear();
}
}  // namespace ltx

extern "C" {

const char* ltx_version(void) { return "ltxcuda 0.1.0 (sm_100a)"; }

void ltx_config_default(ltx_config* cfg) {
  if (!cfg) return;
  cfg->num_layers = 48;
  cfg->num_heads = 32;
  cfg->head_dim = 128;
  cfg->in_channels = 128;
  cfg->out_channels = 128;
  cfg->caption_channels = 3840;
  cfg->ffn_mult = 4;
  cfg->rope_theta = 10000.0f;
  cfg->max_pos[0] = 20;
  cfg->max_pos[1] = 2048;
  cfg->max_pos[2] = 2048;
  cfg->timestep_scale_multiplier = 1000.0f;
  cfg->norm_eps = 1e-6f;
  cfg->vae_latent_channels = 128;
  cfg->vae_base_channels = 1024;
  cfg->vae_blocks_per_stage = 5;
  cfg->vae_patch_size = 4;
  cfg->vae_encoder_base_channels = 128;
  cfg->upscaler_mid_channels = 1024;
  cfg->upscaler_blocks = 4;
  cfg->audio_num_heads = 32;
  cfg->audio_head_dim = 64;
  cfg->audio_in_channels = 128;
  cfg->audio_max_pos = 20;
}

int ltx_ctx_create(const ltx_config* cfg, int device, ltx_ctx** out) {
  if (!cfg || !out) return LTX_ERR_INVALID_ARGUMENT;
  *out = nullptr;
  try {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    LTX_CHECK(e == cudaSuccess && ndev > 0, LTX_ERR_CUDA, "no CUDA device available (libltxcuda has no CPU fallback)");
    LTX_CHECK(device >= 0 && device < ndev, LTX_ERR_INVALID_ARGUMENT, "bad device index");
    cudaDeviceProp prop;
    LTX_CUDA(cudaGetDeviceProperties(&prop, device));
    LTX_CHECK(prop.major == 10, LTX_ERR_CUDA,
              std::string("libltxcuda requires an sm_100a (Blackwell) device, found ") + prop.name);
    LTX_CHECK(cfg->head_dim == 128, LTX_ERR_INVALID_CONFIGURATION, "head_dim must be 128");
    LTX_CHECK(cfg->num_layers > 0 && cfg->num_heads > 0 && cfg->ffn_mult > 0, LTX_ERR_INVALID_CONFIGURATION,
              "bad transformer configuration");
    LTX_CUDA(cudaSetDevice(device));
    ltx_ctx* c = new ltx_ctx();
    c->cfg = *cfg;
    c->device = device;
    LTX_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    *out = c;
    return LTX_OK;
  } catch (const LtxError& e) {
    g_create_error = e.what();
    return e.code;
  } catch (const std::exception& e) {
    g_create_error = e.what();
    return LTX_ERR_CUDA;
  }
}

int ltx_ctx_destroy(ltx_ctx* c) {
  if (!c) return LTX_OK;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  graphs_clear(c);
  try { dist_destroy(c); } catch (...) {}
  for (auto& kv : c->tensors)
    if (kv.second.ptr) cudaFree(kv.second.ptr);
  for (void* p : c->owned) cudaFree(p);
  DevBuf* bufs[] = {&c->sp_send, &c->sp_recv, &c->sp_vt, &c->sp_vel, &c->api_lat, &c->api_ctx, &c->lat_in, &c->ctx_in, &c->ts_in, &c->mask_in, &c->x, &c->xb, &c->h, &c->qk, &c->vt, &c->att, &c->q2,
                    &c->ffh, &c->vel, &c->se, &c->t1, &c->emb, &c->ada, &c->c1, &c->c2, &c->rope_cos, &c->rope_sin,
                    &c->scratch, &c->s_latent, &c->s_tok, &c->s_vc, &c->s_vu, &c->s_vs, &c->s_vprev, &c->s_ctx_pos,
                    &c->s_ctx_neg, &c->s_mask_pos, &c->s_mask_neg, &c->s_ctx_pair, &c->s_mask_pair, &c->s_sigma, &c->v_a, &c->v_b, &c->v_h, &c->v_pad,
                    &c->v_lat, &c->v_noise, &c->v_frames, &c->v_mix, &c->v_te, &c->v_split, &c->v_pad2, &c->snap_x, &c->s_ts, &c->f_asplit, &c->f_wsplit, &c->f_h,
                    &c->f_q, &c->f_k, &c->f_v, &c->f_att, &c->f_ffh, &c->f_ctx, &c->f_c1, &c->f_c2, &c->f_tk, &c->f_tv, &c->f_lat,
                    &c->f_bias, &c->q_panel, &c->gemm_ws, &c->u_part, &c->u_ab, &c->u_stats, &c->u_in, &c->u_out, &c->u_ref, &c->av.ws, &c->av.a_cos, &c->av.a_sin, &c->av.xv_cos, &c->av.xv_sin, &c->av_in[0], &c->av_in[1], &c->av_in[2], &c->av_in[3], &c->av_in[4], &c->av_in[5], &c->av_in[6], &c->av_in[7],
                    &c->v_tile_lat, &c->v_tile_noise, &c->v_tile_frames, &c->s_alat, &c->s_avc, &c->s_avu, &c->s_actx_pos, &c->s_actx_neg, &c->s_alat_pair, &c->s_actx_pair};
  for (DevBuf* b : bufs) b->release();
  for (auto& t : c->text) { t.k.release(); t.vt.release(); t.bias.release(); }
  for (auto& t : c->av.text) { t.k.release(); t.vt.release(); t.bias.release(); }
  cudaStreamDestroy(c->stream);
  delete c;
  return LTX_OK;
}

const char* ltx_last_error(const ltx_ctx* c) { return c ? c->last_error.c_str() : g_create_error.c_str(); }

int ltx_sync(ltx_ctx* c) {
  return guarded(c, [&] { LTX_CUDA(cudaStreamSynchronize(c->stream)); });
}

uint64_t ltx_launch_count(const ltx_ctx* c) { return c ? c->launches : 0; }

int ltx_host_alloc(void** ptr, size_t bytes) {
  if (!ptr || bytes == 0) return LTX_ERR_INVALID_ARGUMENT;
  *ptr = nullptr;
  return cudaHostAlloc(ptr, bytes, cudaHostAllocDefault) == cudaSuccess ? LTX_OK : LTX_ERR_CUDA;
}

int ltx_host_free(void* ptr) {
  if (!ptr) return LTX_OK;
  return cudaFreeHost(ptr) == cudaSuccess ? LTX_OK : LTX_ERR_CUDA;
}

int ltx_dist_get_unique_id(void* id_out_128) {
  if (!id_out_128) return LTX_ERR_INVALID_ARGUMENT;
  try {
    dist_get_unique_id(id_out_128);
    return LTX_OK;
  } catch (const LtxError& e) {
    g_create_error = e.what();
    return e.code;
  }
}

int ltx_dist_init(ltx_ctx* c, const void* unique_id_128, int rank, int world_size, int sp_size, int pass_groups) {
  return guarded(c, [&] {
    graphs_clear(c);
    LTX_CHECK(unique_id_128 != nullptr, LTX_ERR_INVALID_ARGUMENT, "null unique id");
    dist_init(c, unique_id_128, rank, world_size, sp_size, pass_groups);
  });
}

int ltx_dist_init_local(ltx_ctx** contexts, int n, int sp_size, int pass_groups) {
  if (!contexts || n < 1 || !contexts[0]) return LTX_ERR_INVALID_ARGUMENT;
  return guarded(contexts[0], [&] {
    for (int i = 0; i < n; ++i)
      if (contexts[i]) graphs_clear(contexts[i]);
    dist_init_local(contexts, n, sp_size, pass_groups);
  });
}

int ltx_dist_shutdown(ltx_ctx* c) {
  return guarded(c, [&] {
    graphs_clear(c);
    LTX_CUDA(cudaStreamSynchronize(c->stream));
    dist_destroy(c);
  });
}

int ltx_dist_info(const ltx_ctx* c, int* rank, int* world_size, int* sp_size, int* pass_groups) {
  if (!c) return LTX_ERR_INVALID_ARGUMENT;
  if (rank) *rank = c->dist.rank;
  if (world_size) *world_size = c->dist.world;
  if (sp_size) *sp_size = c->dist.sp;
  if (pass_groups) *pass_groups = c->dist.groups;
  return LTX_OK;
}

int ltx_dist_p2p_active(const ltx_ctx* c) { return (c && c->dist.p2p) ? 1 : 0; }

int ltx_get_stream(ltx_ctx* c, void** stream) {
  return guarded(c, [&] {
    LTX_CHECK(stream != nullptr, LTX_ERR_INVALID_ARGUMENT, "null out pointer");
    *stream = reinterpret_cast<void*>(c->stream);
  });
}

int ltx_set_graphs(ltx_ctx* c, int enabled) {
  return guarded(c, [&] {
    c->graphs_enabled = enabled ? 1 : 0;
    if (!enabled) graphs_clear(c);
  });
}

int ltx_graph_stats(const ltx_ctx* c, uint64_t* captures, uint64_t* replays) {
  if (!c) return LTX_ERR_INVALID_ARGUMENT;
  if (captures) *captures = c->graph_captures;
  if (replays) *replays = c->graph_replays;
  return LTX_OK;
}

int ltx_set_profiling(ltx_ctx* c, int enabled) {
  return guarded(c, [&] {
    LTX_CUDA(cudaStreamSynchronize(c->stream));
    for (auto& r : c->prof_recs) { c->prof_pool.push_back(r.a); c->prof_pool.push_back(r.b); }
    c->prof_recs.clear();
    c->prof_on = enabled != 0;
  });
}

int ltx_get_profile(ltx_ctx* c, double* ms, double* flops, double* bytes, uint64_t* counts, int n_classes) {
  return guarded(c, [&] {
    LTX_CHECK(ms && flops && bytes && counts && n_classes >= PROF_NCLASS, LTX_ERR_INVALID_ARGUMENT, "bad profile buffers");
    LTX_CUDA(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < n_classes; ++i) { ms[i] = 0; flops[i] = 0; bytes[i] = 0; counts[i] = 0; }
    for (auto& r : c->prof_recs) {
      float t = 0.f;
      LTX_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
      ms[r.cls] += t; flops[r.cls] += r.flops; bytes[r.cls] += r.bytes; counts[r.cls] += 1;
      c->prof_pool.push_back(r.a); c->prof_pool.push_back(r.b);
    }
    c->prof_recs.clear();
  });
}

int ltx_load_tensor(ltx_ctx* c, const char* key, const void* host_data, ltx_dtype dtype, const int64_t* shape, int ndim) {
  return guarded(c, [&] {
    LTX_CHECK(key != nullptr, LTX_ERR_INVALID_ARGUMENT, "null key");
    load_tensor_host(c, key, host_data, dtype, shape, ndim);
  });
}

int ltx_load_safetensors(ltx_ctx* c, const char* path, int which, int* n_loaded) {
  return guarded(c, [&] {
    const int n = load_safetensors(c, path, which);
    if (n_loaded) *n_loaded = n;
    static const char* kWhat[] = {"", "transformer", "VAE decoder", "VAE encoder", "upscaler", "audio/video transformer"};
    LTX_CHECK(n > 0, LTX_ERR_WEIGHTS, std::string("no ") + kWhat[which] + " tensors found in '" + (path ? path : "") + "'");
  });
}

int ltx_map_weight_key(int which, const char* file_key, char* out, size_t cap) {
  if (!file_key || !out || cap == 0 || which < 1 || which > 6) return LTX_ERR_INVALID_ARGUMENT;
  try {
    const std::string m = which == 1   ? map_transformer_key(file_key)
                          : which == 2 ? map_vae_key(file_key)
                          : which == 3 ? map_vae_encoder_key(file_key)
                          : which == 4 ? map_upscaler_key(file_key)
                          : which == 5 ? map_transformer_key(file_key, true)
                                       : map_lora_key(file_key);
    if (m.size() + 1 > cap) return LTX_ERR_INVALID_ARGUMENT;
    memcpy(out, m.c_str(), m.size() + 1);
    return LTX_OK;
  } catch (...) {
    return LTX_ERR_WEIGHTS;
  }
}

int ltx_fuse_lora(ltx_ctx* c, const char* key, const void* down, const void* up, ltx_dtype dtype, int rank, float scale) {
  return guarded(c, [&] {
    LTX_CHECK(key != nullptr, LTX_ERR_INVALID_ARGUMENT, "null key");
    fuse_lora(c, key, down, up, dtype, rank, scale);
  });
}

int ltx_init_random_weights(ltx_ctx* c, int which, uint64_t seed) {
  return guarded(c, [&] { init_random_weights(c, which, seed); });
}

int ltx_set_precision(ltx_ctx* c, int bits) {
  return guarded(c, [&] {
    LTX_CHECK(bits == 16 || bits == 32 || bits == 8, LTX_ERR_UNSUPPORTED,
              "precision must be 16 (bf16 mode), 32 (fp32 mode) or 8 (FP8 mode)");
    LTX_CHECK(bits != 8 || (!c->dit_ready && c->tensors.count("patchify_proj.weight") == 0), LTX_ERR_UNSUPPORTED,
              "FP8 mode must be set before the DiT weights are loaded");
    LTX_CHECK(!c->dit_ready && c->tensors.count("patchify_proj.weight") == 0, LTX_ERR_INVALID_ARGUMENT,
              "ltx_set_precision must be called before the DiT weights are loaded");
    c->precision = bits;
  });
}

int ltx_set_quant_storage(ltx_ctx* c, int materialise) {
  return guarded(c, [&] { c->quant_materialise = materialise ? 1 : 0; });
}

int ltx_finalize_weights(ltx_ctx* c, int quant_bits, int group_size) {
  return guarded(c, [&] {
    LTX_CHECK(quant_bits == 16 || quant_bits == 8 || quant_bits == 4, LTX_ERR_UNSUPPORTED, "quant_bits must be 16, 8 or 4");
    LTX_CHECK(quant_bits == 16 || group_size == 64, LTX_ERR_UNSUPPORTED, "only group_size 64 is implemented");
    LTX_CHECK(quant_bits == 16 || c->precision == 16, LTX_ERR_UNSUPPORTED,
              "fp32 and FP8 modes cannot be combined with quantised weights");
    graphs_clear(c);
    // each component is packed once; a later call (after loading another component) only packs what is new
    if (c->tensors.count("patchify_proj.weight") && !c->dit_ready) {
      if (c->precision == 32) dit_finalize_f32(c);
      else dit_finalize(c);
      if (c->tensors.count("audio_patchify_proj.weight")) {
        LTX_CHECK(c->precision == 16, LTX_ERR_UNSUPPORTED, "the dual audio/video model has no fp32 or FP8 mode");
        dit_av_finalize(c);
      }
      if (quant_bits != 16) dit_quantize(c, quant_bits);
      if (c->precision == 8) dit_convert_fp8(c);
    }
    if (c->tensors.count("vae.conv_in.conv.weight") && !c->vae.ready) vae_finalize(c);
    if (c->tensors.count("vae_encoder.conv_in.conv.weight") && !c->enc.ready) vae_encoder_finalize(c);
    if (c->tensors.count("upscaler.initial_conv.weight") && !c->ups.ready) upscaler_finalize(c);
    LTX_CHECK(c->dit_ready || c->vae.ready || c->enc.ready || c->ups.ready, LTX_ERR_WEIGHTS, "no weights loaded");
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_dit_forward_dev(ltx_ctx* c, const void* latent, ltx_dtype latent_dtype, const void* context,
                        ltx_dtype context_dtype, const float* timesteps, int ts_per_token, const int32_t* mask, int B, int N,
                        int S, int F, int H, int W, const ltx_dit_flags* flags, float* out_velocity) {
  return guarded(c, [&] {
    dit_forward_dev(c, latent, latent_dtype, context, context_dtype, timesteps, ts_per_token, mask, B, N, S, F, H, W, flags,
                    out_velocity);
  });
}

int ltx_dit_forward(ltx_ctx* c, const void* latent, ltx_dtype latent_dtype, const void* context, ltx_dtype context_dtype,
                    const float* timesteps, int ts_per_token, const int32_t* mask, int B, int N, int S, int F, int H,
                    int W, const ltx_dit_flags* flags, float* out_velocity) {
  return guarded(c, [&] {
    LTX_CHECK(latent && context && timesteps && out_velocity, LTX_ERR_INVALID_ARGUMENT, "null tensor");
    LTX_CHECK(B >= 1 && N >= 1 && S >= 1, LTX_ERR_INVALID_ARGUMENT, "bad B/N/S");
    const ltx_config& g = c->cfg;
    const size_t R = static_cast<size_t>(B) * N;
    // the staged copies live in dedicated buffers (dit_forward_dev's own staging buffers are distinct: it is told bf16
    // inputs are already on the device only when no cast is needed)
    DevBuf& lat = c->api_lat;
    DevBuf& ctx = c->api_ctx;
    h2d(c, lat, latent, R * g.in_channels * dsize(latent_dtype));
    const uint64_t key = flags ? flags->context_key : 0;
    const size_t ctx_bytes = static_cast<size_t>(B) * S * g.caption_channels * dsize(context_dtype);
    const uint64_t fp = key ? host_text_fingerprint(context, ctx_bytes, mask, static_cast<size_t>(B) * S) : 0;
    text_cache_guard(c->text, key, fp);
    const bool cached = flags && flags->context_key != 0 &&
                        ((c->text[0].key == flags->context_key && c->text[0].B == B && c->text[0].S == S) ||
                         (c->text[1].key == flags->context_key && c->text[1].B == B && c->text[1].S == S));
    if (!cached) h2d(c, ctx, context, ctx_bytes);
    h2d(c, c->ts_in, timesteps, (ts_per_token ? R : static_cast<size_t>(B)) * 4);
    const int32_t* mask_dev = nullptr;
    if (mask) {
      h2d(c, c->mask_in, mask, static_cast<size_t>(B) * S * 4);
      mask_dev = c->mask_in.as<int32_t>();
    }
    c->vel.reserve(R * g.out_channels * 4);
    // steady state of a denoise loop at this seam (text cached under the key, RoPE table built): the forward is a fixed launch
    // sequence on fixed buffers -> replay it as a graph
    const TextCache* tcache = find_text(c->text, key, B, S);
    const bool steady = tcache != nullptr && c->precision != 32 && c->rope_f == F && c->rope_h == H && c->rope_w == W && c->rope_cos.ptr;
    KeyBuilder kb;
    if (steady) {
      kb.add('F').add(B).add(N).add(S).add(F).add(H).add(W).add(static_cast<int>(latent_dtype)).add(static_cast<int>(context_dtype))
          .add(ts_per_token).add(mask_dev).add(lat.ptr).add(ctx.ptr).add(c->ts_in.ptr).add(c->vel.ptr).add(tcache->k.ptr).add(tcache->vt.ptr)
          .add(tcache->has_bias).add(c->rope_cos.ptr).add(c->dist.sp).add(c->dist.sp_rank).add(c->dist.p2p).add(c->quant_bits)
          .add(c->precision);
      kb.add(flags->n_stg_blocks).add(flags->skip_self_attn).add(flags->skip_ff).add(flags->n_cas_blocks).add(flags->cross_attn_scale);
      for (int i = 0; i < flags->n_stg_blocks && i < LTX_MAX_FLAG_BLOCKS; ++i) kb.add(flags->stg_blocks[i]);
      for (int i = 0; i < flags->n_cas_blocks && i < LTX_MAX_FLAG_BLOCKS; ++i) kb.add(flags->cas_blocks[i]);
    }
    run_graphed(c, kb.s, steady, [&] {
      dit_forward_dev(c, lat.ptr, latent_dtype, ctx.ptr, context_dtype, c->ts_in.as<float>(), ts_per_token, mask_dev, B, N, S, F,
                      H, W, flags, c->vel.as<float>());
    });
    text_cache_stamp(c->text, key, fp);
    LTX_CUDA(cudaMemcpyAsync(out_velocity, c->vel.ptr, R * g.out_channels * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

// The dual model shares the video block weights, which FP8 mode converts to e4m3: its forwards and loop are refused there.
static void av_precision_check(ltx_ctx* c) {
  LTX_CHECK(c->precision != 8, LTX_ERR_UNSUPPORTED, "the dual audio/video model has no FP8 mode");
}

int ltx_av_forward_dev(ltx_ctx* c, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                       ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                       const float* video_sigma, const float* audio_sigma, const int32_t* video_mask, const int32_t* audio_mask,
                       int N, int Ta, int S, int F, int H, int W, uint64_t context_key, float* out_video, float* out_audio) {
  return guarded(c, [&] {
    av_precision_check(c);
    dit_av_forward_dev(c, video_latent, video_dtype, audio_latent, audio_dtype, video_context, audio_context, context_dtype,
                       video_sigma, 0, audio_sigma, video_mask, audio_mask, 1, N, Ta, S, F, H, W, context_key, out_video, out_audio);
  });
}

int ltx_av_forward_tokens_dev(ltx_ctx* c, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                              ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                              const float* video_sigmas, const float* audio_sigma, const int32_t* video_mask,
                              const int32_t* audio_mask, int N, int Ta, int S, int F, int H, int W, uint64_t context_key,
                              float* out_video, float* out_audio) {
  return guarded(c, [&] {
    av_precision_check(c);
    dit_av_forward_dev(c, video_latent, video_dtype, audio_latent, audio_dtype, video_context, audio_context, context_dtype,
                       video_sigmas, 1, audio_sigma, video_mask, audio_mask, 1, N, Ta, S, F, H, W, context_key, out_video, out_audio);
  });
}

// refusals of the batched dual forward that come before any work: B outside 1..2, B = 2 under Ulysses, null tensors
static void av_batch_check(ltx_ctx* c, int B, const void* vl, const void* al, const void* vc, const void* ac, const float* vs,
                           const float* as, const void* ov, const void* oa) {
  av_precision_check(c);
  LTX_CHECK(B >= 1, LTX_ERR_INVALID_ARGUMENT, "dual forward: B must be >= 1");
  LTX_CHECK(B <= 2, LTX_ERR_UNSUPPORTED, "dual forward: batches of 1 or 2 items");
  LTX_CHECK(B == 1 || !(c->dist.comm_world && c->dist.sp > 1), LTX_ERR_UNSUPPORTED, "the batched dual forward is single-GPU");
  LTX_CHECK(vl && al && vc && ac && vs && as && ov && oa, LTX_ERR_INVALID_ARGUMENT, "null tensor");
}

int ltx_av_forward_batch_dev(ltx_ctx* c, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                             ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                             const float* video_sigmas, int video_ts_per_token, const float* audio_sigmas,
                             const int32_t* video_mask, const int32_t* audio_mask, int B, int N, int Ta, int S, int F, int H, int W,
                             uint64_t context_key, float* out_video, float* out_audio) {
  return guarded(c, [&] {
    av_batch_check(c, B, video_latent, audio_latent, video_context, audio_context, video_sigmas, audio_sigmas, out_video, out_audio);
    dit_av_forward_dev(c, video_latent, video_dtype, audio_latent, audio_dtype, video_context, audio_context, context_dtype,
                       video_sigmas, video_ts_per_token ? 1 : 0, audio_sigmas, video_mask, audio_mask, B, N, Ta, S, F, H, W,
                       context_key, out_video, out_audio);
  });
}

// host-buffer form of the dual forward for B items; video_sigmas holds B values, or B * N when per_token; audio_sigmas B
static int av_forward_host(ltx_ctx* c, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                           ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                           const float* video_sigmas, int per_token, const float* audio_sigmas, const int32_t* video_mask,
                           const int32_t* audio_mask, int B, int N, int Ta, int S, int F, int H, int W, uint64_t context_key,
                           float* out_video, float* out_audio) {
  return guarded(c, [&] {
    av_batch_check(c, B, video_latent, audio_latent, video_context, audio_context, video_sigmas, audio_sigmas, out_video, out_audio);
    LTX_CHECK(N >= 1 && Ta >= 1 && S >= 1 && c->av.ready, LTX_ERR_INVALID_ARGUMENT, "bad sizes, or dual-model weights not finalized");
    const ltx_config& g = c->cfg;
    const int Ca = c->av.Cin;
    DevBuf* b = c->av_in;   // staged host inputs: video latent, audio latent, contexts, sigmas, masks, outputs
    h2d(c, b[0], video_latent, static_cast<size_t>(B) * N * g.in_channels * dsize(video_dtype));
    h2d(c, b[1], audio_latent, static_cast<size_t>(B) * Ta * Ca * dsize(audio_dtype));
    const size_t cbytes = static_cast<size_t>(B) * S * g.caption_channels * dsize(context_dtype), nm = static_cast<size_t>(B) * S;
    h2d(c, b[2], video_context, cbytes);
    h2d(c, b[3], audio_context, cbytes);
    // sigmas: [audio x B, video...] so the video values start 4-byte aligned right behind the audio ones
    const size_t nvs = static_cast<size_t>(B) * (per_token ? N : 1);
    b[4].reserve((B + nvs) * 4);
    LTX_CUDA(cudaMemcpyAsync(b[4].ptr, audio_sigmas, B * 4, cudaMemcpyHostToDevice, c->stream));
    LTX_CUDA(cudaMemcpyAsync(b[4].as<float>() + B, video_sigmas, nvs * 4, cudaMemcpyHostToDevice, c->stream));
    const int32_t *vm = nullptr, *am = nullptr;
    b[5].reserve(2 * nm * 4);
    if (video_mask) {
      LTX_CUDA(cudaMemcpyAsync(b[5].ptr, video_mask, nm * 4, cudaMemcpyHostToDevice, c->stream));
      vm = b[5].as<int32_t>();
    }
    if (audio_mask) {
      LTX_CUDA(cudaMemcpyAsync(b[5].as<int32_t>() + nm, audio_mask, nm * 4, cudaMemcpyHostToDevice, c->stream));
      am = b[5].as<int32_t>() + nm;
    }
    const size_t nov = static_cast<size_t>(B) * N * g.out_channels, noa = static_cast<size_t>(B) * Ta * Ca;
    b[6].reserve(nov * 4);
    b[7].reserve(noa * 4);
    const uint64_t fpv = context_key ? host_text_fingerprint(video_context, cbytes, video_mask, nm) : 0;
    const uint64_t fpa = context_key ? host_text_fingerprint(audio_context, cbytes, audio_mask, nm) : 0;
    text_cache_guard(c->text, context_key, fpv);
    text_cache_guard(c->av.text, context_key, fpa);
    dit_av_forward_dev(c, b[0].ptr, video_dtype, b[1].ptr, audio_dtype, b[2].ptr, b[3].ptr, context_dtype, b[4].as<float>() + B,
                       per_token, b[4].as<float>(), vm, am, B, N, Ta, S, F, H, W, context_key, b[6].as<float>(), b[7].as<float>());
    text_cache_stamp(c->text, context_key, fpv);
    text_cache_stamp(c->av.text, context_key, fpa);
    LTX_CUDA(cudaMemcpyAsync(out_video, b[6].ptr, nov * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaMemcpyAsync(out_audio, b[7].ptr, noa * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_av_forward(ltx_ctx* c, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent, ltx_dtype audio_dtype,
                   const void* video_context, const void* audio_context, ltx_dtype context_dtype, float video_sigma,
                   float audio_sigma, const int32_t* video_mask, const int32_t* audio_mask, int N, int Ta, int S, int F, int H,
                   int W, uint64_t context_key, float* out_video, float* out_audio) {
  return av_forward_host(c, video_latent, video_dtype, audio_latent, audio_dtype, video_context, audio_context, context_dtype,
                         &video_sigma, 0, &audio_sigma, video_mask, audio_mask, 1, N, Ta, S, F, H, W, context_key, out_video, out_audio);
}

int ltx_av_forward_batch(ltx_ctx* c, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                         ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                         const float* video_sigmas, int video_ts_per_token, const float* audio_sigmas, const int32_t* video_mask,
                         const int32_t* audio_mask, int B, int N, int Ta, int S, int F, int H, int W, uint64_t context_key,
                         float* out_video, float* out_audio) {
  return av_forward_host(c, video_latent, video_dtype, audio_latent, audio_dtype, video_context, audio_context, context_dtype,
                         video_sigmas, video_ts_per_token ? 1 : 0, audio_sigmas, video_mask, audio_mask, B, N, Ta, S, F, H, W,
                         context_key, out_video, out_audio);
}

int ltx_av_forward_tokens(ltx_ctx* c, const void* video_latent, ltx_dtype video_dtype, const void* audio_latent,
                          ltx_dtype audio_dtype, const void* video_context, const void* audio_context, ltx_dtype context_dtype,
                          const float* video_sigmas, float audio_sigma, const int32_t* video_mask, const int32_t* audio_mask, int N,
                          int Ta, int S, int F, int H, int W, uint64_t context_key, float* out_video, float* out_audio) {
  return av_forward_host(c, video_latent, video_dtype, audio_latent, audio_dtype, video_context, audio_context, context_dtype,
                         video_sigmas, 1, &audio_sigma, video_mask, audio_mask, 1, N, Ta, S, F, H, W, context_key, out_video, out_audio);
}

int ltx_dit_clear_caches(ltx_ctx* c) {
  return guarded(c, [&] { dit_clear_caches(c); });
}

int ltx_guided_euler_step_dev(ltx_ctx* c, float* latent, const float* v_cond, const float* v_uncond, const float* v_stg,
                              float* v_prev, int use_prev, size_t n, float cfg_scale, float rescale_phi, float stg_scale,
                              float ge_gamma, float sigma, float sigma_next) {
  return guarded(c, [&] {
    c->scratch.reserve(64 * sizeof(double));
    GuidedEulerArgs a;
    a.latent = latent; a.v_cond = v_cond; a.v_uncond = v_uncond; a.v_stg = v_stg; a.v_prev = v_prev;
    a.use_prev = use_prev; a.v_out = nullptr; a.n = n; a.cfg = cfg_scale; a.phi = rescale_phi; a.stg = stg_scale;
    a.ge_gamma = ge_gamma; a.sigma = sigma; a.sigma_next = sigma_next; a.scratch = c->scratch.as<double>();
    launch_guided_euler(a, c->stream);
    c->launches += (v_uncond && rescale_phi > 0.f) ? 2 : 1;
  });
}

int ltx_guided_euler_step(ltx_ctx* c, float* latent, const float* v_cond, const float* v_uncond, const float* v_stg,
                          float* v_prev, int use_prev, size_t n, float cfg_scale, float rescale_phi, float stg_scale,
                          float ge_gamma, float sigma, float sigma_next) {
  return guarded(c, [&] {
    LTX_CHECK(latent && v_cond && n > 0, LTX_ERR_INVALID_ARGUMENT, "null tensor");
    const size_t bytes = n * 4;
    h2d(c, c->s_latent, latent, bytes);
    h2d(c, c->s_vc, v_cond, bytes);
    if (v_uncond) h2d(c, c->s_vu, v_uncond, bytes);
    if (v_stg) h2d(c, c->s_vs, v_stg, bytes);
    if (v_prev) {
      if (use_prev) h2d(c, c->s_vprev, v_prev, bytes);
      else c->s_vprev.reserve(bytes);
    }
    c->scratch.reserve(64 * sizeof(double));
    GuidedEulerArgs a;
    a.latent = c->s_latent.as<float>(); a.v_cond = c->s_vc.as<float>();
    a.v_uncond = v_uncond ? c->s_vu.as<float>() : nullptr;
    a.v_stg = v_stg ? c->s_vs.as<float>() : nullptr;
    a.v_prev = v_prev ? c->s_vprev.as<float>() : nullptr;
    a.use_prev = use_prev; a.v_out = nullptr; a.n = n; a.cfg = cfg_scale; a.phi = rescale_phi; a.stg = stg_scale;
    a.ge_gamma = ge_gamma; a.sigma = sigma; a.sigma_next = sigma_next; a.scratch = c->scratch.as<double>();
    launch_guided_euler(a, c->stream);
    c->launches += (v_uncond && rescale_phi > 0.f) ? 2 : 1;
    LTX_CUDA(cudaMemcpyAsync(latent, c->s_latent.ptr, bytes, cudaMemcpyDeviceToHost, c->stream));
    if (v_prev) LTX_CUDA(cudaMemcpyAsync(v_prev, c->s_vprev.ptr, bytes, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

// ---------------------------------------------------------------- resident denoise session
int ltx_denoise_begin(ltx_ctx* c, const float* noise, int F, int H, int W, float sigma0, const void* context,
                      ltx_dtype context_dtype, const int32_t* mask, const void* neg_context, const int32_t* neg_mask, int S) {
  return guarded(c, [&] {
    LTX_CHECK(noise && context && F > 0 && H > 0 && W > 0 && S > 0, LTX_ERR_INVALID_ARGUMENT, "bad denoise_begin arguments");
    const ltx_config& g = c->cfg;
    LTX_CHECK(g.in_channels == g.out_channels, LTX_ERR_INVALID_CONFIGURATION, "in/out channels must match");
    const size_t n = static_cast<size_t>(g.in_channels) * F * H * W;
    c->s_F = F; c->s_H = H; c->s_W = W; c->s_S = S;
    c->s_Ta = 0;   // a video-only session: ltx_av_denoise_step is refused until ltx_av_denoise_begin
    c->s_ctx_dtype = context_dtype;
    h2d(c, c->s_latent, noise, n * 4);
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * n);
      launch_scale_f32(c->s_latent.as<float>(), sigma0, static_cast<int64_t>(n), c->stream);  // P/LTXPipeline.swift:793
    }
    const size_t cbytes = static_cast<size_t>(S) * g.caption_channels * dsize(context_dtype);
    h2d(c, c->s_ctx_pos, context, cbytes);
    c->s_has_mask_pos = mask != nullptr;
    if (mask) h2d(c, c->s_mask_pos, mask, static_cast<size_t>(S) * 4);
    c->s_has_neg = neg_context != nullptr;
    if (neg_context) {
      h2d(c, c->s_ctx_neg, neg_context, cbytes);
      c->s_has_mask_neg = neg_mask != nullptr;
      if (neg_mask) h2d(c, c->s_mask_neg, neg_mask, static_cast<size_t>(S) * 4);
      // batched guidance (denoise(), P/LTXPipeline.swift:2234-2269: latent doubled, one B = 2 forward): both prompts in one
      // [2, S, Cc] buffer, and one [2, S] mask when either prompt has one (all ones for the other)
      c->s_ctx_pair.reserve(2 * cbytes);
      LTX_CUDA(cudaMemcpyAsync(c->s_ctx_pair.ptr, c->s_ctx_pos.ptr, cbytes, cudaMemcpyDeviceToDevice, c->stream));
      LTX_CUDA(cudaMemcpyAsync(c->s_ctx_pair.as<uint8_t>() + cbytes, c->s_ctx_neg.ptr, cbytes, cudaMemcpyDeviceToDevice, c->stream));
      if (mask || neg_mask) {
        std::vector<int32_t> pm(static_cast<size_t>(2) * S, 1);
        if (mask) memcpy(pm.data(), mask, static_cast<size_t>(S) * 4);
        if (neg_mask) memcpy(pm.data() + S, neg_mask, static_cast<size_t>(S) * 4);
        h2d(c, c->s_mask_pair, pm.data(), pm.size() * 4);
        LTX_CUDA(cudaStreamSynchronize(c->stream));   // pm goes out of scope
      }
    }
    const size_t nb = neg_context ? 2 : 1;   // rows of the batched conditional + unconditional forward
    c->s_tok.reserve(nb * n * 2);
    c->s_vc.reserve(n * 4);
    c->s_vu.reserve(n * 4);
    c->s_vs.reserve(n * 4);
    c->s_vprev.reserve(n * 4);
    c->vel.reserve(nb * n * 4);
    c->s_sigma.reserve(16);
    c->s_serial += 2;  // fresh context-cache keys for this session
    dit_clear_caches(c);
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

namespace {
// LTX_BATCHED_CFG=0: the guidance passes of both denoise loops run as separate B = 1 forwards
bool batched_cfg_env() {
  static const bool on = [] { const char* e = getenv("LTX_BATCHED_CFG"); return e ? atoi(e) != 0 : true; }();
  return on;
}
// (re)sizes the per-session work buffers for a [C, F, H, W] latent and records the geometry
void session_resize(ltx_ctx* c, int F, int H, int W) {
  const size_t n = static_cast<size_t>(c->cfg.in_channels) * F * H * W;
  c->s_F = F; c->s_H = H; c->s_W = W;
  const size_t nb = c->s_has_neg ? 2 : 1;
  c->s_tok.reserve(nb * n * 2);
  c->s_vc.reserve(n * 4);
  c->s_vu.reserve(n * 4);
  c->s_vs.reserve(n * 4);
  c->s_vprev.reserve(n * 4);
  c->vel.reserve(nb * n * 4);
  c->s_sigma.reserve(16);
}
// latent[:, 0, :, :] = frame0 (host [C, 1, H, W]): the clean conditioning frame of the image-to-video loops
void session_set_frame0(ltx_ctx* c, const float* frame0_host) {
  const size_t hw = static_cast<size_t>(c->s_H) * c->s_W;
  LTX_CUDA(cudaMemcpy2DAsync(c->s_latent.ptr, static_cast<size_t>(c->s_F) * hw * 4, frame0_host, hw * 4, hw * 4,
                             static_cast<size_t>(c->cfg.in_channels), cudaMemcpyHostToDevice, c->stream));
}
}  // namespace

int ltx_denoise_begin_from_latent(ltx_ctx* c, const float* latent, const float* noise, float noise_scale,
                                  const float* frame0_latent, int F, int H, int W, const void* context, ltx_dtype context_dtype,
                                  const int32_t* mask, const void* neg_context, const int32_t* neg_mask, int S) {
  // same session set-up as ltx_denoise_begin, then the stage-2 start point (P/LTXPipeline.swift:2636-2657)
  int rc = ltx_denoise_begin(c, noise, F, H, W, 1.0f, context, context_dtype, mask, neg_context, neg_mask, S);
  if (rc != LTX_OK) return rc;
  return guarded(c, [&] {
    LTX_CHECK(latent != nullptr, LTX_ERR_INVALID_ARGUMENT, "null latent");
    const size_t n = static_cast<size_t>(c->cfg.in_channels) * F * H * W;
    h2d(c, c->u_in, latent, n * 4);
    // s_latent holds the noise: swap roles so that latent = s * noise + (1 - s) * latent lands in s_latent
    renoise_dev(c, c->u_in.as<float>(), c->s_latent.as<float>(), static_cast<int64_t>(n), noise_scale);
    LTX_CUDA(cudaMemcpyAsync(c->s_latent.ptr, c->u_in.ptr, n * 4, cudaMemcpyDeviceToDevice, c->stream));
    if (frame0_latent) session_set_frame0(c, frame0_latent);
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_denoise_set_frame0(ltx_ctx* c, const float* frame0_latent) {
  return guarded(c, [&] {
    LTX_CHECK(frame0_latent && c->s_F > 0, LTX_ERR_INVALID_ARGUMENT, "no denoise session");
    session_set_frame0(c, frame0_latent);
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_denoise_upscale_stage(ltx_ctx* c, const float* noise, float noise_scale, float adain_factor) {
  return guarded(c, [&] {
    LTX_CHECK(noise && c->s_F > 0, LTX_ERR_INVALID_ARGUMENT, "denoise_upscale_stage before denoise_begin");
    const int C = c->cfg.in_channels, F = c->s_F, H = c->s_H, W = c->s_W;
    const size_t n1 = static_cast<size_t>(C) * F * H * W, n2 = 4 * n1;
    // the stage-1 output is both the upscaler input and the AdaIN reference (P/LTXPipeline.swift:2604-2624)
    c->u_ref.reserve(n1 * 4);
    LTX_CUDA(cudaMemcpyAsync(c->u_ref.ptr, c->s_latent.ptr, n1 * 4, cudaMemcpyDeviceToDevice, c->stream));
    c->u_out.reserve(n2 * 4);
    upscale_latent_dev(c, c->u_ref.as<float>(), F, H, W, c->u_out.as<float>());
    adain_filter_dev(c, c->u_out.as<float>(), static_cast<int64_t>(4) * F * H * W, c->u_ref.as<float>(),
                     static_cast<int64_t>(F) * H * W, C, adain_factor);
    h2d(c, c->u_in, noise, n2 * 4);
    renoise_dev(c, c->u_out.as<float>(), c->u_in.as<float>(), static_cast<int64_t>(n2), noise_scale);   // :2644-2647
    LTX_CUDA(cudaStreamSynchronize(c->stream));   // s_latent is re-allocated below: nothing may still read it
    c->s_latent.reserve(n2 * 4);
    LTX_CUDA(cudaMemcpyAsync(c->s_latent.ptr, c->u_out.ptr, n2 * 4, cudaMemcpyDeviceToDevice, c->stream));
    session_resize(c, F, 2 * H, 2 * W);
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_denoise_step(ltx_ctx* c, const ltx_step_params* p) {
  return guarded(c, [&] {
    LTX_CHECK(p != nullptr && c->s_F > 0, LTX_ERR_INVALID_ARGUMENT, "denoise_step before denoise_begin");
    LTX_CHECK(p->sigma > 0.f, LTX_ERR_INVALID_ARGUMENT, "sigma must be > 0");
    const ltx_config& g = c->cfg;
    const int C = g.in_channels, F = c->s_F, H = c->s_H, W = c->s_W, S = c->s_S;
    const int T = F * H * W;
    const size_t n = static_cast<size_t>(C) * T;
    cudaStream_t st = c->stream;
    // the only per-step scalar the forward passes read lives in device memory (the captured step re-reads it on replay);
    // twice: the batched forward takes one timestep per batch row
    const float sig2[2] = {p->sigma, p->sigma};
    LTX_CUDA(cudaMemcpyAsync(c->s_sigma.ptr, sig2, 8, cudaMemcpyHostToDevice, st));
    const bool i2v = p->i2v_frame0_conditioned != 0;
    if (i2v) c->s_ts.reserve(static_cast<size_t>(2) * T * 4);
    const float* ts_dev = i2v ? c->s_ts.as<float>() : c->s_sigma.as<float>();
    const uint64_t key_pos = 0x5000000000000000ull + c->s_serial, key_neg = key_pos + 1;
    const uint64_t key_pair = 0x5800000000000000ull + c->s_serial;
    // SURVEY H10: the STG pass differs from the conditional pass only from its first perturbed block on; when both run
    // on this rank the conditional pass saves the stream there and the STG pass resumes from it (bit-identical result).
    int first_stg = -1;
    for (int i = 0; i < p->n_stg_blocks && i < LTX_MAX_FLAG_BLOCKS; ++i)
      if (first_stg < 0 || p->stg_blocks[i] < first_stg) first_stg = p->stg_blocks[i];
    auto pass = [&](bool neg, bool stg, float* v_lat, int snapshot_block, int resume_block) {
      ltx_dit_flags fl = {};
      fl.cross_attn_scale = 1.0f;
      fl.context_key = neg ? key_neg : key_pos;
      if (stg) {
        fl.n_stg_blocks = p->n_stg_blocks;
        for (int i = 0; i < p->n_stg_blocks && i < LTX_MAX_FLAG_BLOCKS; ++i) fl.stg_blocks[i] = p->stg_blocks[i];
        fl.skip_self_attn = 1;
      }
      const void* cx = neg ? c->s_ctx_neg.ptr : c->s_ctx_pos.ptr;
      const int32_t* mk = neg ? (c->s_has_mask_neg ? c->s_mask_neg.as<int32_t>() : nullptr)
                              : (c->s_has_mask_pos ? c->s_mask_pos.as<int32_t>() : nullptr);
      dit_forward_dev(c, c->s_tok.ptr, LTX_BF16, cx, c->s_ctx_dtype, ts_dev, i2v ? 1 : 0, mk, 1, T, S, F, H, W, &fl,
                      c->vel.as<float>(), snapshot_block, resume_block);
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * n);
      launch_unpatchify(c->vel.as<float>(), v_lat, C, T, st);  // velocity back to [C, F, H, W]
    };
    const bool use_cfg = p->cfg_scale > 1.0f && c->s_has_neg;
    const bool use_stg = p->stg_scale > 0.f && p->n_stg_blocks > 0;
    // pass p runs on pass group p % groups (all groups when there is one); velocities are then broadcast from the
    // first rank of the owning group so that every rank applies the same guided Euler update to its replicated latent
    struct PassDef { bool neg, stg; float* v; };
    PassDef passes[3];
    int n_pass = 0;
    passes[n_pass++] = {false, false, c->s_vc.as<float>()};
    if (use_cfg) passes[n_pass++] = {true, false, c->s_vu.as<float>()};
    if (use_stg) passes[n_pass++] = {false, true, c->s_vs.as<float>()};
    const int groups = c->dist.groups;
    // Conditional + unconditional as ONE B = 2 forward when both run on this GPU alone: M = 3072 rows fill the tile waves
    // better (N = 4096 GEMMs: 192 tiles instead of 2 x 96 on 74 CTA pairs; attention: 768 CTAs instead of 2 x 384 on 296
    // slots) and the weights are read once.  Batch row 0 is the conditional pass, so the STG pass can still resume from its
    // stream.  Per batch row the arithmetic is that of the separate passes.
    const bool batched = batched_cfg_env() && use_cfg && groups == 1 && !(c->dist.comm_world && c->dist.sp > 1) && c->precision != 32 &&
                         !p->disable_batched_cfg;
    const int stg_idx = use_stg ? n_pass - 1 : -1;
    const bool share = use_stg && !p->disable_stg_prefix_sharing && first_stg > 0 && first_stg < g.num_layers &&
                       (groups == 1 || (stg_idx % groups) == 0);   // conditional pass (index 0) and STG pass on the same group
    // everything up to the guided Euler update: patchify, the forward passes of this rank's group, velocity exchange
    auto forwards = [&] {
      {
        // patchify(latent).asType(.bfloat16)  (P/LTXPipeline.swift:815)
        ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * n);
        launch_patchify(c->s_latent.as<float>(), c->s_tok.as<bf16>(), nullptr, C, T, st);
      }
      // image-conditioned loop (denoise(), P/LTXPipeline.swift:2237-2252, 2344-2357): frame-0 tokens are clean -> per-token
      // timesteps sigma * (1 - mask), and the Euler update leaves frame 0 untouched
      if (i2v) {
        ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * T);
        launch_fill_token_timesteps(c->s_ts.as<float>(), batched ? 2 * T : T, T, H * W, c->s_sigma.as<float>(), st);
      }
      if (batched) {
        bf16* tok = c->s_tok.as<bf16>();
        LTX_CUDA(cudaMemcpyAsync(tok + n, tok, n * 2, cudaMemcpyDeviceToDevice, st));   // the same latent under both prompts
        ltx_dit_flags fl = {};
        fl.cross_attn_scale = 1.0f;
        fl.context_key = key_pair;
        const int32_t* mk = (c->s_has_mask_pos || c->s_has_mask_neg) ? c->s_mask_pair.as<int32_t>() : nullptr;
        dit_forward_dev(c, tok, LTX_BF16, c->s_ctx_pair.ptr, c->s_ctx_dtype, ts_dev, i2v ? 1 : 0, mk, 2, T, S, F, H, W, &fl,
                        c->vel.as<float>(), share ? first_stg : -1, -1);
        ProfScope ps(c, PROF_OTHER, 0.0, 16.0 * n, 2);
        launch_unpatchify(c->vel.as<float>(), c->s_vc.as<float>(), C, T, st);
        launch_unpatchify(c->vel.as<float>() + n, c->s_vu.as<float>(), C, T, st);
      }
      for (int i = 0; i < n_pass; ++i) {
        if (batched && !passes[i].stg) continue;   // done above
        if (groups == 1 || (i % groups) == c->dist.group)
          pass(passes[i].neg, passes[i].stg, passes[i].v, (share && i == 0) ? first_stg : -1, (share && passes[i].stg) ? first_stg : -1);
      }
      if (groups > 1) {
        ProfScope ps(c, PROF_COMM, 0.0, 4.0 * n * n_pass, n_pass);
        for (int i = 0; i < n_pass; ++i) dist_broadcast(c, passes[i].v, n * 4, (i % groups) * c->dist.sp);
      }
    };
    // Steady state (every step of a session but the first): the projected text of each prompt this rank needs is cached and
    // the RoPE table is built, so the step is a fixed launch sequence on fixed buffers -> captured once, then replayed.
    bool steady = c->precision != 32 && c->rope_f == F && c->rope_h == H && c->rope_w == W && c->rope_cos.ptr != nullptr;
    KeyBuilder kb;
    kb.add('S').add(F).add(H).add(W).add(S).add(i2v).add(use_cfg).add(use_stg).add(share).add(first_stg).add(p->n_stg_blocks).add(batched)
        .add(c->dist.world).add(c->dist.rank).add(c->dist.sp).add(groups).add(c->dist.p2p).add(c->quant_bits).add(c->precision).add(c->s_ctx_dtype)
        .add(c->s_latent.ptr).add(c->s_tok.ptr).add(c->s_sigma.ptr).add(c->s_ts.ptr).add(c->vel.ptr).add(c->rope_cos.ptr);
    for (int i = 0; i < p->n_stg_blocks && i < LTX_MAX_FLAG_BLOCKS; ++i) kb.add(p->stg_blocks[i]);
    if (batched) {
      const TextCache* tcache = find_text(c->text, key_pair, 2, S);
      if (!tcache) steady = false;
      else kb.add(tcache->k.ptr).add(tcache->vt.ptr).add(tcache->has_bias).add(c->s_ctx_pair.ptr);
    }
    for (int i = 0; i < n_pass && steady; ++i) {
      if (batched && !passes[i].stg) continue;
      if (!(groups == 1 || (i % groups) == c->dist.group)) continue;
      const TextCache* tcache = find_text(c->text, passes[i].neg ? key_neg : key_pos, 1, S);
      if (!tcache) { steady = false; break; }
      kb.add(i).add(tcache->k.ptr).add(tcache->vt.ptr).add(tcache->has_bias).add(passes[i].v);
    }
    run_graphed(c, kb.s, steady, forwards);
    GuidedEulerArgs a;
    a.latent = c->s_latent.as<float>(); a.v_cond = c->s_vc.as<float>();
    a.v_uncond = use_cfg ? c->s_vu.as<float>() : nullptr;
    a.v_stg = use_stg ? c->s_vs.as<float>() : nullptr;
    a.v_prev = c->s_vprev.as<float>();
    a.use_prev = p->step_index > 0 ? 1 : 0;
    a.v_out = nullptr; a.n = n; a.cfg = p->cfg_scale; a.phi = p->rescale_phi; a.stg = p->stg_scale;
    a.ge_gamma = p->ge_gamma; a.sigma = p->sigma; a.sigma_next = p->sigma_next; a.scratch = c->scratch.as<double>();
    if (i2v) { a.period = static_cast<size_t>(T); a.frozen = static_cast<size_t>(H) * W; }
    ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * n * (4.0 + (use_cfg ? 1.0 : 0.0) + (use_stg ? 1.0 : 0.0)),
                 (use_cfg && p->rescale_phi > 0.f) ? 2 : 1);
    launch_guided_euler(a, st);
  });
}

int ltx_denoise_get_latent(ltx_ctx* c, float* out) {
  return guarded(c, [&] {
    LTX_CHECK(out && c->s_F > 0, LTX_ERR_INVALID_ARGUMENT, "no denoise session");
    const size_t n = static_cast<size_t>(c->cfg.in_channels) * c->s_F * c->s_H * c->s_W;
    LTX_CUDA(cudaMemcpyAsync(out, c->s_latent.ptr, n * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_denoise_latent_dev(ltx_ctx* c, float** p) {
  return guarded(c, [&] {
    LTX_CHECK(p && c->s_F > 0, LTX_ERR_INVALID_ARGUMENT, "no denoise session");
    *p = c->s_latent.as<float>();
  });
}

// ---------------------------------------------------------------- resident audio + video denoise session
int ltx_av_denoise_begin(ltx_ctx* c, const float* video_noise, const float* audio_noise, int F, int H, int W, int Ta, float sigma0,
                         const void* video_context, const void* audio_context, ltx_dtype context_dtype, const int32_t* mask,
                         const void* neg_video_context, const void* neg_audio_context, const int32_t* neg_mask, int S) {
  return guarded(c, [&] {
    av_precision_check(c);
    LTX_CHECK(video_noise && audio_noise && video_context && audio_context && F > 0 && H > 0 && W > 0 && Ta > 0 && S > 0,
              LTX_ERR_INVALID_ARGUMENT, "bad av_denoise_begin arguments");
    LTX_CHECK((neg_video_context == nullptr) == (neg_audio_context == nullptr), LTX_ERR_INVALID_ARGUMENT,
              "the negative contexts come as a pair");
    LTX_CHECK(c->av.ready, LTX_ERR_WEIGHTS, "dual audio/video weights not loaded / finalized");
    const ltx_config& g = c->cfg;
    LTX_CHECK(g.in_channels == g.out_channels, LTX_ERR_INVALID_CONFIGURATION, "in/out channels must match");
    const size_t n = static_cast<size_t>(g.in_channels) * F * H * W, na = static_cast<size_t>(Ta) * c->av.Cin;
    session_resize(c, F, H, W);
    c->s_S = S; c->s_Ta = Ta;
    c->s_ctx_dtype = context_dtype;
    h2d(c, c->s_latent, video_noise, n * 4);
    h2d(c, c->s_alat, audio_noise, na * 4);
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * (n + na), 2);
      launch_scale_f32(c->s_latent.as<float>(), sigma0, static_cast<int64_t>(n), c->stream);   // P/LTXPipeline.swift:1255-1259
      launch_scale_f32(c->s_alat.as<float>(), sigma0, static_cast<int64_t>(na), c->stream);
    }
    const size_t cbytes = static_cast<size_t>(S) * g.caption_channels * dsize(context_dtype);
    h2d(c, c->s_ctx_pos, video_context, cbytes);
    h2d(c, c->s_actx_pos, audio_context, cbytes);
    c->s_has_mask_pos = mask != nullptr;
    if (mask) h2d(c, c->s_mask_pos, mask, static_cast<size_t>(S) * 4);
    c->s_has_neg = neg_video_context != nullptr;
    if (c->s_has_neg) {
      h2d(c, c->s_ctx_neg, neg_video_context, cbytes);
      h2d(c, c->s_actx_neg, neg_audio_context, cbytes);
      c->s_has_mask_neg = neg_mask != nullptr;
      if (neg_mask) h2d(c, c->s_mask_neg, neg_mask, static_cast<size_t>(S) * 4);
      // inputs of the batched guidance forward: both prompts of each stream in one [2, S, Cc] buffer, one [2, S] mask when
      // either prompt has one (all ones for the other), room for two latents / velocities of each stream
      c->s_ctx_pair.reserve(2 * cbytes);
      c->s_actx_pair.reserve(2 * cbytes);
      LTX_CUDA(cudaMemcpyAsync(c->s_ctx_pair.ptr, c->s_ctx_pos.ptr, cbytes, cudaMemcpyDeviceToDevice, c->stream));
      LTX_CUDA(cudaMemcpyAsync(c->s_ctx_pair.as<uint8_t>() + cbytes, c->s_ctx_neg.ptr, cbytes, cudaMemcpyDeviceToDevice, c->stream));
      LTX_CUDA(cudaMemcpyAsync(c->s_actx_pair.ptr, c->s_actx_pos.ptr, cbytes, cudaMemcpyDeviceToDevice, c->stream));
      LTX_CUDA(cudaMemcpyAsync(c->s_actx_pair.as<uint8_t>() + cbytes, c->s_actx_neg.ptr, cbytes, cudaMemcpyDeviceToDevice, c->stream));
      if (mask || neg_mask) {
        std::vector<int32_t> pm(static_cast<size_t>(2) * S, 1);
        if (mask) memcpy(pm.data(), mask, static_cast<size_t>(S) * 4);
        if (neg_mask) memcpy(pm.data() + S, neg_mask, static_cast<size_t>(S) * 4);
        h2d(c, c->s_mask_pair, pm.data(), pm.size() * 4);
        LTX_CUDA(cudaStreamSynchronize(c->stream));   // pm goes out of scope
      }
      c->s_tok.reserve(2 * n * 2);
      c->vel.reserve(2 * n * 4);
      c->s_alat_pair.reserve(2 * na * 4);
    }
    c->s_avc.reserve((c->s_has_neg ? 2 : 1) * na * 4);   // batched: [conditional | unconditional] audio velocities
    c->s_avu.reserve(na * 4);
    c->scratch.reserve(64 * sizeof(double));
    c->s_serial += 2;
    dit_clear_caches(c);
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_av_denoise_step(ltx_ctx* c, const ltx_step_params* p) {
  return guarded(c, [&] {
    av_precision_check(c);
    LTX_CHECK(p != nullptr && c->s_F > 0 && c->s_Ta > 0, LTX_ERR_INVALID_ARGUMENT, "av_denoise_step before av_denoise_begin");
    LTX_CHECK(p->sigma > 0.f, LTX_ERR_INVALID_ARGUMENT, "sigma must be > 0");
    LTX_CHECK(p->stg_scale == 0.f && p->ge_gamma == 0.f, LTX_ERR_UNSUPPORTED,
              "the audio + video loop has no STG / GE terms (Pipeline/LTXPipeline.swift:1300-1404)");
    const ltx_config& g = c->cfg;
    const int C = g.in_channels, F = c->s_F, H = c->s_H, W = c->s_W, S = c->s_S, Ta = c->s_Ta;
    const int T = F * H * W;
    const size_t n = static_cast<size_t>(C) * T, na = static_cast<size_t>(Ta) * c->av.Cin;
    cudaStream_t st = c->stream;
    {
      ProfScope ps(c, PROF_OTHER, 0.0, 6.0 * n);
      launch_patchify(c->s_latent.as<float>(), c->s_tok.as<bf16>(), nullptr, C, T, st);
    }
    const bool use_cfg = p->cfg_scale > 1.0f && c->s_has_neg;
    // Conditional + unconditional as ONE B = 2 forward on one GPU (as ltx_denoise_step does): the audio stream's Linears read
    // their weights once for both prompts and the video stream's GEMMs / attention fill their waves better.  Item 0 is the
    // conditional pass; per item the arithmetic is that of the separate passes.
    const bool batched = batched_cfg_env() && use_cfg && c->dist.groups == 1 && !(c->dist.comm_world && c->dist.sp > 1) &&
                         !p->disable_batched_cfg;
    const int nb = batched ? 2 : 1;
    const float sig2[2] = {p->sigma, p->sigma};   // one sigma per item, for both streams
    LTX_CUDA(cudaMemcpyAsync(c->s_sigma.ptr, sig2, 8, cudaMemcpyHostToDevice, st));
    // image-to-video (:1293-1298): video timesteps sigma * (1 - conditioningMask) per token; the audio stream keeps sigma
    const bool i2v = p->i2v_frame0_conditioned != 0;
    const float* ts_dev = c->s_sigma.as<float>();
    if (i2v) {
      c->s_ts.reserve(static_cast<size_t>(nb) * T * 4);
      ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * nb * T);
      launch_fill_token_timesteps(c->s_ts.as<float>(), nb * T, T, H * W, c->s_sigma.as<float>(), st);
      ts_dev = c->s_ts.as<float>();
    }
    const uint64_t key_pos = 0x6000000000000000ull + c->s_serial, key_neg = key_pos + 1;
    const uint64_t key_pair = 0x6800000000000000ull + c->s_serial;
    auto pass = [&](bool neg, float* v_lat, float* a_vel) {
      const int32_t* mk = neg ? (c->s_has_mask_neg ? c->s_mask_neg.as<int32_t>() : nullptr)
                              : (c->s_has_mask_pos ? c->s_mask_pos.as<int32_t>() : nullptr);
      dit_av_forward_dev(c, c->s_tok.ptr, LTX_BF16, c->s_alat.ptr, LTX_F32, neg ? c->s_ctx_neg.ptr : c->s_ctx_pos.ptr,
                         neg ? c->s_actx_neg.ptr : c->s_actx_pos.ptr, c->s_ctx_dtype, ts_dev, i2v ? 1 : 0, c->s_sigma.as<float>(), mk,
                         mk, 1, T, Ta, S, F, H, W, neg ? key_neg : key_pos, c->vel.as<float>(), a_vel);
      ProfScope ps(c, PROF_OTHER, 0.0, 8.0 * n);
      launch_unpatchify(c->vel.as<float>(), v_lat, C, T, st);
    };
    float* avu = c->s_avu.as<float>();
    if (batched) {
      bf16* tok = c->s_tok.as<bf16>();
      float* alat2 = c->s_alat_pair.as<float>();
      LTX_CUDA(cudaMemcpyAsync(tok + n, tok, n * 2, cudaMemcpyDeviceToDevice, st));   // the same latents under both prompts
      LTX_CUDA(cudaMemcpyAsync(alat2, c->s_alat.ptr, na * 4, cudaMemcpyDeviceToDevice, st));
      LTX_CUDA(cudaMemcpyAsync(alat2 + na, c->s_alat.ptr, na * 4, cudaMemcpyDeviceToDevice, st));
      const int32_t* mk = (c->s_has_mask_pos || c->s_has_mask_neg) ? c->s_mask_pair.as<int32_t>() : nullptr;
      avu = c->s_avc.as<float>() + na;
      dit_av_forward_dev(c, tok, LTX_BF16, alat2, LTX_F32, c->s_ctx_pair.ptr, c->s_actx_pair.ptr, c->s_ctx_dtype, ts_dev, i2v ? 1 : 0,
                         c->s_sigma.as<float>(), mk, mk, 2, T, Ta, S, F, H, W, key_pair, c->vel.as<float>(), c->s_avc.as<float>());
      ProfScope ps(c, PROF_OTHER, 0.0, 16.0 * n, 2);
      launch_unpatchify(c->vel.as<float>(), c->s_vc.as<float>(), C, T, st);
      launch_unpatchify(c->vel.as<float>() + n, c->s_vu.as<float>(), C, T, st);
    } else {
      pass(false, c->s_vc.as<float>(), c->s_avc.as<float>());
      if (use_cfg) pass(true, c->s_vu.as<float>(), avu);
    }
    // video: applyCFG (+ rescale) + scheduler.step, frame 0 untouched in the image-to-video mode (:1364-1391)
    GuidedEulerArgs a;
    a.latent = c->s_latent.as<float>(); a.v_cond = c->s_vc.as<float>();
    a.v_uncond = use_cfg ? c->s_vu.as<float>() : nullptr;
    a.v_stg = nullptr; a.v_prev = nullptr; a.use_prev = 0;
    a.v_out = nullptr; a.n = n; a.cfg = use_cfg ? p->cfg_scale : 1.0f; a.phi = use_cfg ? p->rescale_phi : 0.0f; a.stg = 0.f;
    a.ge_gamma = 0.f; a.sigma = p->sigma; a.sigma_next = p->sigma_next; a.scratch = c->scratch.as<double>();
    if (i2v) { a.period = static_cast<size_t>(T); a.frozen = static_cast<size_t>(H) * W; }
    ProfScope ps(c, PROF_OTHER, 0.0, 4.0 * n * (3.0 + (use_cfg ? 1.0 : 0.0)) + 4.0 * na * (3.0 + (use_cfg ? 1.0 : 0.0)),
                 ((use_cfg && p->rescale_phi > 0.f) ? 2 : 1) + 1);
    launch_guided_euler(a, st);
    // audio: applyCFG + a += (sigma' - sigma) v (:1402)
    const float dt = static_cast<float>(static_cast<double>(p->sigma_next) - static_cast<double>(p->sigma));
    launch_audio_cfg_euler(c->s_alat.as<float>(), c->s_avc.as<float>(), use_cfg ? avu : nullptr, p->cfg_scale, dt,
                           static_cast<int64_t>(na), st);
  });
}

int ltx_av_denoise_get_latents(ltx_ctx* c, float* video_out, float* audio_out) {
  return guarded(c, [&] {
    LTX_CHECK(c->s_F > 0 && c->s_Ta > 0, LTX_ERR_INVALID_ARGUMENT, "no audio + video denoise session");
    const size_t n = static_cast<size_t>(c->cfg.in_channels) * c->s_F * c->s_H * c->s_W;
    if (video_out) LTX_CUDA(cudaMemcpyAsync(video_out, c->s_latent.ptr, n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (audio_out)
      LTX_CUDA(cudaMemcpyAsync(audio_out, c->s_alat.ptr, static_cast<size_t>(c->s_Ta) * c->av.Cin * 4, cudaMemcpyDeviceToHost,
                               c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

// ---------------------------------------------------------------- VAE
int ltx_vae_decode_dev(ltx_ctx* c, const float* latent, int Fp, int Hp, int Wp, float timestep, const float* decode_noise,
                       int causal, float* out_frames) {
  return guarded(c, [&] { vae_decode_dev(c, latent, Fp, Hp, Wp, timestep, decode_noise, causal, out_frames); });
}

int ltx_vae_decode(ltx_ctx* c, const float* latent, int Fp, int Hp, int Wp, float timestep, const float* decode_noise,
                   int causal, float* out_frames) {
  return guarded(c, [&] {
    LTX_CHECK(latent && out_frames && Fp > 0 && Hp > 0 && Wp > 0, LTX_ERR_INVALID_ARGUMENT, "bad vae_decode arguments");
    const size_t n = static_cast<size_t>(c->cfg.vae_latent_channels) * Fp * Hp * Wp;
    h2d(c, c->v_lat, latent, n * 4);
    const float* nz = nullptr;
    if (timestep >= 0.f) {
      LTX_CHECK(decode_noise != nullptr, LTX_ERR_INVALID_ARGUMENT, "decode_noise is required when timestep >= 0");
      h2d(c, c->v_noise, decode_noise, n * 4);
      nz = c->v_noise.as<float>();
    }
    const size_t fo = static_cast<size_t>(8 * (Fp - 1) + 1) * (32 * Hp) * (32 * Wp) * 3;
    c->v_frames.reserve(fo * 4);
    vae_decode_dev(c, c->v_lat.as<float>(), Fp, Hp, Wp, timestep, nz, causal, c->v_frames.as<float>());
    LTX_CUDA(cudaMemcpyAsync(out_frames, c->v_frames.ptr, fo * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_vae_tiled_frames(int Fp, int tile_size, int tile_overlap) {
  if (Fp <= 0 || (tile_size > 0 && Fp > tile_size && (tile_overlap < 0 || tile_overlap >= tile_size))) return -1;
  return vae_tiled_frames(Fp, tile_size, tile_overlap);
}

int ltx_vae_decode_tiled_dev(ltx_ctx* c, const float* latent, int Fp, int Hp, int Wp, float timestep, const float* decode_noise,
                             int causal, int tile_size, int tile_overlap, float* out_frames, int* out_num_frames) {
  return guarded(c, [&] {
    const int n = vae_decode_tiled_dev(c, latent, Fp, Hp, Wp, timestep, decode_noise, causal, tile_size, tile_overlap, out_frames);
    if (out_num_frames) *out_num_frames = n;
  });
}

int ltx_vae_decode_tiled(ltx_ctx* c, const float* latent, int Fp, int Hp, int Wp, float timestep, const float* decode_noise,
                         int causal, int tile_size, int tile_overlap, float* out_frames, int* out_num_frames) {
  return guarded(c, [&] {
    LTX_CHECK(latent && out_frames && Fp > 0 && Hp > 0 && Wp > 0, LTX_ERR_INVALID_ARGUMENT, "bad vae_decode arguments");
    const int nf = ltx_vae_tiled_frames(Fp, tile_size, tile_overlap);
    LTX_CHECK(nf > 0, LTX_ERR_INVALID_ARGUMENT, "temporal tile overlap must be in [0, tile size)");
    const size_t n = static_cast<size_t>(c->cfg.vae_latent_channels) * Fp * Hp * Wp;
    h2d(c, c->v_lat, latent, n * 4);
    const float* nz = nullptr;
    if (timestep >= 0.f) {
      LTX_CHECK(decode_noise != nullptr, LTX_ERR_INVALID_ARGUMENT, "decode_noise is required when timestep >= 0");
      h2d(c, c->v_noise, decode_noise, n * 4);
      nz = c->v_noise.as<float>();
    }
    const size_t fe = static_cast<size_t>(32 * Hp) * (32 * Wp) * 3;
    c->v_frames.reserve(static_cast<size_t>(nf) * fe * 4);
    const int got = vae_decode_tiled_dev(c, c->v_lat.as<float>(), Fp, Hp, Wp, timestep, nz, causal, tile_size, tile_overlap,
                                         c->v_frames.as<float>());
    LTX_CHECK(got == nf, LTX_ERR_CUDA, "tiled decode frame count mismatch");
    if (out_num_frames) *out_num_frames = got;
    LTX_CUDA(cudaMemcpyAsync(out_frames, c->v_frames.ptr, static_cast<size_t>(got) * fe * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

// ---------------------------------------------------------------- VAE encoder, latent upscaler, AdaIN, re-noise
int ltx_vae_encode_dev(ltx_ctx* c, const float* pixels, int T, int H, int W, int normalize, float* latent_out) {
  return guarded(c, [&] { vae_encode_dev(c, pixels, T, H, W, normalize, latent_out); });
}

int ltx_vae_encode(ltx_ctx* c, const float* pixels, int T, int H, int W, int normalize, float* latent_out) {
  return guarded(c, [&] {
    LTX_CHECK(pixels && latent_out && T >= 1 && H >= 64 && W >= 64 && H % 32 == 0 && W % 32 == 0, LTX_ERR_INVALID_ARGUMENT,
              "bad vae_encode arguments");
    const size_t n_in = static_cast<size_t>(3) * T * H * W;
    const size_t n_out = static_cast<size_t>(c->cfg.vae_latent_channels) * ((T + 7) / 8) * (H / 32) * (W / 32);
    h2d(c, c->u_in, pixels, n_in * 4);
    c->u_out.reserve(n_out * 4);
    vae_encode_dev(c, c->u_in.as<float>(), T, H, W, normalize, c->u_out.as<float>());
    LTX_CUDA(cudaMemcpyAsync(latent_out, c->u_out.ptr, n_out * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_upscale_latent_dev(ltx_ctx* c, const float* latent, int F, int H, int W, float* out) {
  return guarded(c, [&] { upscale_latent_dev(c, latent, F, H, W, out); });
}

int ltx_upscale_latent(ltx_ctx* c, const float* latent, int F, int H, int W, float* out) {
  return guarded(c, [&] {
    LTX_CHECK(latent && out && F >= 1 && H > 1 && W > 1, LTX_ERR_INVALID_ARGUMENT, "bad upscale_latent arguments");
    const size_t n = static_cast<size_t>(c->cfg.vae_latent_channels) * F * H * W;
    h2d(c, c->u_in, latent, n * 4);
    c->u_out.reserve(4 * n * 4);
    upscale_latent_dev(c, c->u_in.as<float>(), F, H, W, c->u_out.as<float>());
    LTX_CUDA(cudaMemcpyAsync(out, c->u_out.ptr, 4 * n * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

int ltx_adain_filter_dev(ltx_ctx* c, float* latent, size_t n_per_channel, const float* reference, size_t n_ref_per_channel,
                         int channels, float factor) {
  return guarded(c, [&] {
    adain_filter_dev(c, latent, static_cast<int64_t>(n_per_channel), reference, static_cast<int64_t>(n_ref_per_channel), channels,
                     factor);
  });
}

int ltx_adain_filter(ltx_ctx* c, float* latent, size_t n_per_channel, const float* reference, size_t n_ref_per_channel, int channels,
                     float factor) {
  return guarded(c, [&] {
    LTX_CHECK(latent && reference && channels > 0, LTX_ERR_INVALID_ARGUMENT, "bad adain arguments");
    h2d(c, c->u_in, latent, n_per_channel * channels * 4);
    h2d(c, c->u_ref, reference, n_ref_per_channel * channels * 4);
    adain_filter_dev(c, c->u_in.as<float>(), static_cast<int64_t>(n_per_channel), c->u_ref.as<float>(),
                     static_cast<int64_t>(n_ref_per_channel), channels, factor);
    LTX_CUDA(cudaMemcpyAsync(latent, c->u_in.ptr, n_per_channel * channels * 4, cudaMemcpyDeviceToHost, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
  });
}

// ---------------------------------------------------------------- diagnostic single-kernel ops
int ltx_op_gemm(ltx_ctx* c, const void* A, const void* B, const float* bias, void* C, int M, int N, int K, int mode,
                int force_bn) {
  return guarded(c, [&] {
    GemmEpi e;
    e.mode = mode; e.out = C; e.ldo = N; e.bias = bias;
    LTX_CHECK(mode == EPI_BF16 || mode == EPI_GELU_BF16 || mode == EPI_F32 || mode == EPI_SILU_BF16, LTX_ERR_INVALID_ARGUMENT, "bad mode");
    if (force_bn == -1) {   // the weight-streaming kernel for M <= 32, or an error: never a silent switch to the tile kernel
      LTX_CHECK(gemm_skinny_eligible(K, K, M, N, K, e, 0), LTX_ERR_INVALID_ARGUMENT, "shape not eligible for the skinny GEMM");
      launch_gemm_skinny(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, M, N, K, e, c->stream);
    } else if (force_bn == -2 || force_bn == -3) {   // the swap-AB weight-streaming kernel (M <= 512): -2 with split-K workspace, -3 without
      LTX_CHECK(gemm_swapab_eligible(K, K, M, N, K, e), LTX_ERR_INVALID_ARGUMENT, "shape not eligible for the swap-AB GEMM");
      if (force_bn == -2) gemm_attach_workspace(c, e);
      launch_gemm_swapab(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, M, N, K, e, c->stream);
    } else {
      launch_gemm(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, M, N, K, e, c->stream, force_bn);
    }
    c->launches++;
  });
}

int ltx_op_gemm_blocked(ltx_ctx* c, const void* A, const void* B, const float* bias, void* plain_out, void* blocks_out, int M, int N,
                        int K, int col_from, int col_block, int64_t block_stride, int force_bn) {
  return guarded(c, [&] {
    LTX_CHECK(col_block > 0 && col_from >= 0 && col_from < N && (N - col_from) % col_block == 0 && (N - col_from) / col_block <= LTX_MAX_PEERS,
              LTX_ERR_INVALID_ARGUMENT, "bad column blocking");
    GemmEpi e;
    e.mode = EPI_BF16; e.out = plain_out; e.ldo = col_from > 0 ? col_from : col_block; e.bias = bias;
    e.col_block = col_block; e.col_block_from = col_from; e.blocked_ld = col_block; e.use_col_ptrs = 1;
    for (int j = 0; j < (N - col_from) / col_block; ++j)   // one base per block, as the peer-memory path hands out one per rank
      e.col_ptrs.p[j] = reinterpret_cast<bf16*>(blocks_out) + static_cast<int64_t>(j) * block_stride;
    if (force_bn == -2) {
      gemm_attach_workspace(c, e);
      launch_gemm_swapab(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, M, N, K, e, c->stream);
    } else {
      launch_gemm(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, M, N, K, e, c->stream, force_bn);
    }
    c->launches++;
  });
}

int ltx_op_gemm_resid(ltx_ctx* c, const void* A, const void* B, const float* bias, float* x, const float* gate_a,
                      const float* gate_b, void* shadow, int M, int N, int K, float scale) {
  return guarded(c, [&] {
    GemmEpi e;
    e.mode = EPI_GATE_RESID; e.resid = x; e.ldr = N; e.bias = bias; e.gate_a = gate_a; e.gate_b = gate_b; e.gate_ld = 0;
    e.rows_per_gate = M > 0 ? M : 1; e.shadow = reinterpret_cast<bf16*>(shadow); e.lds = N; e.scale = scale;
    if (M > 32 && M <= 512) gemm_attach_workspace(c, e);   // as the DiT forward does for few-row problems (swap-AB kernel)
    // LTX_GEMM_FORCE_BN: a launch_gemm force_bn for this op, which has no argument for it (tools/gemm_bench.py's sweeps)
    const char* fb = getenv("LTX_GEMM_FORCE_BN");
    launch_gemm(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, M, N, K, e, c->stream, fb ? atoi(fb) : 0, 0, 0,
                32 /* M <= 32: the weight-streaming kernel, as on the dual model's audio stream */);
    c->launches++;
  });
}

int ltx_op_gemm_skinny(ltx_ctx* c, const void* A, const void* B, const float* bias, void* out, float* x, const float* gate_a,
                       const float* gate_b, int rows_per_gate, int M, int N, int K, int mode, int items, int64_t vt_item_ld) {
  return guarded(c, [&] {
    LTX_CHECK(A && B && (mode == EPI_GATE_RESID ? x != nullptr : out != nullptr) && (items == 1 || items == 2) &&
                  (vt_item_ld == 0 || (M % items == 0 && vt_item_ld >= M / items)),
              LTX_ERR_INVALID_ARGUMENT, "bad skinny GEMM arguments");
    LTX_CHECK(mode >= EPI_BF16 && mode <= EPI_SILU_BF16 && (vt_item_ld == 0 || mode == EPI_BF16), LTX_ERR_INVALID_ARGUMENT, "bad mode");
    GemmEpi e;
    e.mode = mode; e.bias = bias;
    if (mode == EPI_GATE_RESID) {
      e.resid = x; e.ldr = N; e.gate_a = gate_a; e.gate_b = gate_b; e.gate_ld = N;
      e.rows_per_gate = rows_per_gate > 0 ? rows_per_gate : M;
    } else if (vt_item_ld > 0) {
      e.out = out; e.ldo = items * vt_item_ld; e.transpose_out = 1;
      if (items > 1) { e.t_item_rows = M / items; e.t_item_ld = vt_item_ld; }
    } else {
      e.out = out; e.ldo = N;
    }
    LTX_CHECK(gemm_skinny_eligible(K, K, M, N, K, e, 0, 32 * items), LTX_ERR_INVALID_ARGUMENT, "shape not eligible for the skinny GEMM");
    launch_gemm(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), K, M, N, K, e, c->stream, 0, 0, 0, 32 * items);
    c->launches++;
  });
}

int ltx_op_quantize(ltx_ctx* c, const void* w_bf16, int N, int K, int bits, void* q_out, float* scales_out, float* biases_out) {
  return guarded(c, [&] {
    launch_quantize(reinterpret_cast<const bf16*>(w_bf16), N, K, bits, reinterpret_cast<uint8_t*>(q_out), scales_out, biases_out,
                    c->stream);
    c->launches++;
  });
}

int ltx_op_dequantize(ltx_ctx* c, const void* q, const float* scales, const float* biases, int N, int K, int bits, void* w_bf16) {
  return guarded(c, [&] {
    QuantW W;
    W.q = reinterpret_cast<const uint8_t*>(q); W.scales = scales; W.biases = biases; W.bits = bits; W.n = N; W.k = K;
    launch_dequantize(W, reinterpret_cast<bf16*>(w_bf16), c->stream);
    c->launches++;
  });
}

int ltx_op_gemm_q(ltx_ctx* c, const void* A, const void* q, const float* scales, const float* biases, int bits, const float* bias,
                  void* C, int M, int N, int K, int mode, int force_bn) {
  return guarded(c, [&] {
    LTX_CHECK(mode == EPI_BF16 || mode == EPI_GELU_BF16 || mode == EPI_F32, LTX_ERR_INVALID_ARGUMENT, "bad mode");
    QuantW W;
    W.q = reinterpret_cast<const uint8_t*>(q); W.scales = scales; W.biases = biases; W.bits = bits; W.n = N; W.k = K;
    GemmEpi e;
    e.mode = mode; e.out = C; e.ldo = N; e.bias = bias;
    launch_gemm_q(reinterpret_cast<const bf16*>(A), K, W, M, N, K, e, c->stream, force_bn);
    c->launches++;
  });
}

int ltx_op_quantize_fp8(ltx_ctx* c, const void* x_bf16, int M, int K, int64_t ld, void* codes, float* scales) {
  return guarded(c, [&] {
    LTX_CHECK(x_bf16 && codes && scales, LTX_ERR_INVALID_ARGUMENT, "null tensor");
    launch_quantize_rows_fp8(reinterpret_cast<const bf16*>(x_bf16), ld, M, K, reinterpret_cast<uint8_t*>(codes), scales, c->stream);
    c->launches++;
  });
}

int ltx_op_gemm_fp8(ltx_ctx* c, const void* Aq, const float* sa, const void* Bq, const float* sb, const float* bias, void* C, int M,
                    int N, int K, int mode, int force_bn) {
  return guarded(c, [&] {
    LTX_CHECK(Aq && sa && Bq && sb && C, LTX_ERR_INVALID_ARGUMENT, "null tensor");
    LTX_CHECK(mode == EPI_BF16 || mode == EPI_GELU_BF16 || mode == EPI_F32 || mode == EPI_SILU_BF16, LTX_ERR_INVALID_ARGUMENT, "bad mode");
    GemmEpi e;
    e.mode = mode; e.out = C; e.ldo = N; e.bias = bias;
    launch_gemm_fp8(reinterpret_cast<const uint8_t*>(Aq), K, sa, reinterpret_cast<const uint8_t*>(Bq), K, sb, M, N, K, e, c->stream,
                    force_bn);
    c->launches++;
  });
}

int ltx_op_gemm_fp8_ex(ltx_ctx* c, const void* Aq, const float* sa, const void* Bq, const float* sb, const float* bias, void* C,
                       void* Ct, int tsplit_col, int64_t ldt, float* x, const float* gate_a, const float* gate_b, void* shadow,
                       int M, int N, int K, int force_bn) {
  return guarded(c, [&] {
    LTX_CHECK(Aq && sa && Bq && sb && (x != nullptr) != (C != nullptr), LTX_ERR_INVALID_ARGUMENT,
              "bad FP8 GEMM arguments: one of C (bf16, with optional V^T split) or x (gate * residual)");
    GemmEpi e;
    e.bias = bias;
    if (x) {
      e.mode = EPI_GATE_RESID; e.resid = x; e.ldr = N; e.gate_a = gate_a; e.gate_b = gate_b; e.gate_ld = 0;
      e.rows_per_gate = M; e.shadow = reinterpret_cast<bf16*>(shadow); e.lds = N;
    } else {
      e.mode = EPI_BF16; e.out = C; e.ldo = tsplit_col > 0 ? tsplit_col : N;
      if (tsplit_col > 0) { e.tsplit_col = tsplit_col; e.out_t = reinterpret_cast<bf16*>(Ct); e.ldt = ldt; }
    }
    launch_gemm_fp8(reinterpret_cast<const uint8_t*>(Aq), K, sa, reinterpret_cast<const uint8_t*>(Bq), K, sb, M, N, K, e, c->stream,
                    force_bn);
    c->launches++;
  });
}

int ltx_op_attention(ltx_ctx* c, const void* Q, const void* K, const void* Vt, int64_t ldvb, const float* key_bias, void* O,
                     int B, int H, int Nq, int Nk, float scale) {
  return guarded(c, [&] {
    const int D = H * 128;
    launch_attention(reinterpret_cast<const bf16*>(Q), D, reinterpret_cast<const bf16*>(K), D,
                     reinterpret_cast<const bf16*>(Vt), ldvb, key_bias, reinterpret_cast<bf16*>(O), D, B, H, Nq, Nk, D, scale,
                     c->stream);
    c->launches++;
  });
}

int ltx_op_attention_hd(ltx_ctx* c, const void* Q, const void* K, const void* Vt, int64_t ldvb, const float* key_bias, void* O,
                        int B, int H, int head_dim, int Nq, int Nk, float scale) {
  return guarded(c, [&] {
    LTX_CHECK(head_dim == 128 || head_dim == 64, LTX_ERR_UNSUPPORTED, "head_dim must be 128 or 64");
    const int D = H * head_dim;
    launch_attention(reinterpret_cast<const bf16*>(Q), D, reinterpret_cast<const bf16*>(K), D,
                     reinterpret_cast<const bf16*>(Vt), ldvb, key_bias, reinterpret_cast<bf16*>(O), D, B, H, Nq, Nk, D, scale,
                     c->stream);
    c->launches++;
  });
}

int ltx_op_attention_blocks(ltx_ctx* c, const void* Q, const void* K, const void* Vt, int64_t ldvb, int H, int Nq, int Nk,
                            float scale, void* const* o_blocks, int n_blocks, int rows_per_block) {
  return guarded(c, [&] {
    LTX_CHECK(o_blocks && n_blocks >= 1 && n_blocks <= LTX_MAX_PEERS && rows_per_block > 0 && n_blocks * rows_per_block >= Nq,
              LTX_ERR_INVALID_ARGUMENT, "bad output blocks");
    const int D = H * 128;
    PeerTable t = {};
    for (int i = 0; i < n_blocks; ++i) t.p[i] = o_blocks[i];
    launch_attention(reinterpret_cast<const bf16*>(Q), D, reinterpret_cast<const bf16*>(K), D, reinterpret_cast<const bf16*>(Vt), ldvb,
                     nullptr, reinterpret_cast<bf16*>(o_blocks[0]), D, 1, H, Nq, Nk, D, scale, c->stream, &t, rows_per_block);
    c->launches++;
  });
}

int ltx_op_rmsnorm_mod(ltx_ctx* c, const float* x, void* out_bf16, int M, int D, const float* tbl_shift,
                       const float* tbl_scale, const float* ada_shift, const float* ada_scale, float eps, int layernorm) {
  return guarded(c, [&] {
    launch_rmsnorm_mod(x, reinterpret_cast<bf16*>(out_bf16), M, D, tbl_shift, tbl_scale, ada_shift, ada_scale, 0, M, eps,
                       layernorm, c->stream);
    c->launches++;
  });
}

int ltx_op_qknorm_rope(ltx_ctx* c, void* x_bf16, int M, int D, const float* w, const float* cos_tab, const float* sin_tab,
                       int rows_per_rope, float eps) {
  return guarded(c, [&] {
    launch_qknorm_rope(reinterpret_cast<bf16*>(x_bf16), D, M, D, w, cos_tab, sin_tab, rows_per_rope, eps, c->stream);
    c->launches++;
  });
}

int ltx_conv3d_plan(int T, int H, int W, int Cin, int Cout, int mode, int ntaps, int sm_count, int32_t* plan7) {
  // host-only: no context, no device
  if (plan7 == nullptr || T <= 0 || H <= 1 || W <= 1 || Cin <= 0 || Cout <= 0 || (ntaps != 27 && ntaps != 9) || sm_count <= 0 || mode < 0 ||
      mode > 4)
    return LTX_ERR_INVALID_ARGUMENT;
  const ConvPlan p = conv3d_plan(T, H, W, Cin, Cout, mode, ntaps, /*scratch_ok=*/true, sm_count, conv3d_pair_default(), conv3d_slab_default());
  plan7[0] = p.bn; plan7[1] = p.pair; plan7[2] = p.slab; plan7[3] = p.bt; plan7[4] = p.bh; plan7[5] = p.bw; plan7[6] = p.ksplit;
  return LTX_OK;
}

int ltx_op_conv3d(ltx_ctx* c, const float* x, const void* w, const float* bias, float* out, int T, int H, int W, int Cin,
                  int Cout, int causal) {
  return guarded(c, [&] {
    c->v_pad.reserve(static_cast<size_t>(T + 2) * (H + 2) * (W + 2) * Cin * 2);
    launch_vae_prep(x, c->v_pad.as<bf16>(), T, H, W, Cin, 0, nullptr, nullptr, causal, c->stream);
    ConvEpi e;
    e.mode = 0; e.out = out; e.bias = bias; e.resid = nullptr; e.Cin = Cin;
    float* scratch = nullptr;
    const size_t slab3 = static_cast<size_t>(3) * T * H * W * Cout * 4;
    if (conv3d_wants_tap_split(H, W, Cin, Cout)) {
      c->v_split.reserve(slab3);
      scratch = c->v_split.as<float>();
    }
    launch_conv3d(c->v_pad.as<bf16>(), reinterpret_cast<const bf16*>(w), T, H, W, Cin, Cout, e, c->stream, 27, scratch, scratch ? slab3 : 0);
    c->launches += 2;
  });
}

int ltx_op_vae_prep(ltx_ctx* c, const float* x, void* out_pad, int T, int H, int W, int C, int mode, const float* a, const float* b,
                    int pad) {
  return guarded(c, [&] {
    launch_vae_prep(x, reinterpret_cast<bf16*>(out_pad), T, H, W, C, mode, a, b, pad, c->stream);
    c->launches++;
  });
}

int ltx_op_vae_halo_fill(ltx_ctx* c, void* vol, int T, int H, int W, int C, int pad) {
  return guarded(c, [&] {
    launch_vae_halo_fill(reinterpret_cast<bf16*>(vol), T, H, W, C, pad, c->stream);
    c->launches++;
  });
}

int ltx_op_conv3d_epi(ltx_ctx* c, const void* x_pad, const void* w, const float* bias, int T, int H, int W, int Cin, int Cout,
                      int ntaps, int mode, float* out, const float* resid, int t_shift, int no_clip, void* next_pad,
                      const float* next_scale, const float* next_shift, int next_tshift) {
  return guarded(c, [&] {
    ConvEpi e;
    e.mode = mode; e.out = out; e.bias = bias; e.resid = resid; e.Cin = Cin; e.t_shift = t_shift; e.no_clip = no_clip;
    e.next_pad = reinterpret_cast<bf16*>(next_pad); e.next_scale = next_scale; e.next_shift = next_shift; e.next_tshift = next_tshift;
    // the split-K scratch as vae_conv reserves it, so that every shape gets the plan the decoder gets
    float* scratch = nullptr;
    const size_t slab3 = static_cast<size_t>(3) * T * H * W * Cout * 4;
    if (mode == 0 && ntaps == 27 && conv3d_wants_tap_split(H, W, Cin, Cout)) {
      c->v_split.reserve(slab3);
      scratch = c->v_split.as<float>();
    }
    launch_conv3d(reinterpret_cast<const bf16*>(x_pad), reinterpret_cast<const bf16*>(w), T, H, W, Cin, Cout, e, c->stream, ntaps,
                  scratch, scratch ? slab3 : 0);
    c->launches++;
  });
}

}  // extern "C"
