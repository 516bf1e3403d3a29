// Weight ingestion for libltxcuda: host tensors under the reference's post-mapping key names
// (Utils/ModelDownloader.swift:756-899) are copied to the device as bf16 (matrices / conv kernels, mirroring the
// loader's fp32->bf16 cast at :1005-1012) or fp32 (biases, norm weights, scale-shift tables).  Transformer Linears of a
// scaled-FP8 checkpoint (e4m3 codes + scales) are decoded on the device to the same storage, or kept as codes in FP8 mode.
#include <cuda_fp16.h>
#include <cuda_fp8.h>

#include <cstring>
#include <type_traits>

#include "ctx.h"

namespace ltx {

namespace {

template <typename S>
__device__ __forceinline__ float to_f32(S v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<bf16>(bf16 v) { return __bfloat162float(v); }
template <>
__device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }

template <typename S, typename D>
__global__ void convert_kernel(const S* __restrict__ in, D* __restrict__ out, int64_t n) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float v = to_f32<S>(in[i]);
    if (sizeof(D) == 2)
      reinterpret_cast<bf16*>(out)[i] = __float2bfloat16(v);
    else
      reinterpret_cast<float*>(out)[i] = v;
  }
}

template <typename S>
void convert_to(const void* src, void* dst, int dst_dtype, int64_t n, cudaStream_t s) {
  int64_t blocks = (n + 255) / 256;
  if (blocks > 8192) blocks = 8192;
  if (dst_dtype == LTX_BF16)
    convert_kernel<S, bf16><<<static_cast<int>(blocks), 256, 0, s>>>(reinterpret_cast<const S*>(src),
                                                                     reinterpret_cast<bf16*>(dst), n);
  else
    convert_kernel<S, float><<<static_cast<int>(blocks), 256, 0, s>>>(reinterpret_cast<const S*>(src),
                                                                      reinterpret_cast<float*>(dst), n);
  LTX_CUDA(cudaGetLastError());
}

// Scaled-FP8 decode: w[i] = e4m3(codes[i]) * scales[i / K] (K = n for one scale per tensor), stored as bf16
// (__float2bfloat16_rn of the fp32 product: what an fp32 checkpoint of the same values gets) or as the fp32 product; D = void
// only scans.  Every thread reads 16 codes per 16-byte load; the n % 16 tail is read byte by byte.  Each thread that met a NaN
// code (0x7F / 0xFF) adds one to *nan_count.
template <typename D>
__global__ void decode_e4m3_kernel(const uint8_t* __restrict__ codes, const float* __restrict__ scales, int64_t K, int64_t n,
                                   D* __restrict__ out, unsigned int* __restrict__ nan_count) {
  const int64_t chunks = n / 16, stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t tid = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  bool nan = false;
  auto value = [&](uint8_t b, float s) {
    nan |= (b & 0x7F) == 0x7F;
    return __half2float(__half(__nv_cvt_fp8_to_halfraw(b, __NV_E4M3))) * s;
  };
  for (int64_t t = tid; t < chunks; t += stride) {
    const uint4 v = reinterpret_cast<const uint4*>(codes)[t];
    const uint8_t* b = reinterpret_cast<const uint8_t*>(&v);
    const int64_t e0 = t * 16;
    int64_t row = e0 / K, col = e0 - row * K;
    float s = scales[row];
    float f[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      if (col == K) { ++row; col = 0; s = scales[row]; }
      f[j] = value(b[j], s);
      ++col;
    }
    if constexpr (std::is_same<D, bf16>::value) {
      alignas(16) bf16 h[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) h[j] = __float2bfloat16_rn(f[j]);
      uint4* o = reinterpret_cast<uint4*>(out + e0);
      o[0] = reinterpret_cast<const uint4*>(h)[0];
      o[1] = reinterpret_cast<const uint4*>(h)[1];
    } else if constexpr (std::is_same<D, float>::value) {
      float4* o = reinterpret_cast<float4*>(out + e0);
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
    }
  }
  for (int64_t i = chunks * 16 + tid; i < n; i += stride) {
    const float f = value(codes[i], scales[i / K]);
    if constexpr (std::is_same<D, bf16>::value) out[i] = __float2bfloat16_rn(f);
    else if constexpr (std::is_same<D, float>::value) out[i] = f;
  }
  if (nan) atomicAdd(nan_count, 1u);
}

// codes / scales on the device (codes 16-byte aligned); out: bf16, fp32 or nullptr (scan only).  Returns how many threads met a
// NaN code (0: none).
unsigned int decode_e4m3(ltx_ctx* c, const uint8_t* codes, const float* scales, int64_t K, int64_t n, int out_dtype, void* out) {
  unsigned int* nan_count = nullptr;
  LTX_CUDA(cudaMalloc(&nan_count, sizeof(unsigned int)));
  LTX_CUDA(cudaMemsetAsync(nan_count, 0, sizeof(unsigned int), c->stream));
  int64_t blocks = (n / 16 + 255) / 256;
  blocks = blocks < 1 ? 1 : blocks > 8192 ? 8192 : blocks;
  const dim3 grid(static_cast<unsigned>(blocks)), block(256);
  if (!out)
    decode_e4m3_kernel<void><<<grid, block, 0, c->stream>>>(codes, scales, K, n, nullptr, nan_count);
  else if (out_dtype == LTX_BF16)
    decode_e4m3_kernel<bf16><<<grid, block, 0, c->stream>>>(codes, scales, K, n, static_cast<bf16*>(out), nan_count);
  else
    decode_e4m3_kernel<float><<<grid, block, 0, c->stream>>>(codes, scales, K, n, static_cast<float*>(out), nan_count);
  LTX_CUDA(cudaGetLastError());
  unsigned int h = 0;
  LTX_CUDA(cudaMemcpyAsync(&h, nan_count, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
  LTX_CUDA(cudaStreamSynchronize(c->stream));
  LTX_CUDA(cudaFree(nan_count));
  c->launches += 1;
  return h;
}

size_t dtype_size(int dt) { return dt == LTX_F32 ? 4 : 2; }

bool ends_with(const std::string& s, const std::string& suf) {
  return s.size() >= suf.size() && s.compare(s.size() - suf.size(), suf.size(), suf) == 0;
}

int storage_dtype(const ltx_ctx* c, const std::string& key, int ndim) {
  if (!(ends_with(key, ".weight") && ndim >= 2)) return LTX_F32;
  // fp32 mode keeps the DiT matrices in fp32; VAE conv kernels are always bf16
  if (c->precision == 32 && key.compare(0, 4, "vae.") != 0 && key.compare(0, 12, "vae_encoder.") != 0 &&
      key.compare(0, 9, "upscaler.") != 0)
    return LTX_F32;
  return LTX_BF16;
}

void erase_tensor(ltx_ctx* c, const std::string& key) {
  auto it = c->tensors.find(key);
  if (it == c->tensors.end()) return;
  it->second.free_storage();
  c->tensors.erase(it);
}

// dtype -1: the storage dtype of the mode (storage_dtype)
DevTensor& alloc_tensor(ltx_ctx* c, const std::string& key, const std::vector<int64_t>& shape, int dtype = -1) {
  erase_tensor(c, key);
  DevTensor t;
  t.shape = shape;
  t.dtype = dtype >= 0 ? dtype : storage_dtype(c, key, static_cast<int>(shape.size()));
  size_t bytes = static_cast<size_t>(t.numel()) * (t.dtype == DT_E4M3 ? 1 : dtype_size(t.dtype));
  LTX_CUDA(cudaMalloc(&t.ptr, bytes < 16 ? 16 : bytes));
  DevTensor& r = c->tensors[key] = t;
  if (r.dtype == DT_E4M3) LTX_CUDA(cudaMalloc(&r.scales, static_cast<size_t>(shape[0]) * 4));
  return r;
}

// The Linears FP8 mode runs on e4m3 codes (dit_convert_fp8): "transformer_blocks.<i>." + one of kLinears.
bool fp8_block_linear(const std::string& key) {
  static const char* kPrefix = "transformer_blocks.";
  static const char* kLinears[] = {"attn1.to_q.weight", "attn1.to_k.weight", "attn1.to_v.weight", "attn1.to_out.weight",
                                   "attn2.to_q.weight", "attn2.to_k.weight", "attn2.to_v.weight", "attn2.to_out.weight",
                                   "ff.project_in.proj.weight", "ff.project_out.weight"};
  const size_t np = strlen(kPrefix);
  if (key.compare(0, np, kPrefix) != 0) return false;
  size_t i = np;
  while (i < key.size() && key[i] >= '0' && key[i] <= '9') ++i;
  if (i == np || i >= key.size() || key[i] != '.') return false;
  const std::string rest = key.substr(i + 1);
  for (const char* l : kLinears)
    if (rest == l) return true;
  return false;
}

// device allocation freed on every exit path
struct DevScratch {
  void* p = nullptr;
  explicit DevScratch(size_t bytes) { LTX_CUDA(cudaMalloc(&p, bytes)); }
  ~DevScratch() { cudaFree(p); }
};

void fill(ltx_ctx* c, const std::string& key, const std::vector<int64_t>& shape, float stdv, float mean, uint64_t& seed) {
  DevTensor& t = alloc_tensor(c, key, shape);
  seed += 0x632BE59BD9B4E019ull;
  if (t.dtype == LTX_BF16)
    launch_fill_normal_bf16(reinterpret_cast<bf16*>(t.ptr), t.numel(), stdv, mean, seed, c->stream);
  else
    launch_fill_normal_f32(reinterpret_cast<float*>(t.ptr), t.numel(), stdv, mean, seed, c->stream);
}

}  // namespace

const DevTensor& get_tensor(ltx_ctx* c, const std::string& key) {
  auto it = c->tensors.find(key);
  LTX_CHECK(it != c->tensors.end(), LTX_ERR_WEIGHTS, "missing weight tensor '" + key + "'");
  return it->second;
}

void load_tensor_host(ltx_ctx* c, const std::string& key, const void* host, int dtype, const int64_t* shape, int ndim) {
  LTX_CHECK(host != nullptr && ndim >= 0 && ndim <= 8, LTX_ERR_INVALID_ARGUMENT, "load_tensor: bad arguments");
  LTX_CHECK(dtype == LTX_F32 || dtype == LTX_BF16 || dtype == LTX_F16, LTX_ERR_INVALID_ARGUMENT, "load_tensor: bad dtype");
  std::vector<int64_t> shp(shape, shape + ndim);
  DevTensor& t = alloc_tensor(c, key, shp);
  const int64_t n = t.numel();
  if (n == 0) return;
  const size_t src_bytes = static_cast<size_t>(n) * dtype_size(dtype);
  if (dtype == t.dtype) {
    LTX_CUDA(cudaMemcpyAsync(t.ptr, host, src_bytes, cudaMemcpyHostToDevice, c->stream));
    LTX_CUDA(cudaStreamSynchronize(c->stream));
    return;
  }
  void* stage = nullptr;
  LTX_CUDA(cudaMalloc(&stage, src_bytes));
  LTX_CUDA(cudaMemcpyAsync(stage, host, src_bytes, cudaMemcpyHostToDevice, c->stream));
  if (dtype == LTX_F32)
    convert_to<float>(stage, t.ptr, t.dtype, n, c->stream);
  else if (dtype == LTX_BF16)
    convert_to<bf16>(stage, t.ptr, t.dtype, n, c->stream);
  else
    convert_to<__half>(stage, t.ptr, t.dtype, n, c->stream);
  LTX_CUDA(cudaStreamSynchronize(c->stream));
  LTX_CUDA(cudaFree(stage));
}

void load_tensor_e4m3_host(ltx_ctx* c, const std::string& key, const uint8_t* codes, const float* scales, int64_t n_scales,
                           const int64_t* shape, bool keep_codes) {
  const int64_t N = shape[0], K = shape[1], n = N * K;
  unsigned int nan = 0;
  if (keep_codes && c->precision == 8 && fp8_block_linear(key)) {
    // the codes go straight into their final allocation; a per-tensor scale is broadcast to the row scales the GEMM reads
    DevTensor& t = alloc_tensor(c, key, {N, K}, DT_E4M3);
    std::vector<float> rows(static_cast<size_t>(N));
    for (int64_t r = 0; r < N; ++r) rows[r] = scales[n_scales == 1 ? 0 : r];
    LTX_CUDA(cudaMemcpyAsync(t.ptr, codes, static_cast<size_t>(n), cudaMemcpyHostToDevice, c->stream));
    LTX_CUDA(cudaMemcpyAsync(t.scales, rows.data(), static_cast<size_t>(N) * 4, cudaMemcpyHostToDevice, c->stream));
    nan = decode_e4m3(c, t.codes(), t.scales, K, n, 0, nullptr);
  } else {
    DevTensor& t = alloc_tensor(c, key, {N, K});
    const size_t code_bytes = (static_cast<size_t>(n) + 15) / 16 * 16;   // the scales start 16-byte aligned
    DevScratch stage(code_bytes + static_cast<size_t>(n_scales) * 4);
    uint8_t* sc = static_cast<uint8_t*>(stage.p);
    float* ss = reinterpret_cast<float*>(sc + code_bytes);
    LTX_CUDA(cudaMemcpyAsync(sc, codes, static_cast<size_t>(n), cudaMemcpyHostToDevice, c->stream));
    LTX_CUDA(cudaMemcpyAsync(ss, scales, static_cast<size_t>(n_scales) * 4, cudaMemcpyHostToDevice, c->stream));
    nan = decode_e4m3(c, sc, ss, n_scales == 1 ? n : K, n, t.dtype, t.ptr);
  }
  if (nan) {
    erase_tensor(c, key);
    LTX_CHECK(false, LTX_ERR_WEIGHTS, "tensor '" + key + "': NaN e4m3 code (0x7F / 0xFF)");
  }
}

void decode_e4m3_tensor(ltx_ctx* c, DevTensor& t) {
  LTX_CHECK(t.dtype == DT_E4M3 && t.shape.size() == 2, LTX_ERR_WEIGHTS, "decode_e4m3_tensor: not an e4m3 matrix");
  bf16* w = nullptr;
  LTX_CUDA(cudaMalloc(&w, static_cast<size_t>(t.numel()) * 2));
  decode_e4m3(c, t.codes(), t.scales, t.shape[1], t.numel(), LTX_BF16, w);
  t.free_storage();
  t.ptr = w;
  t.dtype = LTX_BF16;
}

namespace {
__global__ void lora_add_kernel(void* w, int w_is_bf16, const float* delta, float scale, int64_t n) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    if (w_is_bf16) {
      bf16* p = reinterpret_cast<bf16*>(w);
      p[i] = __float2bfloat16(__bfloat162float(p[i]) + scale * delta[i]);
    } else {
      float* p = reinterpret_cast<float*>(w);
      p[i] += scale * delta[i];
    }
  }
}
}  // namespace

// LoRA fuse at load time (LoRAAdapter.fuseWeights, LoRA/LoRAAdapter.swift:64-166, standard-Linear path; delta =
// scale * up @ down, LoRA/LoRALoader.swift:162-178): W[out, in] += scale * up[out, r] @ down[r, in], on the raw tensor `key`
// (post-mapping name, LoRAKeyMapper.loraKeyToModelKey :209-243) before ltx_finalize_weights packs / quantises it -- so a
// quantised model is "merge, then quantise", the same result as the reference's dequantise -> merge -> requantise up to one
// rounding.  The product runs on the tensor-core GEMM (bf16 operands, fp32 accumulation), the add in fp32.
namespace {
// fuse_lora's temporaries: the staged factors live in c->tensors under reserved keys, the scratch in plain allocations, and
// the context is switched to bf16 storage while the factors are staged.  All of it is undone on every exit path.
struct LoraScope {
  ltx_ctx* c;
  int saved_precision;
  std::vector<void*> scratch;
  explicit LoraScope(ltx_ctx* ctx) : c(ctx), saved_precision(ctx->precision) {}
  void* alloc(size_t bytes) {
    void* p = nullptr;
    LTX_CUDA(cudaMalloc(&p, bytes));
    scratch.push_back(p);
    return p;
  }
  ~LoraScope() {
    c->precision = saved_precision;
    cudaStreamSynchronize(c->stream);
    for (void* p : scratch) cudaFree(p);
    for (const char* k : {"__lora.down.weight", "__lora.up.weight"}) {
      auto t = c->tensors.find(k);
      if (t == c->tensors.end()) continue;
      if (t->second.ptr) cudaFree(t->second.ptr);
      c->tensors.erase(t);
    }
  }
};
float lora_host_value(const void* p, int dtype, int64_t i) {
  if (dtype == LTX_F32) return static_cast<const float*>(p)[i];
  const uint16_t h = static_cast<const uint16_t*>(p)[i];
  if (dtype == LTX_BF16) {
    const uint32_t u = static_cast<uint32_t>(h) << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
  }
  return __half2float(__ushort_as_half(h));
}
}  // namespace

void fuse_lora(ltx_ctx* c, const std::string& key, const void* down_host, const void* up_host, int dtype, int rank, float scale) {
  auto it = c->tensors.find(key);
  LTX_CHECK(it != c->tensors.end(), LTX_ERR_WEIGHTS,
            "LoRA target '" + key + "' is not loaded (fuse before ltx_finalize_weights, after loading the base weights)");
  DevTensor& w = it->second;
  LTX_CHECK(w.shape.size() == 2 && rank > 0, LTX_ERR_INVALID_ARGUMENT, "LoRA: 2-D target and a positive rank");
  // a weight held as e4m3 codes (FP8 mode, scaled-FP8 checkpoint) is merged in bf16 and converted again at finalize by the
  // per-row rule: "merge, then quantise", as for int8
  LTX_CHECK(down_host && up_host && (dtype == LTX_F32 || dtype == LTX_BF16 || dtype == LTX_F16), LTX_ERR_INVALID_ARGUMENT, "LoRA: bad factors");
  if (w.dtype == DT_E4M3) decode_e4m3_tensor(c, w);
  const int64_t out = w.shape[0], in = w.shape[1];
  // the tensor-core GEMM wants K (= rank) to be a multiple of 8: ranks such as 4 are zero-padded, which adds exact zeros
  const int64_t rpad = (static_cast<int64_t>(rank) + 7) / 8 * 8;
  std::vector<float> down_pad, up_pad;
  if (rpad != rank) {
    down_pad.assign(static_cast<size_t>(rpad) * in, 0.f);
    up_pad.assign(static_cast<size_t>(out) * rpad, 0.f);
    for (int64_t r = 0; r < rank; ++r)
      for (int64_t i = 0; i < in; ++i) down_pad[r * in + i] = lora_host_value(down_host, dtype, r * in + i);
    for (int64_t o = 0; o < out; ++o)
      for (int64_t r = 0; r < rank; ++r) up_pad[o * rpad + r] = lora_host_value(up_host, dtype, o * rank + r);
    down_host = down_pad.data(); up_host = up_pad.data(); dtype = LTX_F32;
  }
  LoraScope scope(c);
  // stage both factors as bf16 device tensors through the regular loader (temporary keys), also in fp32 mode
  const int64_t ds[2] = {rpad, in}, us[2] = {out, rpad};
  c->precision = 16;
  load_tensor_host(c, "__lora.down.weight", down_host, dtype, ds, 2);
  load_tensor_host(c, "__lora.up.weight", up_host, dtype, us, 2);
  c->precision = scope.saved_precision;
  const bf16* down = reinterpret_cast<const bf16*>(c->tensors["__lora.down.weight"].ptr);
  const bf16* up = reinterpret_cast<const bf16*>(c->tensors["__lora.up.weight"].ptr);
  bf16* down_t = static_cast<bf16*>(scope.alloc(static_cast<size_t>(in) * rpad * 2));   // [in, rank]: the GEMM's B operand is K-major
  float* delta = static_cast<float*>(scope.alloc(static_cast<size_t>(out) * in * 4));
  launch_transpose_bf16(down, in, static_cast<int>(rpad), static_cast<int>(in), down_t, rpad, c->stream);
  GemmEpi e;
  e.mode = EPI_F32; e.out = delta; e.ldo = in;
  launch_gemm(up, rpad, down_t, rpad, static_cast<int>(out), static_cast<int>(in), static_cast<int>(rpad), e, c->stream);
  const int64_t n = out * in;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 8192) blocks = 8192;
  lora_add_kernel<<<static_cast<int>(blocks), 256, 0, c->stream>>>(w.ptr, w.dtype == LTX_BF16 ? 1 : 0, delta, scale, n);
  LTX_CUDA(cudaGetLastError());
  LTX_CUDA(cudaStreamSynchronize(c->stream));
  c->launches += 3;
}

// Random-init weights of the named architecture (SURVEY Appendix C shapes).  Scales keep activations O(1):
// Linear N(0, 1/in), biases N(0, 0.02^2), scale-shift tables N(0, 0.1^2), q/k norm weights 1 + N(0, 0.1^2).
void init_random_weights(ltx_ctx* c, int which, uint64_t seed) {
  const ltx_config& g = c->cfg;
  const int64_t D = static_cast<int64_t>(g.num_heads) * g.head_dim;
  uint64_t s = seed * 0x9E3779B97F4A7C15ull + 12345;
  auto lin = [&](const std::string& name, int64_t out_f, int64_t in_f, float wscale = 1.0f) {
    fill(c, name + ".weight", {out_f, in_f}, wscale / sqrtf(static_cast<float>(in_f)), 0.f, s);
    fill(c, name + ".bias", {out_f}, 0.02f, 0.f, s);
  };
  if (which & 1) {
    lin("patchify_proj", D, g.in_channels);
    lin("adaln_single.emb.linear_1", D, 256);
    lin("adaln_single.emb.linear_2", D, D);
    lin("adaln_single.linear", 6 * D, D, 0.5f);
    lin("caption_projection.linear_1", D, g.caption_channels);
    lin("caption_projection.linear_2", D, D);
    for (int i = 0; i < g.num_layers; ++i) {
      const std::string p = "transformer_blocks." + std::to_string(i) + ".";
      fill(c, p + "scale_shift_table", {6, D}, 0.1f, 0.f, s);
      for (const char* a : {"attn1", "attn2"}) {
        for (const char* l : {"to_q", "to_k", "to_v", "to_out"}) lin(p + a + "." + l, D, D);
        fill(c, p + a + ".q_norm.weight", {D}, 0.1f, 1.0f, s);
        fill(c, p + a + ".k_norm.weight", {D}, 0.1f, 1.0f, s);
      }
      lin(p + "ff.project_in.proj", g.ffn_mult * D, D);
      lin(p + "ff.project_out", D, g.ffn_mult * D);
    }
    fill(c, "scale_shift_table", {2, D}, 0.1f, 0.f, s);
    lin("proj_out", g.out_channels, D);
  }
  if (which & 2) {
    auto conv = [&](const std::string& name, int64_t cout, int64_t cin) {
      fill(c, name + ".conv.weight", {cout, cin, 3, 3, 3}, 1.0f / sqrtf(27.0f * cin), 0.f, s);
      fill(c, name + ".conv.bias", {cout}, 0.02f, 0.f, s);
    };
    const int64_t C = g.vae_latent_channels;
    fill(c, "vae.mean_of_means", {C}, 0.1f, 0.f, s);
    fill(c, "vae.std_of_means", {C}, 0.05f, 1.0f, s);
    int64_t ch = g.vae_base_channels;
    conv("vae.conv_in", ch, C);
    for (int st = 0; st < 4; ++st) {
      const std::string blk = "vae.up_blocks_" + std::to_string(2 * st);
      for (int j = 0; j < g.vae_blocks_per_stage; ++j) {
        const std::string rb = blk + ".res_blocks." + std::to_string(j);
        conv(rb + ".conv1", ch, ch);
        conv(rb + ".conv2", ch, ch);
        fill(c, rb + ".scale_shift_table", {4, ch}, 0.1f, 0.f, s);
      }
      lin(blk + ".time_embedder.timestep_embedder.linear_1", 256, 256);
      lin(blk + ".time_embedder.timestep_embedder.linear_2", 4 * ch, 256);
      if (st < 3) {
        conv("vae.up_blocks_" + std::to_string(2 * st + 1) + ".conv", 4 * ch, ch);
        ch /= 2;
      }
    }
    fill(c, "vae.last_scale_shift_table", {2, ch}, 0.1f, 0.f, s);
    lin("vae.last_time_embedder.timestep_embedder.linear_1", 256, 256);
    lin("vae.last_time_embedder.timestep_embedder.linear_2", 2 * ch, 256);
    conv("vae.conv_out", 3 * g.vae_patch_size * g.vae_patch_size, ch);
  }
  if (which & 16) {   // audio / cross-modal tensors of LTX2Transformer (T/LTX2Transformer.swift:20-43, T/LTX2TransformerBlock.swift:44-72)
    const int64_t Ha = g.audio_num_heads > 0 ? g.audio_num_heads : 32, hd = g.audio_head_dim > 0 ? g.audio_head_dim : 64;
    const int64_t Da = Ha * hd, Ca = g.audio_in_channels > 0 ? g.audio_in_channels : 128;
    auto adaln = [&](const std::string& name, int64_t dim, int n) {
      lin(name + ".emb.linear_1", dim, 256);
      lin(name + ".emb.linear_2", dim, dim);
      lin(name + ".linear", n * dim, dim, 0.5f);
    };
    auto attn = [&](const std::string& name, int64_t qdim, int64_t cdim, int64_t inner) {
      lin(name + ".to_q", inner, qdim);
      lin(name + ".to_k", inner, cdim);
      lin(name + ".to_v", inner, cdim);
      lin(name + ".to_out", qdim, inner);
      fill(c, name + ".q_norm.weight", {inner}, 0.1f, 1.0f, s);
      fill(c, name + ".k_norm.weight", {inner}, 0.1f, 1.0f, s);
    };
    lin("audio_patchify_proj", Da, Ca);
    adaln("audio_adaln_single", Da, 6);
    lin("audio_caption_projection.linear_1", Da, g.caption_channels);
    lin("audio_caption_projection.linear_2", Da, Da);
    fill(c, "audio_scale_shift_table", {2, Da}, 0.1f, 0.f, s);
    lin("audio_proj_out", Ca, Da);
    adaln("av_ca_video_scale_shift_adaln_single", D, 4);
    adaln("av_ca_a2v_gate_adaln_single", D, 1);
    adaln("av_ca_audio_scale_shift_adaln_single", Da, 4);
    adaln("av_ca_v2a_gate_adaln_single", Da, 1);
    for (int i = 0; i < g.num_layers; ++i) {
      const std::string p = "transformer_blocks." + std::to_string(i) + ".";
      for (const char* n : {"norm1", "norm2", "norm3", "audio_to_video_norm"}) fill(c, p + n + ".weight", {D}, 0.1f, 1.0f, s);
      for (const char* n : {"audio_norm1", "audio_norm2", "audio_norm3", "video_to_audio_norm"}) fill(c, p + n + ".weight", {Da}, 0.1f, 1.0f, s);
      attn(p + "audio_attn1", Da, Da, Da);
      attn(p + "audio_attn2", Da, Da, Da);
      lin(p + "audio_ff.project_in.proj", g.ffn_mult * Da, Da);
      lin(p + "audio_ff.project_out", Da, g.ffn_mult * Da);
      fill(c, p + "audio_scale_shift_table", {6, Da}, 0.1f, 0.f, s);
      attn(p + "audio_to_video_attn", D, Da, Da);
      attn(p + "video_to_audio_attn", Da, D, Da);
      fill(c, p + "scale_shift_table_a2v_ca_video", {5, D}, 0.1f, 0.f, s);
      fill(c, p + "scale_shift_table_a2v_ca_audio", {5, Da}, 0.1f, 0.f, s);
    }
  }
  if (which & 4) {   // VideoEncoder channel plan (Models/VAE/VideoEncoder.swift:222-268)
    auto conv = [&](const std::string& name, int64_t cout, int64_t cin) {
      fill(c, name + ".conv.weight", {cout, cin, 3, 3, 3}, 1.0f / sqrtf(27.0f * cin), 0.f, s);
      fill(c, name + ".conv.bias", {cout}, 0.02f, 0.f, s);
    };
    static const int kRes[4] = {4, 6, 6, 2}, kProd[4] = {4, 2, 8, 8};
    int64_t ch = g.vae_encoder_base_channels > 0 ? g.vae_encoder_base_channels : 128;
    conv("vae_encoder.conv_in", ch, 48);
    for (int i = 0; i < 4; ++i) {
      const std::string blk = "vae_encoder.down_blocks_" + std::to_string(i);
      for (int j = 0; j < kRes[i]; ++j) {
        conv(blk + ".resnets.resnets." + std::to_string(j) + ".conv1", ch, ch);
        conv(blk + ".resnets.resnets." + std::to_string(j) + ".conv2", ch, ch);
      }
      conv(blk + ".downsamplers.conv", 2 * ch / kProd[i], ch);
      ch *= 2;
    }
    for (int j = 0; j < 2; ++j) {
      conv("vae_encoder.mid_block.resnets." + std::to_string(j) + ".conv1", ch, ch);
      conv("vae_encoder.mid_block.resnets." + std::to_string(j) + ".conv2", ch, ch);
    }
    conv("vae_encoder.conv_out", g.vae_latent_channels + 1, ch);
  }
  if (which & 8) {   // SpatialUpscaler (Models/Upscaler/SpatialUpscaler.swift:181-213), checkpoint layout
    const int64_t mid = g.upscaler_mid_channels > 0 ? g.upscaler_mid_channels : 1024, cin = g.vae_latent_channels;
    const int nb = g.upscaler_blocks > 0 ? g.upscaler_blocks : 4;
    auto conv3 = [&](const std::string& name, int64_t cout, int64_t ci) {
      fill(c, name + ".weight", {cout, ci, 3, 3, 3}, 1.0f / sqrtf(27.0f * ci), 0.f, s);
      fill(c, name + ".bias", {cout}, 0.02f, 0.f, s);
    };
    auto norm = [&](const std::string& name) {
      fill(c, name + ".weight", {mid}, 0.1f, 1.0f, s);
      fill(c, name + ".bias", {mid}, 0.1f, 0.f, s);
    };
    conv3("upscaler.initial_conv", mid, cin);
    norm("upscaler.initial_norm");
    for (const char* grp : {"upscaler.res_blocks.", "upscaler.post_upsample_res_blocks."})
      for (int i = 0; i < nb; ++i) {
        const std::string b = std::string(grp) + std::to_string(i);
        conv3(b + ".conv1", mid, mid);
        norm(b + ".norm1");
        conv3(b + ".conv2", mid, mid);
        norm(b + ".norm2");
      }
    fill(c, "upscaler.upsampler.conv.weight", {4 * mid, mid, 3, 3}, 1.0f / sqrtf(9.0f * mid), 0.f, s);
    fill(c, "upscaler.upsampler.conv.bias", {4 * mid}, 0.02f, 0.f, s);
    conv3("upscaler.final_conv", cin, mid);
  }
  LTX_CUDA(cudaStreamSynchronize(c->stream));
}

}  // namespace ltx
