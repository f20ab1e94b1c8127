// C ABI of the VQ-VAE decoder kernels (include/d3pm_b200.h, "token -> video, second stage").
#include <type_traits>

#include "d3pm_decoder.cuh"
#include "d3pm_host.h"

namespace {
using d3pm::host::fail;
using d3pm::host::check_launch;
using d3pm::host::DeviceGuard;

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
}  // namespace

extern "C" {

int64_t d3pm_dec_image_floats(int nclass, int N, int Ktot, int n_tile) {
  if (nclass <= 0 || N <= 0 || Ktot <= 0 || Ktot % 32 != 0 || (n_tile != 128 && n_tile != 256)) return 0;
  const int Npad = (N + n_tile - 1) / n_tile * n_tile;
  return static_cast<int64_t>(nclass) * d3pm::dec::image_floats(Npad, Ktot);
}

int d3pm_dec_weight_image(const float* w, int nclass, int N, int Ktot, int n_tile, float* image, d3pm_stream_t stream) {
  if (w == nullptr || image == nullptr) return fail(D3PM_ERR_INVALID, "dec_weight_image: null pointer");
  if (nclass <= 0 || nclass > D3PM_DEC_MAX_CLASSES || N <= 0 || Ktot <= 0 || Ktot % 32 != 0 || (n_tile != 128 && n_tile != 256))
    return fail(D3PM_ERR_INVALID, "dec_weight_image: nclass=%d N=%d Ktot=%d n_tile=%d (Ktot %% 32 == 0, n_tile in {128, 256})", nclass, N, Ktot, n_tile);
  if (!aligned16(w) || !aligned16(image)) return fail(D3PM_ERR_ALIGN, "dec_weight_image: w and image must be 16-byte aligned");
  const DeviceGuard on_device(image);
  const int Npad = (N + n_tile - 1) / n_tile * n_tile;
  const int64_t pieces = static_cast<int64_t>(Npad) * (Ktot / 32) * 8;
  const dim3 grid(static_cast<unsigned>((pieces + 255) / 256), static_cast<unsigned>(nclass));
  d3pm::dec::weight_image_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(w, N, Npad, Ktot, n_tile, image);
  return check_launch("dec_weight_image");
}

int d3pm_dec_conv(const d3pm_dec_conv_desc* d) {
  namespace D = d3pm::dec;
  if (d == nullptr) return fail(D3PM_ERR_INVALID, "dec_conv: null descriptor");
  if (d->x == nullptr || d->w_image == nullptr || d->out == nullptr) return fail(D3PM_ERR_INVALID, "dec_conv: x, w_image and out are required");
  if ((d->in_scale == nullptr) != (d->in_shift == nullptr)) return fail(D3PM_ERR_INVALID, "dec_conv: in_scale and in_shift come together");
  if (d->B <= 0 || d->T <= 0 || d->H <= 0 || d->W <= 0 || d->Cin <= 0 || d->Cin % 32 != 0 || d->Cin > D::kMaxCin)
    return fail(D3PM_ERR_UNSUPPORTED, "dec_conv: B=%d T=%d H=%d W=%d must be positive, Cin=%d a multiple of 32 and <= %d", d->B, d->T, d->H, d->W,
                d->Cin, D::kMaxCin);
  if (d->ntaps <= 0 || d->ntaps > D3PM_DEC_MAX_TAPS || d->nclass <= 0 || d->nclass > D3PM_DEC_MAX_CLASSES)
    return fail(D3PM_ERR_UNSUPPORTED, "dec_conv: ntaps=%d (<= %d), nclass=%d (<= %d)", d->ntaps, D3PM_DEC_MAX_TAPS, d->nclass, D3PM_DEC_MAX_CLASSES);
  const long long rows_out = static_cast<long long>(d->B) * d->T * d->H * d->W * d->stride_t * d->stride_h * d->stride_w;
  if (d->out_transposed) {
    if (d->residual != nullptr || d->ldo <= 0 || rows_out % d->ldo != 0)
      return fail(D3PM_ERR_INVALID, "dec_conv: transposed output takes no residual; ldo (rows per plane) must divide the %lld output rows", rows_out);
  } else if (d->Nout <= 0 || d->Nout % 4 != 0 || d->ldo < d->Nout || d->ldo % 4 != 0) {
    return fail(D3PM_ERR_ALIGN, "dec_conv: Nout=%d and ldo=%lld must be multiples of 4, ldo >= Nout", d->Nout, (long long)d->ldo);
  }
  if (d->n_tile != 128 && d->n_tile != 256) return fail(D3PM_ERR_INVALID, "dec_conv: n_tile=%d must be 128 or 256", d->n_tile);
  if (d->terms != 1 && d->terms != 3) return fail(D3PM_ERR_INVALID, "dec_conv: terms=%d must be 1 (TF32) or 3 (3xTF32)", d->terms);
  if (d->stride_t < 1 || d->stride_h < 1 || d->stride_w < 1) return fail(D3PM_ERR_INVALID, "dec_conv: strides must be >= 1");
  for (int c = 0; c < d->nclass; ++c)
    if (d->cls[c][0] < 0 || d->cls[c][0] >= d->stride_t || d->cls[c][1] < 0 || d->cls[c][1] >= d->stride_h || d->cls[c][2] < 0 ||
        d->cls[c][2] >= d->stride_w)
      return fail(D3PM_ERR_INVALID, "dec_conv: class %d offset outside its stride", c);
  if (!aligned16(d->x) || !aligned16(d->w_image) || !aligned16(d->out) || !aligned16(d->bias) || !aligned16(d->residual) ||
      !aligned16(d->in_scale) || !aligned16(d->in_shift))
    return fail(D3PM_ERR_ALIGN, "dec_conv: every pointer must be 16-byte aligned");
  const DeviceGuard on_device(d->out);
  D::GemmParams p;
  p.x = d->x, p.in_scale = d->in_scale, p.in_shift = d->in_shift, p.w_image = d->w_image, p.bias = d->bias;
  p.residual = d->residual, p.out = d->out;
  p.B = d->B, p.T = d->T, p.H = d->H, p.W = d->W, p.Cin = d->Cin, p.ntaps = d->ntaps, p.nclass = d->nclass;
  p.Nout = d->Nout, p.Npad = (d->Nout + d->n_tile - 1) / d->n_tile * d->n_tile, p.ldo = d->ldo;
  p.st = d->stride_t, p.sh = d->stride_h, p.sw = d->stride_w;
  p.To = d->T * p.st, p.Ho = d->H * p.sh, p.Wo = d->W * p.sw;
  p.relu_out = d->relu_out, p.terms = d->terms, p.out_transposed = d->out_transposed ? 1 : 0;
  for (int c = 0; c < D3PM_DEC_MAX_CLASSES; ++c) {
    for (int t = 0; t < D3PM_DEC_MAX_TAPS; ++t)
      for (int e = 0; e < 4; ++e) p.tap[c][t][e] = d->tap[c][t][e];
    for (int e = 0; e < 4; ++e) p.cls[c][e] = d->cls[c][e];
  }
  const long long M = static_cast<long long>(d->B) * d->T * d->H * d->W;
  if (M * d->Cin >= (1LL << 32)) return fail(D3PM_ERR_UNSUPPORTED, "dec_conv: the input has %lld elements; element offsets are 32-bit", M * d->Cin);
  const int ctas = d->cta_pair ? 2 : 1;
  const long long mtiles = ((M + D::kTileM - 1) / D::kTileM + ctas - 1) / ctas;
  const long long tiles = mtiles * (p.Npad / d->n_tile) * d->nclass;
  const int sms = d3pm::host::sm_count();
  if (sms == 0) return fail(D3PM_ERR_CUDA, "dec_conv: cannot query the device");
  const long long units = tiles < sms / ctas ? tiles : sms / ctas;  // persistent: one CTA (or pair) per SM (TPC) walks the tiles
  const cudaStream_t s = static_cast<cudaStream_t>(d->stream);
  auto launch = [&](auto kern, size_t smem) -> int {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
      return fail(D3PM_ERR_CUDA, "dec_conv: %s", cudaGetErrorString(cudaGetLastError()));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(units * ctas));
    cfg.blockDim = dim3(D::kGemmThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = static_cast<unsigned>(ctas), attr[0].val.clusterDim.y = 1, attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr, cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, kern, p) != cudaSuccess) return fail(D3PM_ERR_CUDA, "dec_conv: launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return check_launch("dec_conv");
  };
  const int sel = (d->n_tile == 256 ? 4 : 0) | (d->terms == 1 ? 2 : 0) | (ctas == 2 ? 1 : 0);
  switch (sel) {
    case 0: return launch(D::conv_gemm_kernel<128, 3, 1>, D::gemm_smem_bytes<128, 3, 1>());
    case 1: return launch(D::conv_gemm_kernel<128, 3, 2>, D::gemm_smem_bytes<128, 3, 2>());
    case 2: return launch(D::conv_gemm_kernel<128, 1, 1>, D::gemm_smem_bytes<128, 1, 1>());
    case 3: return launch(D::conv_gemm_kernel<128, 1, 2>, D::gemm_smem_bytes<128, 1, 2>());
    case 4: return launch(D::conv_gemm_kernel<256, 3, 1>, D::gemm_smem_bytes<256, 3, 1>());
    case 5: return launch(D::conv_gemm_kernel<256, 3, 2>, D::gemm_smem_bytes<256, 3, 2>());
    case 6: return launch(D::conv_gemm_kernel<256, 1, 1>, D::gemm_smem_bytes<256, 1, 1>());
    default: return launch(D::conv_gemm_kernel<256, 1, 2>, D::gemm_smem_bytes<256, 1, 2>());
  }
}

int d3pm_dec_embed_rows(const int64_t* tokens, const float* lut, float* out, int64_t rows, int K, int C, uint32_t* status,
                        d3pm_stream_t stream) {
  if (tokens == nullptr || lut == nullptr || out == nullptr || rows <= 0 || K <= 0 || C <= 0 || C % 4 != 0)
    return fail(D3PM_ERR_INVALID, "dec_embed_rows: bad arguments (rows=%lld K=%d C=%d, C %% 4 == 0)", (long long)rows, K, C);
  if (!aligned16(lut) || !aligned16(out)) return fail(D3PM_ERR_ALIGN, "dec_embed_rows: lut and out must be 16-byte aligned");
  const DeviceGuard on_device(out);
  const long long n = rows * (C / 4);
  if ((n + 255) / 256 > 2147483647LL) return fail(D3PM_ERR_UNSUPPORTED, "dec_embed_rows: too many rows");
  d3pm::dec::embed_rows_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(tokens, lut, out, rows, K,
                                                                                                                     C, status);
  return check_launch("dec_embed_rows");
}

int d3pm_dec_axial_attention(const float* qkv, float* att, int B, int T, int H, int W, int heads, int head_dim, float softmax_scale,
                             d3pm_stream_t stream) {
  namespace D = d3pm::dec;
  if (qkv == nullptr || att == nullptr || B <= 0 || T <= 0 || H <= 0 || W <= 0 || heads <= 0)
    return fail(D3PM_ERR_INVALID, "dec_axial_attention: bad arguments");
  if (T > 32 || H > 32 || W > 32) return fail(D3PM_ERR_UNSUPPORTED, "dec_axial_attention: grid %dx%dx%d, every axis must be <= 32", T, H, W);
  if (head_dim != 32 && head_dim != 64 && head_dim != 128)
    return fail(D3PM_ERR_UNSUPPORTED, "dec_axial_attention: head_dim=%d must be 32, 64 or 128", head_dim);
  const DeviceGuard on_device(att);
  const long long M = static_cast<long long>(B) * T * H * W;
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  for (int axis = 0; axis < 3; ++axis) {
    const int L = axis == 0 ? W : (axis == 1 ? H : T);
    const long long jobs = M / L * heads;
    auto launch = [&](auto vpl, auto lmax) {
      constexpr int V = decltype(vpl)::value, LM = decltype(lmax)::value;
      constexpr D::AttnShape SH = D::attn_shape(LM);
      D::axial_attention_kernel<V, LM><<<static_cast<unsigned>((jobs + SH.jpb - 1) / SH.jpb), 32 * SH.bw, 0, s>>>(qkv, att, B, T, H, W, heads,
                                                                                                                 axis, softmax_scale);
    };
    auto by_len = [&](auto vpl) {
      if (L <= 4) launch(vpl, std::integral_constant<int, 4>{});
      else if (L <= 8) launch(vpl, std::integral_constant<int, 8>{});
      else if (L <= 16) launch(vpl, std::integral_constant<int, 16>{});
      else launch(vpl, std::integral_constant<int, 32>{});
    };
    if (head_dim == 32) by_len(std::integral_constant<int, 1>{});
    else if (head_dim == 64) by_len(std::integral_constant<int, 2>{});
    else by_len(std::integral_constant<int, 4>{});
    const int rc = check_launch("dec_axial_attention");
    if (rc != D3PM_OK) return rc;
  }
  return D3PM_OK;
}

int d3pm_dec_col2im(const float* y_t, const float* bias, float* out, int B, int T, int H, int W, int Cout, int st, int sh, int sw,
                    d3pm_stream_t stream) {
  if (y_t == nullptr || out == nullptr || B <= 0 || T <= 0 || H <= 0 || W <= 0) return fail(D3PM_ERR_INVALID, "dec_col2im: bad arguments");
  if (Cout <= 0 || Cout > 4) return fail(D3PM_ERR_UNSUPPORTED, "dec_col2im: Cout=%d must be <= 4", Cout);
  if ((st != 1 && st != 2) || (sh != 1 && sh != 2) || (sw != 1 && sw != 2)) return fail(D3PM_ERR_UNSUPPORTED, "dec_col2im: strides must be 1 or 2");
  const DeviceGuard on_device(out);
  const long long total = static_cast<long long>(B) * T * st * H * sh * W;
  if ((total + 255) / 256 > 2147483647LL) return fail(D3PM_ERR_UNSUPPORTED, "dec_col2im: output too large");
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (sh == 2 && sw == 2 && Cout <= 3) {  // the shape of the decoder's last layer: straight-line loads
    if (st == 1) d3pm::dec::col2im_s22_kernel<1><<<grid, 256, 0, s>>>(y_t, bias, out, B, T, H, W, Cout);
    else d3pm::dec::col2im_s22_kernel<2><<<grid, 256, 0, s>>>(y_t, bias, out, B, T, H, W, Cout);
  } else {
    d3pm::dec::col2im_kernel<<<grid, 256, 0, s>>>(y_t, bias, out, B, T, H, W, Cout, st, sh, sw);
  }
  return check_launch("dec_col2im");
}

}  // extern "C"
