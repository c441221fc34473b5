// The element-wise second passes of the one-sweep Reinhard forms (ReinhardForm, fused_isp.cuh): each turns the map the
// sweep left in reinhard_scratch into the output (normalise by the frame maximum, gamma, quantise).  Every kernel of this
// file is compiled here only; run_fused (fused_api.cu) launches them through the host functions declared in fused_isp.cuh.
#include "fused_isp.cuh"

namespace isp {

// ---------------------------------------------------------------- Camera16 Reinhard in ONE sweep + a light second pass
// pass A: the max sweep with STORE over all frames (scratch = f16 map); pass B: out = quantise((p / max)^(1/gamma))
// element-wise on the scratch, all frames in one launch (blockIdx.y = frame).
template <typename OutT>
__global__ void __launch_bounds__(256) reinhard_scratch_out_kernel(const FramePtrs scratch /* .out = f16 maps */, const FramePtrs fp,
                                                                   long long n_elems /* per frame, % 8 == 0 */, float gamma, const Workspace* ws) {
  const int frame = gridDim.y - 1 - blockIdx.y;       // last frame first: the sweep wrote it last, part of its map is still in L2
  const __half* src = reinterpret_cast<const __half*>(scratch.out[frame]);
  OutT* dst = reinterpret_cast<OutT*>(fp.out[frame]);
  const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, __ldcg(&ws->frame_max[frame])));
  const float inv_gamma = (float)(1.0 / (double)gamma);
  const bool has_gamma = gamma != 1.0f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_elems / 8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 w = __ldcs(reinterpret_cast<const uint4*>(src) + i);
    const __half* t = reinterpret_cast<const __half*>(&w);
    uint32_t v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float q = __saturatef(__half2float(t[j]) * inv_max);
      if (has_gamma) q = fast_pow(q, inv_gamma);
      v[j] = Quant<OutT>::q(q);
    }
    if constexpr (std::is_same<OutT, uint8_t>::value) {
      uint2 o;
      o.x = __byte_perm(__byte_perm(v[0], v[1], 0x0040), __byte_perm(v[2], v[3], 0x0040), 0x5410);
      o.y = __byte_perm(__byte_perm(v[4], v[5], 0x0040), __byte_perm(v[6], v[7], 0x0040), 0x5410);
      __stcs(reinterpret_cast<uint2*>(dst) + i, o);
    } else if constexpr (std::is_same<OutT, uint16_t>::value) {
      uint4 o = make_uint4(__byte_perm(v[0], v[1], 0x5410), __byte_perm(v[2], v[3], 0x5410), __byte_perm(v[4], v[5], 0x5410),
                           __byte_perm(v[6], v[7], 0x5410));
      __stcs(reinterpret_cast<uint4*>(dst) + i, o);
    } else {
      alignas(16) __half o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = __float2half_rn(__uint_as_float(v[j]));
      __stcs(reinterpret_cast<uint4*>(dst) + i, *reinterpret_cast<const uint4*>(o));
    }
  }
}

int run_scratch_out(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, int out_dtype, float gamma,
                    const Workspace* ws, int max_ctas, cudaStream_t s) {
  const dim3 grid((unsigned)std::min<long long>((n_elems / 8 + 255) / 256, max_ctas), (unsigned)n_frames);
  switch (out_dtype) {
    case B200ISP_U8: reinhard_scratch_out_kernel<uint8_t><<<grid, 256, 0, s>>>(sc, fp, n_elems, gamma, ws); break;
    case B200ISP_U16: reinhard_scratch_out_kernel<uint16_t><<<grid, 256, 0, s>>>(sc, fp, n_elems, gamma, ws); break;
    default: reinhard_scratch_out_kernel<__half><<<grid, 256, 0, s>>>(sc, fp, n_elems, gamma, ws); break;
  }
  return cuda_status(cudaPeekAtLastError(), "reinhard_scratch_out_kernel");
}

// pass B of the one-sweep Camera32 Reinhard -> u8 path: out = trunc(255 * ((v + 0.5) / 65535 / max)^(1/gamma)) for the u16
// map v of EpiReinhardMax2<false, CA0, STORE>; frames the map declined are skipped (the gated sweeps write them).
// u16 -> f32 by dropping the halves into the mantissa of 2^23 (PRMT) and one exact packed subtraction -- no conversion
// instruction, packed arithmetic throughout.  Dense outputs: 16 values per thread and iteration (two 16-byte loads, one
// 16-byte store); PITCHED (the outputs are tiles of a grid image, orow > 3 W): 8 values, row / column from the chunk index.
__device__ __forceinline__ void map16_pair(uint32_t w, f2 a2, f2 h2, f2 ig2, bool gamma, uint32_t& v0, uint32_t& v1) {
  const f2 t = add2(pk(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7610)), __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7632))),
                    bc(-8388608.f));
  f2 q = fma2(t, a2, h2);
  if (gamma) {
    float lo, hi, l0, l1;
    upk(q, lo, hi);
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(lo));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(hi));
    upk(mul2(pk(l0, l1), ig2), lo, hi);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(lo));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(hi));
    q = pk(l0, l1);
  }
  float ql, qh;
  upk(fma2_rz(q, bc(255.f), bc(8388608.f)), ql, qh);
  v0 = __float_as_uint(ql);
  v1 = __float_as_uint(qh);
}
__device__ __forceinline__ uint32_t pack4_u8(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

template <bool GAMMA, bool PITCHED>
__global__ void __launch_bounds__(256) reinhard_map16_out_kernel(const FramePtrs scratch /* .out = u16 maps */, const FramePtrs fp,
                                                                 int H, int W, int orow, float gamma, const Workspace* ws) {
  const int frame = gridDim.y - 1 - blockIdx.y;       // last frame first: the sweep wrote it last, part of its map is still in L2
  const float mx = __ldcg(&ws->frame_max[frame]);
  if (reinhard_map16_declined(mx)) return;
  const uint4* src = reinterpret_cast<const uint4*>(scratch.out[frame]);
  const float a = __fdiv_rn(__fdiv_rn(1.0f, mx), kMap16Scale);
  const f2 a2 = bc(a), h2 = bc(0.5f * a), ig2 = bc((float)(1.0 / (double)gamma));
  const long long stride = (long long)gridDim.x * blockDim.x;
  if constexpr (!PITCHED) {
    // two 16-value chunks per iteration, the four 16-byte loads issued before the first use.  Measured on cfg3 (gamma 0.9):
    // 8 CTAs per SM 131 us, 4: 155 us, 2: slower still -- unlike a plain copy this pass wants every thread slot
    // (profiles/r02_reinhard_map16.txt)
    uint4* dst = reinterpret_cast<uint4*>(fp.out[frame]);
    const long long n16 = (long long)H * W * 3 / 16;                   // H even, W % 8 == 0
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += 2 * stride) {
      const long long i2 = i + stride;
      const bool two = i2 < n16;
      const uint4 w0 = __ldcs(src + 2 * i), w1 = __ldcs(src + 2 * i + 1);
      uint4 w2 = w0, w3 = w1;
      if (two) { w2 = __ldcs(src + 2 * i2); w3 = __ldcs(src + 2 * i2 + 1); }
      {
        const uint32_t w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        uint32_t v[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) map16_pair(w[j], a2, h2, ig2, GAMMA, v[2 * j], v[2 * j + 1]);
        __stcs(dst + i, make_uint4(pack4_u8(v[0], v[1], v[2], v[3]), pack4_u8(v[4], v[5], v[6], v[7]), pack4_u8(v[8], v[9], v[10], v[11]),
                                   pack4_u8(v[12], v[13], v[14], v[15])));
      }
      if (two) {
        const uint32_t w[8] = {w2.x, w2.y, w2.z, w2.w, w3.x, w3.y, w3.z, w3.w};
        uint32_t v[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) map16_pair(w[j], a2, h2, ig2, GAMMA, v[2 * j], v[2 * j + 1]);
        __stcs(dst + i2, make_uint4(pack4_u8(v[0], v[1], v[2], v[3]), pack4_u8(v[4], v[5], v[6], v[7]), pack4_u8(v[8], v[9], v[10], v[11]),
                                    pack4_u8(v[12], v[13], v[14], v[15])));
      }
    }
  } else {
    uint8_t* dst = reinterpret_cast<uint8_t*>(fp.out[frame]);
    const int cpr = W * 3 / 8;                                         // 8-value chunks per row
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)H * cpr; i += stride) {
      const int row = (int)(i / cpr), c = (int)(i - (long long)row * cpr);
      const uint4 w0 = __ldcs(src + i);
      const uint32_t w[4] = {w0.x, w0.y, w0.z, w0.w};
      uint32_t v[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) map16_pair(w[j], a2, h2, ig2, GAMMA, v[2 * j], v[2 * j + 1]);
      __stcs(reinterpret_cast<uint2*>(dst + (size_t)row * orow + 8 * c), make_uint2(pack4_u8(v[0], v[1], v[2], v[3]), pack4_u8(v[4], v[5], v[6], v[7])));
    }
  }
}

int run_map16_out(const FramePtrs& sc, const FramePtrs& fp, int n_frames, const IspConsts& k, cudaStream_t s) {
  const long long n_elems = (long long)k.H * k.W * 3;
  const bool gam = k.gamma != 1.0f, pitched = k.orow != 3 * k.W;
  const dim3 grid((unsigned)std::min<long long>((n_elems / 16 + 255) / 256, (8 * kNumSMs + n_frames - 1) / n_frames), (unsigned)n_frames);
  if (gam && pitched) reinhard_map16_out_kernel<true, true><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
  else if (gam) reinhard_map16_out_kernel<true, false><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
  else if (pitched) reinhard_map16_out_kernel<false, true><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
  else reinhard_map16_out_kernel<false, false><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
  return cuda_status(cudaPeekAtLastError(), "reinhard_map16_out_kernel");
}

// pass B through a table (Camera16, gamma != 1, dense u8 outputs): the f16 map has only 65 536 patterns, and the output is a
// pure function of the pattern and the frame maximum.  reinhard_lut_build_kernel evaluates that function once per pattern and
// frame with exactly the arithmetic of reinhard_scratch_out_kernel (so the result is bit-identical to it); reinhard_lut_out_kernel
// keeps the frame's 64 KB table in shared memory and turns every value into one LDS.U8: no MUFU (the arithmetic pass needs 6 per
// pixel and sits at 74 % of the MUFU pipe), 10 instead of 21 instructions per pixel -- the pass becomes a plain HBM stream.
// Camera32 has no table form: its pass (reinhard_map16_out_kernel) is bound by its 2 : 1 read / write DRAM stream (4.75 TB/s),
// not by the MUFU pipe, and the table form measured 134.9 vs 131.5 us on cfg3.
__global__ void __launch_bounds__(256) reinhard_lut_build_kernel(uint8_t* lut /* n_frames x 65536 */, float gamma, const Workspace* ws) {
  const int frame = blockIdx.y;
  const uint32_t v = blockIdx.x * 256 + threadIdx.x;
  const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, __ldcg(&ws->frame_max[frame])));
  float q = __saturatef(__half2float(__ushort_as_half((unsigned short)v)) * inv_max);
  if (gamma != 1.0f) q = fast_pow(q, (float)(1.0 / (double)gamma));
  lut[(size_t)frame * kLutBytes + v] = (uint8_t)Quant<uint8_t>::q(q);
}

__global__ void __launch_bounds__(512) reinhard_lut_out_kernel(const FramePtrs scratch, const FramePtrs fp, long long n16 /* 16-value chunks per frame */,
                                                               const uint8_t* __restrict__ lut) {
  extern __shared__ __align__(16) uint8_t s_lut[];
  const int frame = gridDim.y - 1 - blockIdx.y;       // last frame first: the sweep wrote it last, part of its map is still in L2
  {
    const uint4* g = reinterpret_cast<const uint4*>(lut + (size_t)frame * kLutBytes);
    uint4* s4 = reinterpret_cast<uint4*>(s_lut);
    for (int i = threadIdx.x; i < kLutBytes / 16; i += blockDim.x) s4[i] = __ldg(g + i);
  }
  __syncthreads();
  const uint4* src = reinterpret_cast<const uint4*>(scratch.out[frame]);
  uint4* dst = reinterpret_cast<uint4*>(fp.out[frame]);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x) {
    const uint4 w0 = __ldcs(src + 2 * i), w1 = __ldcs(src + 2 * i + 1);
    const uint32_t w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t a = s_lut[w[2 * j] & 0xFFFFu], b = s_lut[w[2 * j] >> 16], c = s_lut[w[2 * j + 1] & 0xFFFFu], d = s_lut[w[2 * j + 1] >> 16];
      o[j] = a | (b << 8) | (c << 16) | (d << 24);
    }
    __stcs(dst + i, make_uint4(o[0], o[1], o[2], o[3]));
  }
}

int run_lut_pass(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, uint8_t* lut, float gamma, const Workspace* ws,
                 cudaStream_t s) {
  reinhard_lut_build_kernel<<<dim3(kLutBytes / 256, (unsigned)n_frames), 256, 0, s>>>(lut, gamma, ws);
  int st = cuda_status(cudaPeekAtLastError(), "reinhard_lut_build_kernel");
  if (st) return st;
  static bool attr_set = false;          // per process; the attribute belongs to the function, not to a device context
  if (!attr_set) {
    st = cuda_status(cudaFuncSetAttribute(reinhard_lut_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLutBytes), "lut smem attribute");
    if (st) return st;
    attr_set = true;
  }
  const dim3 grid((unsigned)std::min<long long>((n_elems / 16 + 511) / 512, (3 * kNumSMs + n_frames - 1) / n_frames), (unsigned)n_frames);
  reinhard_lut_out_kernel<<<grid, 512, kLutBytes, s>>>(sc, fp, n_elems / 16, lut);
  return cuda_status(cudaPeekAtLastError(), "reinhard_lut_out_kernel");
}

// pass B with planar YUV 4:2:0 output (SURVEY 8f-2, for video encoders): the u8 RGB of reinhard_scratch_out_kernel
// is formed in registers and converted with the arithmetic of color/yuv_420.py:47-64 (csrc/yuv420.cu: x / 255, the
// BT.601 matrix applied to the BGR-swizzled pixel, chroma = mean of the 2x2 quad, one-sided clamp) -- bit-identical
// to rgb_yuv420_image(process_packed12(...)) without writing or re-reading the RGB image: 1.5 B/px out instead of 3.
// Thread = 8 pixel columns x 2 rows (four quads); out = (3H/2, W) u8: H rows of Y, then chroma plane 0 (third
// matrix row) and plane 1 (second matrix row).
__global__ void __launch_bounds__(128) reinhard_scratch_yuv_kernel(const FramePtrs scratch, const FramePtrs fp, int H, int W, float gamma,
                                                            const Workspace* ws) {
  // x / 255 (correctly rounded, yuv_420.py:50) for the 256 possible inputs: a table instead of three IEEE divisions per pixel
  __shared__ float unit[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) unit[i] = __fdiv_rn((float)i, 255.0f);
  __syncthreads();
  const int gx = blockIdx.x * blockDim.x + threadIdx.x, qy = blockIdx.y, frame = blockIdx.z;
  if (gx >= W / 8) return;
  const __half* src = reinterpret_cast<const __half*>(scratch.out[frame]);
  uint8_t* yuv = reinterpret_cast<uint8_t*>(fp.out[frame]);
  const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, __ldcg(&ws->frame_max[frame])));
  const float inv_gamma = (float)(1.0 / (double)gamma);
  const bool has_gamma = gamma != 1.0f;
  constexpr float M[9] = {0.299f, 0.587f, 0.114f, -0.168736f, -0.331264f, 0.5f, 0.5f, -0.418688f, -0.081312f};   // yuv_420.py:12-16
  float rgb[2][24];
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) {
    alignas(16) __half h[24];
    ld_bytes<48>(src + ((size_t)(2 * qy + dy) * W + 8 * gx) * 3, h);
#pragma unroll
    for (int e = 0; e < 24; ++e) {
      float q = __saturatef(__half2float(h[e]) * inv_max);
      if (has_gamma) q = fast_pow(q, inv_gamma);
      rgb[dy][e] = unit[Quant<uint8_t>::q(q) & 0xFFu];                          // the u8 value the RGB path stores, / in_scale
    }
  }
  alignas(8) uint8_t yrow[2][8];
  alignas(4) uint8_t cu4[4], cv4[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float u = 0.f, v = 0.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const float* p = &rgb[dy][3 * (2 * q + dx)];
        float o[3];
#pragma unroll
        for (int r = 0; r < 3; ++r)      // M @ (B, G, R), products and sums rounded separately, left to right
          o[r] = __fadd_rn(__fadd_rn(__fmul_rn(M[3 * r], p[2]), __fmul_rn(M[3 * r + 1], p[1])), __fmul_rn(M[3 * r + 2], p[0]));
        const float cu = __fadd_rn(o[1], 0.5f), cv = __fadd_rn(o[2], 0.5f);
        yrow[dy][2 * q + dx] = cast_from_f32<uint8_t>(__fmul_rn(fminf(1.0f, o[0]), 255.0f));
        if (dy == 0 && dx == 0) { u = cu; v = cv; } else { u = __fadd_rn(u, cu); v = __fadd_rn(v, cv); }
      }
    // u / 4.0 (yuv_420.py:62-63): a power-of-two divisor, the product with 0.25 is the same correctly rounded value
    cu4[q] = cast_from_f32<uint8_t>(__fmul_rn(fminf(1.0f, __fmul_rn(u, 0.25f)), 255.0f));
    cv4[q] = cast_from_f32<uint8_t>(__fmul_rn(fminf(1.0f, __fmul_rn(v, 0.25f)), 255.0f));
  }
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) st_bytes<8>(yuv + (size_t)(2 * qy + dy) * W + 8 * gx, yrow[dy]);
  uint8_t* planes = yuv + (size_t)H * W;
  const size_t plane = (size_t)(H / 2) * (W / 2), idx = (size_t)qy * (W / 2) + 4 * gx;
  st_bytes<4>(planes + plane + idx, cu4);
  st_bytes<4>(planes + idx, cv4);
}

int run_scratch_yuv(const FramePtrs& sc, const FramePtrs& fp, int n_frames, const IspConsts& k, cudaStream_t s) {
  const dim3 grid((unsigned)((k.W / 8 + 127) / 128), (unsigned)(k.H / 2), (unsigned)n_frames);
  reinhard_scratch_yuv_kernel<<<grid, 128, 0, s>>>(sc, fp, k.H, k.W, k.gamma, k.ws);
  return cuda_status(cudaPeekAtLastError(), "reinhard_scratch_yuv_kernel");
}

// pass B with a TRANSPOSING transform (k.flip bit 2: transpose / rotate_90 / rotate_270 / transverse, interpolate.py:36-56 --
// rotate_90 is the rig script's default, scripts/tonemap_scan.py) for both one-sweep Reinhard -> u8 forms: the element-wise
// pass is the cheap place to turn the image, the sweep keeps its plain row stores and the separate transform kernel
// (3 + 3 B/px) disappears.  Output (i, j) = source (r, c), i = c or W-1-c (bit 0), j = r or H-1-r (bit 1), shape (W, H).
// CTA = a tile of 128 output columns (source rows) x 16 source columns.  Load phase: thread = 8 pixels of one source row
// (3 x 16 bytes of the map; the tile's 96-byte row segments are whole sectors), normalise / gamma / quantise exactly like
// the dense pass, one RGBx word per pixel into shared memory at [column][j + (j >> 3)] (row pitch 144 words).  Store phase:
// thread = 8 consecutive pixels of one OUTPUT row (24 bytes, three 8-byte stores): a half warp writes 384 contiguous
// bytes, and with that layout the 32 lanes of every LDS hit 32 different banks.  Default write policy: the two partial
// sectors at the ends of a 384-byte piece meet their neighbours' (blockIdx.x runs along the output row) in L2.
// Camera32: frames the u16 map declined were written as plain (H, W, 3) u8 into the frame's scratch by the gated write sweep
// BEFORE this pass, which then only turns them.
#ifndef ISP_TURNED_MINBLOCKS
#define ISP_TURNED_MINBLOCKS 6     // measured: 8 CTAs per SM (32 registers, no spills) gain 2 % on eager Camera32 calls but lose 1 % on
                                   // Camera16 and 2 % on the graphed look-ahead step (cfg3_rot90 214 -> 207 Gpixel/s)
#endif
constexpr int kTpRows = 128, kTpCols = 16, kTpPitch = 144;
template <bool CAM16, bool GAMMA>
__global__ void __launch_bounds__(256, ISP_TURNED_MINBLOCKS) reinhard_out_transposed_kernel(const FramePtrs scratch, const FramePtrs fp, int H, int W, int orow, int flip,
                                                                      float gamma, const Workspace* ws) {
  __shared__ uint32_t tile[kTpCols * kTpPitch];
  const int frame = gridDim.z - 1 - blockIdx.z;        // last frame first, like the dense pass
  const int j0 = blockIdx.x * kTpRows, c0 = blockIdx.y * kTpCols;
  const float mx = __ldcg(&ws->frame_max[frame]);
  {
    const int cg = threadIdx.x & 1, lr = threadIdx.x >> 1;
    const int j = j0 + lr, c = c0 + 8 * cg;
    if (j < H && c < W) {
      const int r = (flip & 2) ? H - 1 - j : j;
      const size_t px = (size_t)r * W + c;
      uint32_t v[24];
      if constexpr (CAM16) {
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(scratch.out[frame]) + px * 3);
        const uint4 w3[3] = {__ldcs(src), __ldcs(src + 1), __ldcs(src + 2)};
        const __half* t = reinterpret_cast<const __half*>(w3);
        const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, mx));
        const float inv_gamma = (float)(1.0 / (double)gamma);
#pragma unroll
        for (int e = 0; e < 24; ++e) {
          float q = __saturatef(__half2float(t[e]) * inv_max);
          if (GAMMA) q = fast_pow(q, inv_gamma);
          v[e] = Quant<uint8_t>::q(q);
        }
      } else if (reinhard_map16_declined(mx)) {
        const uint2* src = reinterpret_cast<const uint2*>(reinterpret_cast<const uint8_t*>(scratch.out[frame]) + px * 3);
        const uint2 b3[3] = {__ldcs(src), __ldcs(src + 1), __ldcs(src + 2)};
        const uint8_t* t = reinterpret_cast<const uint8_t*>(b3);
#pragma unroll
        for (int e = 0; e < 24; ++e) v[e] = t[e];
      } else {
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(scratch.out[frame]) + px * 3);
        const uint4 w3[3] = {__ldcs(src), __ldcs(src + 1), __ldcs(src + 2)};
        const uint32_t* w = reinterpret_cast<const uint32_t*>(w3);
        const float a = __fdiv_rn(__fdiv_rn(1.0f, mx), kMap16Scale);
        const f2 a2 = bc(a), h2 = bc(0.5f * a), ig2 = bc((float)(1.0 / (double)gamma));
#pragma unroll
        for (int e = 0; e < 12; ++e) map16_pair(w[e], a2, h2, ig2, GAMMA, v[2 * e], v[2 * e + 1]);
      }
      uint32_t* col = tile + (8 * cg) * kTpPitch + lr + (lr >> 3);
#pragma unroll
      for (int q = 0; q < 8; ++q)      // the values' low bytes -> R | G << 8 | B << 16 (the top byte is never read)
        col[q * kTpPitch] = __byte_perm(__byte_perm(v[3 * q], v[3 * q + 1], 0x0040), v[3 * q + 2], 0x0410);
    }
  }
  __syncthreads();
  {
    const int rg = threadIdx.x & 15, lc = threadIdx.x >> 4;
    const int j = j0 + 8 * rg, c = c0 + lc;
    if (j < H && c < W) {                               // H % 8 == 0: the group is inside the row or entirely outside
      const uint32_t* sp = tile + lc * kTpPitch + 9 * rg;
      uint32_t p[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) p[q] = sp[q];
      const int i = (flip & 1) ? W - 1 - c : c;
      uint2* d = reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(fp.out[frame]) + (size_t)i * orow + 3 * j);
      d[0] = make_uint2(__byte_perm(p[0], p[1], 0x4210), __byte_perm(p[1], p[2], 0x5421));
      d[1] = make_uint2(__byte_perm(p[2], p[3], 0x6542), __byte_perm(p[4], p[5], 0x4210));
      d[2] = make_uint2(__byte_perm(p[5], p[6], 0x5421), __byte_perm(p[6], p[7], 0x6542));
    }
  }
}
int run_out_transposed(bool cam16, const FramePtrs& sc, const FramePtrs& fp, int n_frames, const IspConsts& k, cudaStream_t s) {
  const dim3 grid((unsigned)((k.H + kTpRows - 1) / kTpRows), (unsigned)((k.W + kTpCols - 1) / kTpCols), (unsigned)n_frames);
  const bool gam = k.gamma != 1.0f;
  if (cam16 && gam) reinhard_out_transposed_kernel<true, true><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.flip, k.gamma, k.ws);
  else if (cam16) reinhard_out_transposed_kernel<true, false><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.flip, k.gamma, k.ws);
  else if (gam) reinhard_out_transposed_kernel<false, true><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.flip, k.gamma, k.ws);
  else reinhard_out_transposed_kernel<false, false><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.flip, k.gamma, k.ws);
  return cuda_status(cudaPeekAtLastError(), "reinhard_out_transposed_kernel");
}

// pass B of Reinhard on the output-resolution scratch (ISP dtype): out = quantise((p / max_out)^(1/gamma)), camera_isp.py:217-218
template <typename ScratchT, typename OutT>
__global__ void __launch_bounds__(256) resize_normalise_kernel(const FramePtrs scratch, const FramePtrs outs, long long n_elems,
                                                               float gamma, const Workspace* ws) {
  const int frame = blockIdx.y;
  const ScratchT* src = reinterpret_cast<const ScratchT*>(scratch.out[frame]);
  OutT* dst = reinterpret_cast<OutT*>(outs.out[frame]);
  const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, __ldcg(&ws->frame_max[frame])));
  const float inv_gamma = (float)(1.0 / (double)gamma);
  const bool has_gamma = gamma != 1.0f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_elems; i += (long long)gridDim.x * blockDim.x) {
    float q = __saturatef(to_f32(src[i]) * inv_max);
    if (has_gamma) q = fast_pow(q, inv_gamma);
    if constexpr (DT<OutT>::is_int) dst[i] = (OutT)(Quant<OutT>::q(q) & (uint32_t)DT<OutT>::scale);
    else dst[i] = cast_from_f32<OutT>(q);
  }
}

template <typename ScratchT>
static void launch_resize_normalise(dim3 grid, const FramePtrs& sc, const FramePtrs& fp, long long n_elems, int out_dtype, float gamma,
                                    const Workspace* ws, cudaStream_t s) {
  switch (out_dtype) {
    case B200ISP_U8: resize_normalise_kernel<ScratchT, uint8_t><<<grid, 256, 0, s>>>(sc, fp, n_elems, gamma, ws); break;
    case B200ISP_U16: resize_normalise_kernel<ScratchT, uint16_t><<<grid, 256, 0, s>>>(sc, fp, n_elems, gamma, ws); break;
    default: resize_normalise_kernel<ScratchT, __half><<<grid, 256, 0, s>>>(sc, fp, n_elems, gamma, ws); break;
  }
}

int run_resize_normalise(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, bool cam16, int out_dtype,
                         float gamma, const Workspace* ws, cudaStream_t s) {
  const dim3 grid((unsigned)std::min<long long>((n_elems + 255) / 256, 8 * kNumSMs), (unsigned)n_frames);
  if (cam16) launch_resize_normalise<__half>(grid, sc, fp, n_elems, out_dtype, gamma, ws, s);
  else launch_resize_normalise<float>(grid, sc, fp, n_elems, out_dtype, gamma, ws, s);
  return cuda_status(cudaPeekAtLastError(), "resize_normalise_kernel");
}

}  // namespace isp
