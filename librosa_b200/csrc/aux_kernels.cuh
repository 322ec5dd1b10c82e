// aux_kernels.cuh — the small kernels around the FFT path: clamp + DCT for mfcc, mel projection and
// power_to_db for S= inputs, and a batched transpose used as a layout adapter.
#pragma once
#include "common.cuh"
#include "fft_engine.cuh"   // packed FP32 helpers (fma2, bc2)

namespace b2l {

// ------------------------------------------------------------------ clamp + DCT (mfcc pass B)
__device__ __forceinline__ void cp_async4(void* dst_smem, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src)
               : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// in  L   [n_clips][n_mels][T]   log-mel (dB), not yet clamped — or, `tiled`, the mfcc scratch of fwd_kernel:
//         [n_clips][ceil(T/64)][n_mels][64], every 64-frame tile one contiguous block (full DRAM bursts
//         instead of 256-byte pieces 4*T bytes apart)
// out C   [n_clips][n_mfcc][T]   C[k][t] = sum_m dct[k][m] * max(L[m][t], clipmax - top_db)
// Reference: np.maximum(log_spec, log_spec.max(...) - top_db) (librosa/core/spectrum.py:1881) followed by
// scipy.fft.dct(S, axis=-2, type, norm)[..., :n_mfcc, :] (* lifter) (librosa/feature/spectral.py:2005-2015);
// the DCT (any type / norm, lifter folded in) arrives transposed and zero padded: dctT[m][8*KG].
//
// Persistent blocks walk (clip, 128-frame tile) pairs; warp w owns coefficients 8*(w % KG) .. +7, DCT rows
// are warp-uniform float4 loads and the top_db clamp is applied as the values are read.  The loop is bound by
// the shared-memory pipe: a warp-uniform 16-byte load of four DCT coefficients costs four wavefronts.  A tile is
// two 64-frame blocks of the tiled scratch, contiguous in memory; lane l owns frames 4l .. 4l+3 — one 16-byte
// load per mel row — and the 32 accumulators of a lane are 16 register pairs fed by packed FMAs (coefficient
// broadcast, frame pair): 12 wavefronts and 16 FFMA2 per mel row and warp, 0.375 wavefronts per FMA.  One tile
// buffer per block; two blocks per SM alternate between streaming and multiplying (cp.async).
// KS = 2: two warp sets split the mel rows of a tile and add their partial sums through the (then idle) tile
// buffer — twice the warps per SM (20 for 40 coefficients, five per scheduler) for one more barrier per tile.
constexpr int DCT4_TILE = 128;
template <int KS>
__global__ void __launch_bounds__(KS == 2 ? 640 : 512) dct_clamp4_kernel(const float* __restrict__ L, const float* __restrict__ dctT,
                                  const unsigned int* __restrict__ clip_max, float top_db, int n_mels, int n_mfcc,
                                  int T, int tiles_per_clip, long long total_tiles, int tiled, float* __restrict__ C) {
  extern __shared__ __align__(16) float s_dyn[];
  const int KG = (blockDim.x >> 5) / KS, KP = 8 * KG;
  float* s_dct = s_dyn;                       // [n_mels][KP]
  float* s_tile = s_dyn + n_mels * KP;        // [2][n_mels][64]
  const int blk_words = n_mels * 64;
  const int tid = threadIdx.x, lane = tid & 31, warp = (tid >> 5) % KG, kset = (tid >> 5) / KG;
  const int m_split = KS == 1 ? n_mels : (n_mels + 1) >> 1;
  const int m_lo = kset == 0 ? 0 : m_split, m_hi = kset == 0 ? m_split : n_mels;
  for (int i = tid; i < n_mels * KP; i += blockDim.x) s_dct[i] = dctT[i];
  const bool vec_ok = (T % 4 == 0) && ((reinterpret_cast<uintptr_t>(L) & 15) == 0);
  const bool vec_out = (T % 4 == 0) && ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
  const int blocks64 = (T + 63) >> 6;
  const float* xlane = s_tile + (lane >> 4) * blk_words + (lane & 15) * 4;

  for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    const int clip = (int)(tile / tiles_per_clip);
    const int t0 = (int)(tile % tiles_per_clip) * DCT4_TILE;
    if (tiled) {
      const int b0 = t0 >> 6;
      const int words = (blocks64 - b0 >= 2 ? 2 : 1) * blk_words;   // the clip's last tile may hold one block only
      const float* Lt = L + ((long long)clip * blocks64 + b0) * blk_words;
      for (int i = tid; i < words / 4; i += blockDim.x) cp_async16(s_tile + 4 * i, Lt + 4 * i);
    } else {
      const float* Lc = L + (long long)clip * n_mels * T + t0;
      if (vec_ok && t0 + DCT4_TILE <= T) {
        for (int i = tid; i < 2 * blk_words / 4; i += blockDim.x) {
          const int sb = i / (blk_words / 4), r = i % (blk_words / 4), m = r >> 4, q = r & 15;
          cp_async16(s_tile + 4 * i, Lc + (long long)m * T + sb * 64 + 4 * q);
        }
      } else {
        for (int i = tid; i < 2 * blk_words; i += blockDim.x) {
          const int sb = i / blk_words, r = i % blk_words, m = r >> 6, x = r & 63;
          if (t0 + sb * 64 + x < T) cp_async4(s_tile + i, Lc + (long long)m * T + sb * 64 + x);
          else s_tile[i] = 0.0f;
        }
      }
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    float floor_v = -INFINITY;
    if (clip_max != nullptr && top_db >= 0.0f) floor_v = key_to_float(clip_max[clip]) - top_db;
    float2 acc[8][2];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = make_float2(0.0f, 0.0f);
#pragma unroll 4
    for (int m = m_lo; m < m_hi; ++m) {
      const float4 d0 = *reinterpret_cast<const float4*>(s_dct + m * KP + 8 * warp);
      const float4 d1 = *reinterpret_cast<const float4*>(s_dct + m * KP + 8 * warp + 4);
      const float dv[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
      float4 x = *reinterpret_cast<const float4*>(xlane + m * 64);
      const float2 xa = make_float2(fmaxf(x.x, floor_v), fmaxf(x.y, floor_v));
      const float2 xb = make_float2(fmaxf(x.z, floor_v), fmaxf(x.w, floor_v));
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[j][0] = fma2(bc2(dv[j]), xa, acc[j][0]);
        acc[j][1] = fma2(bc2(dv[j]), xb, acc[j][1]);
      }
    }
    if constexpr (KS == 2) {
      // partial sums of the second warp set travel through the tile buffer: word (4j + i) * KG*32 + warp*32 + lane
      __syncthreads();   // every warp is done with the tile
      float* s_red = s_tile + warp * 32 + lane;
      const int rs = KG * 32;
      if (kset == 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          s_red[(4 * j + 0) * rs] = acc[j][0].x;
          s_red[(4 * j + 1) * rs] = acc[j][0].y;
          s_red[(4 * j + 2) * rs] = acc[j][1].x;
          s_red[(4 * j + 3) * rs] = acc[j][1].y;
        }
      }
      __syncthreads();
      if (kset == 0) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[j][0].x += s_red[(4 * j + 0) * rs];
          acc[j][0].y += s_red[(4 * j + 1) * rs];
          acc[j][1].x += s_red[(4 * j + 2) * rs];
          acc[j][1].y += s_red[(4 * j + 3) * rs];
        }
      }
    }
    const int t = t0 + 4 * lane;
    float* Cc = C + (long long)clip * n_mfcc * T + t;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = 8 * warp + j;
      if (k < n_mfcc && kset == 0) {
        float* o = Cc + (long long)k * T;
        if (vec_out && t + 3 < T) {
          *reinterpret_cast<float4*>(o) = make_float4(acc[j][0].x, acc[j][0].y, acc[j][1].x, acc[j][1].y);
        } else {
          if (t < T) o[0] = acc[j][0].x;
          if (t + 1 < T) o[1] = acc[j][0].y;
          if (t + 2 < T) o[2] = acc[j][1].x;
          if (t + 3 < T) o[3] = acc[j][1].y;
        }
      }
    }
    __syncthreads();   // tile consumed before the next one streams in
  }
}

// Same product without a shared-memory tile, for inputs whose row count does not fit (mfcc(S=...) on a full
// 1025-bin dB spectrogram, as the reference's multichannel tests do): one thread per frame, eight coefficients
// at a time, the input column re-read from L1 / L2 for every group of eight.
__global__ void dct_generic_kernel(const float* __restrict__ L, const float* __restrict__ dctT,
                                   const unsigned int* __restrict__ clip_max, float top_db, int n_mels, int n_mfcc,
                                   int KP, int T, float* __restrict__ C) {
  const int clip = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= T) return;
  const float* Lc = L + (long long)clip * n_mels * T + t;
  float* Cc = C + (long long)clip * n_mfcc * T + t;
  float floor_v = -INFINITY;
  if (clip_max != nullptr && top_db >= 0.0f) floor_v = key_to_float(clip_max[clip]) - top_db;
  for (int k0 = 0; k0 < n_mfcc; k0 += 8) {
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.0f;
    for (int m = 0; m < n_mels; ++m) {
      const float x = fmaxf(Lc[(long long)m * T], floor_v);
      const float4 d0 = __ldg(reinterpret_cast<const float4*>(dctT + (long long)m * KP + k0));
      const float4 d1 = __ldg(reinterpret_cast<const float4*>(dctT + (long long)m * KP + k0 + 4));
      acc[0] = fmaf(d0.x, x, acc[0]); acc[1] = fmaf(d0.y, x, acc[1]); acc[2] = fmaf(d0.z, x, acc[2]); acc[3] = fmaf(d0.w, x, acc[3]);
      acc[4] = fmaf(d1.x, x, acc[4]); acc[5] = fmaf(d1.y, x, acc[5]); acc[6] = fmaf(d1.z, x, acc[6]); acc[7] = fmaf(d1.w, x, acc[7]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (k0 + j < n_mfcc) Cc[(long long)(k0 + j) * T] = acc[j];
  }
}

// ------------------------------------------------------------------ mel projection of a given spectrogram
// S [n_clips][T][F] (bins contiguous) -> mel [n_clips][n_mels][T]; band-sparse rows as in the fused kernel.
// One warp per (clip, frame-tile of 32); lanes own frames, band weights are warp-uniform.
__global__ void mel_project_kernel(const float* __restrict__ S, const float* __restrict__ mel_w,
                                   const MelBand* __restrict__ band, int n_mels, int F, int T,
                                   int tiles_per_clip, float* __restrict__ out) {
  extern __shared__ __align__(16) float s_tile[];   // [F][33]
  const int clip = blockIdx.x / tiles_per_clip;
  const int t0 = (blockIdx.x % tiles_per_clip) * 32;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, NWp = blockDim.x >> 5;
  const float* Sc = S + ((long long)clip * T + t0) * F;
  for (int f = warp; f < 32; f += NWp) {
    const bool ok = t0 + f < T;
    for (int k = lane; k < F; k += 32) s_tile[k * 33 + f] = ok ? Sc[(long long)f * F + k] : 0.0f;
  }
  __syncthreads();
  for (int m = warp; m < n_mels; m += NWp) {
    const MelBand b = band[m];
    float acc = 0.0f;
    for (int kx = 0; kx < b.len; ++kx) acc = fmaf(__ldg(mel_w + b.off + kx), s_tile[(b.lo + kx) * 33 + lane], acc);
    if (t0 + lane < T) out[((long long)clip * n_mels + m) * T + t0 + lane] = acc;
  }
}


// ------------------------------------------------------------------ projection onto a FEW dense rows (chroma)
// filters.chroma gives 12 rows that are dense over all 1 + n_fft/2 bins (librosa/feature/spectral.py:1283-1285,
// einsum "cf,...ft->...ct"): mel_project_kernel's one-warp-per-row walk is a 1025-long dependent FMA chain on 12 of
// a CTA's warps.  Here a persistent CTA keeps the transposed weights wT[bin][16] (rows zero padded to 16) in shared
// memory next to a [F][33] tile of 32 frames; warp w takes the bins w, w + NW, ...: one tile read and three / four
// broadcast 16-byte weight reads feed 12 / 16 FMAs into lane-private accumulators (lane = frame); the NW partial
// sums meet in shared memory and are written along the frame axis.  S [n_clips][T][F] -> out [n_clips][rows][T].
template <int ROWS4>   // rows / 4 rounded up: 1 .. 4
__global__ void __launch_bounds__(256, 1) dense_project_kernel(const float* __restrict__ S, const float* __restrict__ wT,
                                                               int rows, int F, int T, int tiles_per_clip,
                                                               long long total_tiles, float* __restrict__ out) {
  extern __shared__ __align__(16) float s_dense[];
  constexpr int NW = 8;
  float* s_tile = s_dense;                                 // [F][33]
  float4* s_w = reinterpret_cast<float4*>(s_dense + (((size_t)F * 33 + 3) & ~(size_t)3));   // [F][4] float4
  float* s_part = reinterpret_cast<float*>(s_w + (size_t)F * 4);                             // [NW][16][32]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < F * 4; i += 256) s_w[i] = reinterpret_cast<const float4*>(wT)[i];
  for (long long tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
    const int clip = (int)(tile / tiles_per_clip);
    const int t0 = (int)(tile - (long long)clip * tiles_per_clip) * 32;
    const float* Sc = S + ((long long)clip * T + t0) * F;
    __syncthreads();                                       // previous tile consumed (and the weights staged)
    for (int f = warp; f < 32; f += NW) {
      const bool ok = t0 + f < T;
      for (int k = lane; k < F; k += 32) s_tile[k * 33 + f] = ok ? __ldg(Sc + (long long)f * F + k) : 0.0f;
    }
    __syncthreads();
    float acc[4 * ROWS4];
#pragma unroll
    for (int r = 0; r < 4 * ROWS4; ++r) acc[r] = 0.0f;
    for (int k = warp; k < F; k += NW) {
      const float x = s_tile[k * 33 + lane];
#pragma unroll
      for (int q = 0; q < ROWS4; ++q) {
        const float4 w = s_w[k * 4 + q];
        acc[4 * q + 0] = fmaf(w.x, x, acc[4 * q + 0]);
        acc[4 * q + 1] = fmaf(w.y, x, acc[4 * q + 1]);
        acc[4 * q + 2] = fmaf(w.z, x, acc[4 * q + 2]);
        acc[4 * q + 3] = fmaf(w.w, x, acc[4 * q + 3]);
      }
    }
#pragma unroll
    for (int r = 0; r < 4 * ROWS4; ++r) s_part[(warp * 16 + r) * 32 + lane] = acc[r];
    __syncthreads();
    for (int o = tid; o < rows * 32; o += 256) {
      const int r = o >> 5, f = o & 31;
      float v = 0.0f;
#pragma unroll
      for (int w = 0; w < NW; ++w) v += s_part[(w * 16 + r) * 32 + f];
      if (t0 + f < T) out[((long long)clip * rows + r) * T + t0 + f] = v;
    }
  }
}

// ------------------------------------------------------------------ polyphase resampling
// librosa.resample(res_type="polyphase") = scipy.signal.resample_poly(y, up, down) (librosa/core/audio.py:1129-1145):
// upfirdn(h, x, up, down) cropped to [n_pre_remove, n_pre_remove + n_out) with the zero-padded low-pass h the host
// designs exactly as SciPy does (firwin(2 * 10 * max(up, down) + 1, 1 / max(up, down), window=("kaiser", 5.0)) * up,
// float32 for float32 data).  Output sample j is
//     y[j] = sum_m x[m] * h[(n_pre_remove + j) * down - m * up],
// accumulated over increasing m like SciPy's upfirdn loop; one thread per output sample (about 20 * max(1, down / up)
// taps each).  Samples j >= n_keep of a row are the zeros of util.fix_length; out_scale carries 1 / sqrt(ratio).
__global__ void resample_poly_kernel(const float* __restrict__ x, long long x_stride, int n_in, const float* __restrict__ h,
                                     int n_h, int up, int down, long long n_pre_remove, int n_keep, int n_total,
                                     long long n_clips, float out_scale, float* __restrict__ out) {
  const long long total = n_clips * n_total;
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (long long)gridDim.x * blockDim.x) {
    const long long clip = o / n_total;
    const int j = (int)(o - clip * n_total);
    float acc = 0.0f;
    if (j < n_keep) {
      const long long t = (n_pre_remove + j) * (long long)down;          // position in the up-sampled stream
      long long m_hi = t / up;
      if (m_hi > n_in - 1) m_hi = n_in - 1;
      long long m_lo = t - (n_h - 1);                                    // smallest m with t - m * up <= n_h - 1
      m_lo = m_lo <= 0 ? 0 : (m_lo + up - 1) / up;
      const float* xc = x + clip * x_stride;
      long long k = t - m_lo * up;
      for (long long m = m_lo; m <= m_hi; ++m, k -= up) acc = fmaf(__ldg(h + k), __ldg(xc + m), acc);
      acc *= out_scale;
    }
    out[o] = acc;
  }
}

// ------------------------------------------------------------------ power_to_db
__global__ void db_kernel(const float* __restrict__ in, long long per_clip, float amin, float db_sub,
                          unsigned int* __restrict__ clip_max, float* __restrict__ out) {
  const int clip = blockIdx.y;
  const float* ic = in + (long long)clip * per_clip;
  float* oc = out + (long long)clip * per_clip;
  float mx = -INFINITY;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_clip;
       i += (long long)gridDim.x * blockDim.x) {
    float v = 10.0f * log10f(fmaxf(amin, ic[i])) - db_sub;
    oc[i] = v;
    mx = fmaxf(mx, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0 && mx > -INFINITY) atomicMax(clip_max + clip, float_to_key(mx));
}

__global__ void db_clamp_kernel(float* __restrict__ x, long long per_clip, const unsigned int* __restrict__ clip_max,
                                float top_db) {
  const int clip = blockIdx.y;
  float* xc = x + (long long)clip * per_clip;
  const float floor_v = key_to_float(clip_max[clip]) - top_db;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_clip;
       i += (long long)gridDim.x * blockDim.x)
    xc[i] = fmaxf(xc[i], floor_v);
}

// ------------------------------------------------------------------ finite scan of samples no frame reads
// y [n_clips][stride]; checks samples [begin, n) of every clip (the uncovered tail when the last frame
// ends before the clip does, or the whole clip when hop > n_fft leaves gaps).
// grid.x = blocks per clip (bx), grid.y strides the clips: any number of clips, like the kernels it accompanies.
__global__ void finite_scan_kernel(const float* __restrict__ y, long long stride, int n, int begin, long long n_clips,
                                   int* status) {
  bool bad = false;
  for (long long clip = blockIdx.y; clip < n_clips; clip += gridDim.y) {
    const float* yc = y + clip * stride;
    for (long long i = begin + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
      bad |= !(fabsf(yc[i]) <= 3.0e38f);
  }
  if (bad) *status = 1;
}

// ------------------------------------------------------------------ Griffin-Lim phase update
// angles <- rebuilt - scale * tprev ;  angles <- angles / (|angles| + eps) * S      (elementwise)
// librosa/core/spectrum.py:2898-2903 (scale = momentum / (1 + momentum), eps = tiny(complex64)).
__global__ void gl_update_kernel(const float2* __restrict__ rebuilt, const float2* __restrict__ tprev,
                                 const float* __restrict__ S, float scale, float eps, float2* __restrict__ out,
                                 long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float2 a = rebuilt[i];
    if (tprev != nullptr) {
      const float2 p = tprev[i];
      a.x = fmaf(-scale, p.x, a.x);
      a.y = fmaf(-scale, p.y, a.y);
    }
    const float mag = hypotf(a.x, a.y) + eps;
    const float s = S[i];
    out[i] = make_float2(a.x / mag * s, a.y / mag * s);
  }
}

// ------------------------------------------------------------------ overlap-add of chirp-z inverse frames
// Gather-form overlap-add of scratch frames [clip][n_frames][L] into y [clip][out_len], frames added in
// increasing index (the reference's order), then the WOLA normalisation.
__global__ void ola_kernel(const float* __restrict__ ytmp, int n_frames, int L, int hop, int start, int out_len,
                           long long y_stride, const float* __restrict__ inv_wss, float* __restrict__ y) {
  const int clip = blockIdx.y;
  const float* yt = ytmp + (long long)clip * n_frames * L;
  float* yc = y + (long long)clip * y_stride;
  for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < out_len;
       o += (long long)gridDim.x * blockDim.x) {
    const long long u = o + start;
    long long t_hi = u / hop;
    if (t_hi > n_frames - 1) t_hi = n_frames - 1;
    long long t_lo = u - L + 1;
    t_lo = t_lo <= 0 ? 0 : (t_lo + hop - 1) / hop;
    float val = 0.0f;
    for (long long tt = t_lo; tt <= t_hi; ++tt) val += yt[tt * L + (u - tt * hop)];
    yc[o] = val * __ldg(inv_wss + o);
  }
}

// ------------------------------------------------------------------ batched transpose
template <typename T>
__global__ void transpose_kernel(const T* __restrict__ in, int rows, int cols, T* __restrict__ out) {
  __shared__ T tile[32][33];
  const long long base = (long long)blockIdx.z * rows * cols;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int r = r0 + j, c = c0 + threadIdx.x;
    if (r < rows && c < cols) tile[j][threadIdx.x] = in[base + (long long)r * cols + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    int c = c0 + j, r = r0 + threadIdx.x;
    if (r < rows && c < cols) out[base + (long long)c * rows + r] = tile[threadIdx.x][j];
  }
}

}  // namespace b2l
