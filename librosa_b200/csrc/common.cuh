// common.cuh — shared declarations for the b2l kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2l {

enum PadMode : int {   // librosa/_typing.py:60-71 (_PadModeSTFT); callables are rejected on the host
  PAD_CONSTANT = 0,
  PAD_EDGE = 1,
  PAD_REFLECT = 2,
  PAD_SYMMETRIC = 3,
  PAD_LINEAR_RAMP = 4,
  PAD_EMPTY = 5,       // values undefined in NumPy; zeros here
};

enum FwdMode : int {
  MODE_STFT = 0,   // complex64 [clip][frame][bin]
  MODE_MEL = 1,    // |X|^power -> band-sparse mel projection -> float32 [clip][mel][frame]
  MODE_SPEC = 2,   // |X|^power -> float32 [clip][frame][bin]
  MODE_STATS = 3,  // per-frame statistics of |X| (centroid, bandwidth, rolloff, flatness, rms) [clip][stat][frame]
};

struct MelBand { int lo, len, off, pad; };   // bins [lo, lo+len), weights at mel_w[off ..] (mel_project kernel)
// Fused-kernel form of one mel row: `quads` groups of 4 consecutive bins starting at bin `lo` (a multiple of
// 4), weights at mel_w[off ..] (zero padded to 4*quads, off % 4 == 0).  Rows are grouped H at a time (a work
// item; H = 32 / frame lanes): the rows of an item share `quads`, and their `lo` follow the bank rule of
// MelLayout.
struct MelRow { unsigned short lo, quads; unsigned int off; };

// Shared-memory layout of the power tile used by the mel phase: frame f keeps its row in the exchange region of
// its own frame group (so no other group has to be waited for before it is written), P[f][k] at word f*RS + k
// with RS = 2 * GS, GS = the group stride in float2 — the exchange buffer (M + M/32 float2) plus a few pad
// entries chosen so that RS is congruent to max(H, 4) modulo 32.
// A lane of the mel loop owns one mel row and a PAIR of frames (f, f + FT/2) — one weight fetch serves both —
// so a warp covers FP = FT/2 frame pairs x H = 32/FP rows (tiles of fewer than 8 frames: one frame per lane,
// H = 32/FT rows).  Weights and power values are both read four bins at a time (16-byte shared loads).  A
// 16-byte load is served a quarter warp at a time: lanes (fp < min(FP, 8), j < 8/FP) — with RS as above and row
// starts lo_j congruent to 4*(j mod G) modulo 4*G, G = max(H, 4)/4 (host: get_row_table), the eight 16-byte
// pieces fall into eight different bank groups.  Rows hold bins 0 .. M plus three zero bins so that 4-bin
// groups may run past the Nyquist bin.
template <int M, int FT>
struct MelLayout {
  static constexpr bool PAIR = (FT % 2) == 0 && FT >= 8;   // few frames per tile: H would exceed 8 rows sharing one trip count
  static constexpr int FP = PAIR ? FT / 2 : FT;     // lanes along the frame axis
  static constexpr int H = 32 / FP;                 // mel rows handled concurrently by one warp
  static constexpr int RSM = H < 4 ? 4 : H;         // residue of the row stride modulo 32
  static constexpr int XB = M + M / 32;             // FftCfg::XBUF_F2
  static constexpr int GS = XB + ((((RSM - 2 * XB) % 32) + 32) % 32) / 2;   // group stride, float2
  static constexpr int RS = 2 * GS;                 // row stride, words
  static_assert(RS >= M + 4 && RS % 32 == RSM % 32 && RS % 4 == 0, "row stride");
};
// host mirrors of MelLayout<M, FT>
__host__ __device__ inline int mel_rows_per_warp(int ft) { return 32 / (((ft % 2) == 0 && ft >= 8) ? ft / 2 : ft); }
__host__ __device__ inline int mel_group_stride(int m, int ft) {
  const int h = mel_rows_per_warp(ft), rsm = h < 4 ? 4 : h, xb = m + m / 32;
  return xb + ((((rsm - 2 * xb) % 32) + 32) % 32) / 2;
}

// Per-frame spectral statistics (stats.cuh): the rows of the [clip][N_STATS][frame] output.
enum StatRow : int { STAT_CENTROID = 0, STAT_BANDWIDTH = 1, STAT_ROLLOFF = 2, STAT_FLATNESS = 3, STAT_RMS = 4, STAT_TOTAL = 5 };
constexpr int N_STATS = 6;
struct StatsParams {
  float roll_percent;            // spectral_rolloff
  float flat_amin, flat_power;   // spectral_flatness: max(amin, S^power)
  float bw_p;                    // spectral_bandwidth: (sum S |f - centroid|^p)^(1/p)
  int bw_norm;                   //   ... with S normalised to unit sum per frame
  int frame_length;              // rms(S=...): DC (and Nyquist when even) count half
  int want;                      // bit r set: row r is needed (the others may hold anything)
};

struct FwdArgs {
  // input
  const float* y;            // [n_clips][clip_stride] (first n samples of each row are valid)
  long long clip_stride;
  int n, n_clips;
  int n_fft, hop, pad, pad_mode, n_frames;
  int tiles_per_clip;
  long long total_tiles;
  int tma_ok;                // host-checked alignment of base pointer / stride / span
  // constants (device)
  const float* window;       // [n_fft] float32, already scaled by 1/2 for the packed real FFT
  const float2* tw;          // inter-pass twiddles, FftCfg::tw_offset layout
  const float2* twn;         // exp(-2*pi*i*k/n_fft), k = 0 .. n_fft/4
  // outputs
  float2* out_c;             // MODE_STFT
  float* out_r;              // MODE_MEL / MODE_SPEC
  // power / mel / dB epilogue
  int power_mode;            // 2: re^2+im^2, 1: sqrt, 0: powf(|X|, power)
  float power;
  int n_mels, mel_w_count;
  const float* mel_w;        // padded weights of the MelRow table built for this tile geometry
  const MelRow* mel_rows;    // n_mel_rows = n_mels rounded up to a multiple of H
  int n_mel_rows;
  const unsigned short* mel_order;   // [mel_list_len][warps per half]: k-th work item of each warp (0xffff: none)
  int mel_list_len;
  int log_mode;              // 1: write 10*log10(max(amin, S)) - db_sub and track the per-clip max
  int out_tiled;             // MODE_MEL: out_r is the mfcc scratch [clip][tile of 64 frames][mel][64] (dct_clamp4_kernel)
  float amin, db_sub;
  unsigned int* clip_max;    // order-preserving uint keys of the per-clip max (log_mode)
  int* status;               // bit 0 is set when a non-finite sample reached a frame (util.valid_audio)
  StatsParams stats;         // MODE_STATS (the frequency table travels in mel_w / mel_w_count)
  // dynamic shared-memory layout (byte offsets)
  int off_win, off_tw, off_in, off_xbuf, off_melw, off_melband, off_melorder, off_bar;
  int in_stride, xbuf_stride; // per-half strides (bytes) of the staging / exchange areas (DUAL)
  int in_floats;             // staged span length (floats)
};

struct InvArgs {
  const float2* D;           // [n_clips][n_frames_total][n_bins]
  long long d_clip_stride;   // in float2 elements
  int n_clips, n_frames;     // frames actually used (<= frames stored)
  int n_fft, hop, start;     // start = n_fft/2 when center else 0
  int out_len;
  long long y_clip_stride;
  float* y;                  // [n_clips][y_clip_stride]
  const float* window;       // [n_fft] float32 scaled by 1/n_fft
  const float* inv_wss;      // [out_len] 1/wss where wss > tiny else 1
  const float2* tw;
  const float2* twn;
  int frames_per_slot;       // consecutive (clip, frame) pairs per half-CTA, a multiple of the round size
  int vec4;                  // gather 4 samples per thread (alignment conditions checked on the host)
  int off_win, off_tw, off_xbuf, off_acc;
  int xbuf_stride, acc_stride;   // per-half strides in bytes (DUAL)
  int acc_floats;
};

// order-preserving float <-> uint mapping for atomicMax on floats
__host__ __device__ inline unsigned int float_to_key(float f) {
#ifdef __CUDA_ARCH__
  unsigned int u = __float_as_uint(f);
#else
  union { float f; unsigned int u; } c; c.f = f; unsigned int u = c.u;
#endif
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float key_to_float(unsigned int k) {
  unsigned int u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  union { float f; unsigned int u; } c; c.u = u; return c.f;
#endif
}

}  // namespace b2l
