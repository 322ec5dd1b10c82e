// fwd_kernel.cuh — fused frame + pad + window + real FFT kernel with three epilogues
// (complex STFT / power spectrogram / band-sparse mel projection with optional dB + per-clip max).
//
// Replaces, per frame, the reference's  util.frame -> float64 window product -> scipy.fft.rfft
// (librosa/core/spectrum.py:341-390),  np.abs(.)**power (:3000-3013) and the mel einsum
// (librosa/feature/spectral.py:2160).
//
// Work decomposition: a persistent CTA walks tiles of FT consecutive frames of one clip.  The
// contiguous sample span of a tile, (FT-1)*hop + n_fft floats, is staged once into shared memory
// (frames overlap *inside* shared memory) — by a single 1-D TMA bulk copy (cp.async.bulk + mbarrier)
// for interior tiles, prefetched one tile ahead, or by a cooperative gather with the pad-mode index
// map for tiles that touch the clip edges.  Each group of TPF threads then transforms one frame in
// registers (fft_engine.cuh).
#pragma once
#include "common.cuh"
#include "fft_engine.cuh"
#include "stats.cuh"

namespace b2l {

// ------------------------------------------------------------------ mbarrier / TMA (PTX)
// smem_u32(): fft_engine.cuh
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(phase)
      : "memory");
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ------------------------------------------------------------------ Tensor Memory as a per-thread constant store
// (tcgen05.alloc / st / ld; SASS UTCALLOC, STTM, LDTM).  One warp allocates, the address comes back through
// shared memory; a warp reaches only the 32 lanes of its own quarter (warp index mod 4).
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result) {
  constexpr int cols = NCOLS <= 32 ? 32 : NCOLS <= 64 ? 64 : NCOLS <= 128 ? 128 : NCOLS <= 256 ? 256 : 512;
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_free(uint32_t taddr) {
  constexpr int cols = NCOLS <= 32 ? 32 : NCOLS <= 64 ? 64 : NCOLS <= 128 ? 128 : NCOLS <= 256 ? 256 : 512;
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_store1(uint32_t taddr, float v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(__float_as_uint(v)) : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ------------------------------------------------------------------ padded sample fetch
// Virtual sample j of a clip of n samples under np.pad semantics (librosa/core/spectrum.py:252-328,
// equivalence to np.pad(y, n_fft//2, mode) per SURVEY Appendix A.2).
__device__ __forceinline__ float load_padded(const float* __restrict__ y, int n, long long j, int mode, int pad) {
  if (j >= 0 && j < n) return __ldg(y + j);
  switch (mode) {
    case PAD_EDGE:
      return __ldg(y + (j < 0 ? 0 : n - 1));
    case PAD_REFLECT: {
      if (n == 1) return __ldg(y);
      long long P = 2LL * (n - 1);
      long long m = j % P;
      if (m < 0) m += P;
      if (m >= n) m = P - m;
      return __ldg(y + m);
    }
    case PAD_SYMMETRIC: {
      long long P = 2LL * n;
      long long m = j % P;
      if (m < 0) m += P;
      if (m >= n) m = P - 1 - m;
      return __ldg(y + m);
    }
    case PAD_LINEAR_RAMP: {
      long long d = j < 0 ? -j : j - (n - 1);          // distance from the edge sample, 1..pad
      float edge = __ldg(y + (j < 0 ? 0 : n - 1));
      long long i = pad - d;                           // np.linspace(0, edge, pad, endpoint=False)[i]
      if (i <= 0) return 0.0f;
      return (float)((double)i * ((double)edge / (double)pad));
    }
    default:
      return 0.0f;
  }
}

// |X|^power from |X|^2 for power != 2 (kept out of line: the default power-2 path never executes it)
static __device__ __noinline__ float power_from_sq(float p2, int power_mode, float power) {
  float mag = sqrtf(p2);
  return power_mode == 1 ? mag : powf(mag, power);
}
__device__ __forceinline__ float sqmag(float2 x) { return fmaf(x.x, x.x, x.y * x.y); }
// 10 * log10(x) through the hardware base-2 logarithm (MUFU.LG2: 2 ulp, i.e. below 1e-6 dB anywhere in the float32
// range, sub-normal inputs included): the library log10f is 28 instructions per value, and the dB epilogue runs once
// per mel row and frame — for the short rows of n_fft = 1024 it was a third of the projection phase.
__device__ __forceinline__ float db10(float x) { return 3.0102999566398120f * __log2f(x); }
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Exchange-buffer slot of Z[M - k] for k = t + TPF*c (the partner of bin k in the real-FFT un-mix).
// For warp-multiple groups the padded index is affine in the lane with a compile-time offset.
template <int M, int TPF, int C>
__device__ __forceinline__ int partner_slot(int t) {
  if constexpr (TPF % 32 == 0) {
    constexpr int WPG = TPF / 32;                 // warps per group
    const int tl = t & 31, tw = t >> 5;
    const int row = tw + WPG * C;                 // k = tl + 32*row
    const int rows = M / 32;
    // tl != 0: M-k = 32*(rows-1-row) + (32-tl);  tl == 0: M-k = 32*((rows-row) mod rows)
    const int a = 33 * (rows - 1 - row) + 32 - tl;
    const int b = 33 * ((rows - row) & (rows - 1));
    return tl == 0 ? b : a;
  } else {
    const int k = t + TPF * C;
    return xphys((M - k) & (M - 1));
  }
}

// ------------------------------------------------------------------ the kernel
// NW warps per CTA.  With NSPLIT > 1 the CTA is NSPLIT independent parts of NW/NSPLIT warps ("virtual CTAs",
// called halves below): each has
// its own staging buffer, exchange area, mbarrier, named barrier and tile sequence, and only the constant
// tables are shared.  The halves drift apart, so the shared-memory-bound phases of one (operand fetch,
// exchange, mel gather) overlap the FP32-bound butterflies of the other instead of all warps of the SM
// hitting the same pipe at once.
// TM: the window and the inter-pass twiddles live in Tensor Memory (TmemTab, fft_engine.cuh) instead of shared
// memory — a fifth of the shared-memory wavefronts of a frame move to the tcgen05.ld datapath.
template <int LOG2M, int TPF, int NW, int MODE, int NSPLIT, bool TM>
__global__ void __launch_bounds__(NW * 32, 1) fwd_kernel(const FwdArgs a) {
  using Cfg = FftCfg<LOG2M, TPF>;
  constexpr int M = Cfg::M, N = 2 * M, PPT = Cfg::PPT;
  constexpr int NT = NW * 32;
  constexpr int NH = NSPLIT;                   // independent parts ("halves" when 2)
  constexpr bool DUAL = NSPLIT > 1;
  constexpr int HT = NT / NH;                  // threads per half
  constexpr int HW = NW / NH;                  // warps per half
  constexpr int FT = HT / TPF;                 // frames per tile == frame groups per half
  static_assert(NW % NSPLIT == 0, "the warps are split evenly");
  static_assert(TPF <= 32 || NH + NT / TPF <= 15, "named barriers: 1..NH for the halves, then one per frame group");
  static_assert(FT >= 1 && FT <= 32, "tile must hold 1..32 frames");
  static_assert(!TM || (PPT == 32 && NW >= 4 && (TPF <= 32 || (4 * 32) % TPF == 0)), "TMEM tables: 32 points per thread, all four lane quarters in use");
  using Tab = typename std::conditional<TM, TmemTab<Cfg>, SmemTab<Cfg>>::type;
  using ML = MelLayout<M, FT>;
  constexpr int H = ML::H;                     // mel rows handled concurrently by one warp (common.cuh)
  constexpr int NPAIR = PPT / 2;               // bin pairs (k, M-k) per thread

  extern __shared__ __align__(128) unsigned char smem[];
  const int tid = threadIdx.x;
  const int half = DUAL ? tid / HT : 0;
  const int htid = tid - half * HT;
  float* s_win = reinterpret_cast<float*>(smem + a.off_win);
  float2* s_tw = reinterpret_cast<float2*>(smem + a.off_tw);
  float* s_melw = reinterpret_cast<float*>(smem + a.off_melw);
  MelRow* s_row = reinterpret_cast<MelRow*>(smem + a.off_melband);
  float* s_in = reinterpret_cast<float*>(smem + a.off_in + half * a.in_stride);
  float2* s_xall = reinterpret_cast<float2*>(smem + a.off_xbuf + half * a.xbuf_stride);
  float* s_p = reinterpret_cast<float*>(s_xall);               // P rows alias the exchange regions (MelLayout)
  const unsigned short* s_order = reinterpret_cast<const unsigned short*>(smem + a.off_melorder);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + a.off_bar) + half;
  uint64_t* s_empty = reinterpret_cast<uint64_t*>(smem + a.off_bar + 32) + half;   // initialised, never waited on

  const int grp = htid / TPF;                  // frame group == local frame index
  const int t = htid % TPF;
  const int gbar = 1 + NH + half * FT + grp;   // named barrier of this frame group (used when TPF > 32)
  // stride between the exchange regions of consecutive groups: padded in the modes that park the power row there
  constexpr int GS = (MODE == MODE_MEL || MODE == MODE_STATS) ? ML::GS : Cfg::XBUF_F2;
  float2* xbuf = s_xall + grp * GS;
  float2* xb_t = xbuf + xphys(t);                                   // &xbuf[xphys(t)]: base of the affine accesses
  const float2* xb_neg = xbuf - xphys(t) + ((t & 31) == 0 ? 1 : 0);  // base of the mirror (partner) accesses

  auto half_sync = [&]() {
    if constexpr (DUAL) asm volatile("bar.sync %0, %1;" ::"r"(half + 1), "n"(HT) : "memory");   // ids 1 .. NH
    else __syncthreads();
  };

  // ---- one-time table staging (whole CTA)
  Tab tab;
  if constexpr (TM) {
    // Warps 0..3 each fill the lane quarter they can reach: lane i of quarter q serves thread
    // t = (i + 32 q) mod TPF of a frame group (every warp w of the CTA sits in quarter w mod 4).
    uint32_t* s_taddr = reinterpret_cast<uint32_t*>(smem + a.off_bar + 8 * NH);
    if (tid < 32) tmem_alloc<Tab::NCOLS>(s_taddr);
    tmem_fence_before_sync();
    __syncthreads();
    tmem_fence_after_sync();
    const uint32_t tbase = *s_taddr + ((uint32_t)(((tid >> 5) & 3) * 32) << 16);
    if (tid < 128) {
      const int tt = tid % TPF;
      for (int col = 0; col < 64; ++col)          // window pair of pass-0 slot col/2
        tmem_store1(tbase + col, a.window[2 * (tt + pass0_offset<Cfg>(col >> 1)) + (col & 1)]);
      for (int sp = 1; sp < Cfg::NPASS; ++sp) {
        const int R = Cfg::radix(sp), p = Cfg::sublen(sp);
        for (int f = 0; f < PPT; ++f) {
          const int b = f / R, r = f % R, k = (tt + TPF * b) & (p - 1);
          const float2 w = r == 0 ? make_float2(1.0f, 0.0f) : a.tw[Cfg::tw_offset(sp) + (r - 1) * p + k];
          tmem_store1(tbase + 64 * sp + 2 * f, w.x);
          tmem_store1(tbase + 64 * sp + 2 * f + 1, w.y);
        }
      }
      for (int cp = 0; cp < NPAIR; ++cp) {        // un-mix twiddles W_N^(t + TPF*c)
        const float2 w = a.twn[tt + TPF * cp];
        tmem_store1(tbase + Tab::UNMIX_COL + 2 * cp, w.x);
        tmem_store1(tbase + Tab::UNMIX_COL + 2 * cp + 1, w.y);
      }
      tmem_wait_st();
    }
    tmem_fence_before_sync();
    tab.taddr = tbase;
  } else {
    for (int i = tid; i < N; i += NT) s_win[i] = a.window[i];
    for (int i = tid; i < Cfg::TW_COUNT; i += NT) s_tw[i] = a.tw[i];
    tab.win = s_win;
    tab.tw = s_tw;
  }
  if constexpr (MODE == MODE_MEL) {
    for (int i = tid; i < a.mel_w_count; i += NT) s_melw[i] = a.mel_w[i];
    for (int i = tid; i < a.n_mel_rows; i += NT) s_row[i] = a.mel_rows[i];
    unsigned short* so = reinterpret_cast<unsigned short*>(smem + a.off_melorder);
    for (int i = tid; i < a.mel_list_len * HW; i += NT) so[i] = a.mel_order[i];
  }
  if constexpr (MODE == MODE_STATS) {
    for (int i = tid; i < a.mel_w_count; i += NT) s_melw[i] = a.mel_w[i];   // bin frequencies
  }
  if (htid == 0) {
    mbar_init(s_bar, 1);
    mbar_init(s_empty, HW);   // unused, but dropping it reschedules every instantiation: a change to measure on its own
    fence_mbar_init();
  }
  __syncthreads();
  if constexpr (TM) tmem_fence_after_sync();

  const int span = a.in_floats;
  const bool hop_even = (a.hop & 1) == 0;
  // un-mix twiddle of bin k = t + TPF*c: one register x compile-time constant (SmemTab) or a TMEM column pair
  const float2 wt = __ldg(a.twn + t);
  auto unmix_tw = [&](auto C) -> float2 { return tab.template unmix<decltype(C)::value>(wt); };

  // Tile walk without divisions in the loop: tile = clip * tiles_per_clip + tix, advanced by the constant
  // stride (step_c clips, step_t tiles) of this half.
  // How a tile's span gets into shared memory:
  //   TILE_TMA      entirely inside the clip and 16-byte aligned -> one bulk copy
  //   TILE_TMA_ZERO zero ("constant") padding, aligned: bulk-copy the in-range part, threads zero the rest
  //   TILE_GATHER   anything else (reflect / edge / ... padding, unaligned clips): per-sample gather
  enum { TILE_GATHER = 0, TILE_TMA = 1, TILE_TMA_ZERO = 2 };
  struct TileInfo { int clip, tix, kind, lead, valid; };
  auto describe = [&](int clip, int tix) -> TileInfo {
    TileInfo ti;
    ti.clip = clip;
    ti.tix = tix;
    const long long s0 = (long long)tix * FT * a.hop - a.pad;
    ti.lead = s0 < 0 ? (int)(-s0) : 0;                                      // floats before the clip starts
    const long long end = s0 + span;
    ti.valid = (int)((end > a.n ? (long long)a.n : end) - (s0 + ti.lead));  // in-range floats
    if (!a.tma_ok || ((s0 + ti.lead) & 3) != 0) ti.kind = TILE_GATHER;
    else if (ti.lead == 0 && ti.valid == span) ti.kind = TILE_TMA;
    else if (a.pad_mode == PAD_CONSTANT && ti.valid > 0 && (ti.lead & 3) == 0 && (ti.valid & 3) == 0) ti.kind = TILE_TMA_ZERO;
    else ti.kind = TILE_GATHER;
    return ti;
  };
  // Called by the whole half after the staging buffer has been released (B0): start the copy of the tile.
  auto prefetch_copy = [&](const TileInfo& ti) {          // the bulk copy of the tile's in-range part (one thread)
    if (ti.clip >= a.n_clips || ti.kind == TILE_GATHER) return;
    if (htid == 0) {
      const long long s0 = (long long)ti.tix * FT * a.hop - a.pad;
      fence_proxy_async();
      mbar_expect_tx(s_bar, (uint32_t)ti.valid * 4u);
      tma_load_1d(s_in + ti.lead, a.y + (long long)ti.clip * a.clip_stride + s0 + ti.lead, (uint32_t)ti.valid * 4u, s_bar);
    }
  };
  auto prefetch_zeros = [&](const TileInfo& ti) {         // the zero padding around it (every thread of the half)
    if (ti.clip >= a.n_clips || ti.kind != TILE_TMA_ZERO) return;
    for (int i = htid; i < ti.lead; i += HT) s_in[i] = 0.0f;
    for (int i = ti.lead + ti.valid + htid; i < span; i += HT) s_in[i] = 0.0f;
  };
  auto prefetch = [&](const TileInfo& ti) {
    prefetch_copy(ti);
    prefetch_zeros(ti);
  };

  const int tile_step = (int)gridDim.x * NH;
  const int step_c = tile_step / a.tiles_per_clip, step_t = tile_step - step_c * a.tiles_per_clip;
  TileInfo cur;
  {
    const int first = (int)blockIdx.x * NH + half;
    cur = describe(first / a.tiles_per_clip, first % a.tiles_per_clip);
  }
  uint32_t phase = 0;
  prefetch(cur);

  constexpr bool ROWS = (MODE == MODE_MEL || MODE == MODE_STATS);
  float2 v[PPT];
  TileInfo nxt;
  // ---------------- stage a tile's sample span and turn it into windowed pass-0 operands (first stage fused in)
  auto stage_and_fetch = [&](const TileInfo& ti) {
    if constexpr (TM) tab.begin_window();   // first window chunk travels while the tile lands
    if (ti.kind == TILE_GATHER) {
      const float* yc = a.y + (long long)ti.clip * a.clip_stride;
      const long long s0 = (long long)ti.tix * FT * a.hop - a.pad;
      for (int i = htid; i < span; i += HT) s_in[i] = load_padded(yc, a.n, s0 + i, a.pad_mode, a.pad);
      half_sync();
    } else {
      mbar_wait(s_bar, phase);
      phase ^= 1;
      if (ti.kind == TILE_TMA_ZERO) half_sync();   // zeros written by other threads
    }
    const float* fr = s_in + grp * a.hop;
    auto win = [&](auto S) { return tab.template window<decltype(S)::value>(t); };
    if (hop_even) {
      load_pass0_windowed<Cfg>(v, t, [&](int e) { return *reinterpret_cast<const float2*>(fr + 2 * e); }, win);
    } else {
      load_pass0_windowed<Cfg>(v, t, [&](int e) { return make_float2(fr[2 * e], fr[2 * e + 1]); }, win);
    }
  };
  auto advance = [&](const TileInfo& ti) -> TileInfo {   // next tile of this half
    int nc = ti.clip + step_c, nt = ti.tix + step_t;
    if (nt >= a.tiles_per_clip) { nt -= a.tiles_per_clip; ++nc; }
    return describe(nc, nt);
  };
  auto release_staging = [&]() {   // B0: staging buffer consumed -> prefetch the next tile behind the math
    half_sync();
    prefetch(nxt);
  };

  for (; cur.clip < a.n_clips;) {
    const int clip = cur.clip, t0 = cur.tix * FT;
    stage_and_fetch(cur);
    nxt = advance(cur);
    release_staging();

    // ---------------- M-point complex FFT
    // Row modes: the power rows share the exchange regions, so "every warp is done with the previous tile's rows"
    // waits until the first exchange write — the fetch and pass 0 of fast warps overlap slow warps' mel items.
    fft_forward_tab<Cfg, true>(v, t, gbar, xbuf, tab, [&]() {
      if constexpr (ROWS) half_sync();
    });
    if constexpr (ROWS && Cfg::NPASS == 1) half_sync();
    // Bin pair (k, M-k), k = t + TPF*c < M/2: Z[k] is already in one of this thread's registers; only the
    // upper half of the spectrum (indices >= M/2) has to reach its partner thread, through shared memory.
    // un-mix addresses as one pointer per thread plus constants: measured -1.4 % (mel), -1.9 % (statistics) for
    // one-warp groups in the row modes and -0.5 % for the two-warp groups of n_fft 4096, but +6 % for the plain
    // STFT of n_fft 2048 (register allocation), which therefore keeps the index form
    constexpr bool AFFINE_UNMIX = (TPF % 32 == 0) && (TPF > 32 || MODE == MODE_MEL || MODE == MODE_STATS);
    if constexpr (Cfg::NPASS > 1) group_sync<TPF>(gbar);
    static_for<0, PPT>([&](auto S) {
      constexpr int slot = decltype(S)::value;
      constexpr int D = spectrum_offset<Cfg>(slot);
      if constexpr (D >= M / 2) {
        if constexpr (AFFINE_UNMIX && D % 32 == 0) sts_c64(smem_u32(xb_t) + 8u * (D + D / 32), v[slot]);   // xphys(t + D), D a multiple of 32
        else sts_c64(smem_u32(xbuf) + 8u * xphys(t + D), v[slot]);
      }
    });
    tab.begin_unmix();
    group_sync<TPF>(gbar);
    auto pair_operands = [&](auto C, float2& A, float2& B) {
      constexpr int c = decltype(C)::value;
      constexpr int sa = slot_of_pair<Cfg>(c);
      static_assert(sa >= 0, "pair operand must be register resident");
      A = v[sa];
      if constexpr (AFFINE_UNMIX) {
        // padded slot of Z[M - k], k = t + TPF*c:  K_c - xphys(t) (+ 1 in lane 0 of a warp), K_c a constant —
        // see partner_slot; folded into one pointer per thread
        constexpr int K = 33 * (M / 32 - 1 - (TPF / 32) * c) + 32;
        if constexpr (c == 0) B = t == 0 ? A : xb_neg[K];   // k = 0 pairs with itself (Z[M] == Z[0])
        else B = xb_neg[K];
      } else {
        B = xbuf[partner_slot<M, TPF, c>(t)];
        if constexpr (c == 0) {
          if (t == 0) B = A;   // k = 0 pairs with itself (Z[M] == Z[0])
        }
      }
    };

    const int frame = t0 + grp;
    const bool frame_ok = frame < a.n_frames;
    // util.valid_audio (librosa/util/utils.py:303-306) on the device: one NaN / Inf sample makes every
    // bin of every frame that reads it non-finite, so testing one spectrum value per thread and frame
    // catches it without a separate pass over the input.
    if (frame_ok && !(fabsf(v[0].x) + fabsf(v[0].y) <= 3.0e38f)) *a.status = 1;

    if constexpr (MODE == MODE_STFT) {
      float2* orow = a.out_c + ((long long)clip * a.n_frames + frame) * (M + 1);
      static_for<0, NPAIR>([&](auto C) {
        const int k = t + TPF * decltype(C)::value;
        float2 A, B, xa, xb;
        pair_operands(C, A, B);
        r2c_pair(A, B, unmix_tw(C), xa, xb);
        stg_c64_if(orow + k, xa, frame_ok);
        stg_c64_if(orow + (M - k), xb, frame_ok);
      });
      if (t == 0) {
        float2 xa, xb;
        float2 zc = xbuf[xphys(M / 2)];   // Z[M/2]
        r2c_pair(zc, zc, make_float2(0.0f, -1.0f), xa, xb);   // W_N^(M/2) = -i
        stg_c64_if(orow + M / 2, xa, frame_ok);
      }
      group_sync<TPF>(gbar);   // pair reads done before the next tile's exchange writes
    } else {
      float pw[PPT + 1];
      static_for<0, NPAIR>([&](auto C) {
        constexpr int c = decltype(C)::value;
        float2 A, B, xa, xb;
        pair_operands(C, A, B);
        r2c_pair(A, B, unmix_tw(C), xa, xb);
        pw[2 * c] = sqmag(xa);
        pw[2 * c + 1] = sqmag(xb);
      });
      pw[PPT] = 0.0f;
      if (t == 0) {
        float2 xa, xb;
        float2 zc = xbuf[xphys(M / 2)];   // Z[M/2]
        r2c_pair(zc, zc, make_float2(0.0f, -1.0f), xa, xb);
        pw[PPT] = sqmag(xa);
      }
      if (MODE == MODE_STATS || a.power_mode == 1) {
        // |X| (power = 1; the statistics of MODE_STATS are defined on it): MUFU-based square root, inline.
        // sqrt.approx.f32 is accurate to 2^-23 relative; 33 calls of an out-of-line IEEE square root per
        // thread and frame would cost as much as half the FFT.
        static_for<0, PPT + 1>([&](auto S) { pw[decltype(S)::value] = sqrt_approx(pw[decltype(S)::value]); });
      } else if (a.power_mode != 2) {   // warp-uniform, cold: general exponent through powf
        static_for<0, PPT + 1>([&](auto S) {
          pw[decltype(S)::value] = power_from_sq(pw[decltype(S)::value], a.power_mode, a.power);
        });
      }
      if constexpr (MODE == MODE_SPEC) {
        float* orow = a.out_r + ((long long)clip * a.n_frames + frame) * (M + 1);
        if (frame_ok) {
          static_for<0, NPAIR>([&](auto C) {
            constexpr int c = decltype(C)::value;
            const int k = t + TPF * c;
            orow[k] = pw[2 * c];
            orow[M - k] = pw[2 * c + 1];
          });
          if (t == 0) orow[M / 2] = pw[PPT];
        }
        group_sync<TPF>(gbar);
      } else {
        // ---------------- band-sparse mel projection over the tile
        // The power row of frame f goes to the exchange region of its own group (P[f][k] at word f*RS + k,
        // MelLayout): only the group itself has to be done with its Z before the row is written.  Bins
        // M+1 .. M+3 of every row are kept at zero so that 4-bin groups may run past the Nyquist bin.
        constexpr int RS = ML::RS;
        group_sync<TPF>(gbar);   // every thread of the group has fetched its pair operands
        float* prow = reinterpret_cast<float*>(xbuf);
        static_for<0, NPAIR>([&](auto C) {
          constexpr int c = decltype(C)::value;
          const int k = t + TPF * c;
          prow[k] = pw[2 * c];
          prow[M - k] = pw[2 * c + 1];
        });
        if (t == 0) {
          prow[M / 2] = pw[PPT];
          prow[M + 1] = 0.0f;
          prow[M + 2] = 0.0f;
          prow[M + 3] = 0.0f;
        }
        half_sync();   // B2: the tile's rows are complete
        if constexpr (MODE == MODE_STATS) {
          // one warp per frame of the tile: statistics of the magnitude row (stats.cuh)
          const int hwarp = htid >> 5, lane = htid & 31;
          for (int f = hwarp; f < FT; f += HW) {
            bool negative;
            const float r = frame_stats(s_p + f * RS, s_melw, M + 1, lane, a.stats, &negative);
            if (lane < N_STATS && t0 + f < a.n_frames)
              a.out_r[((long long)clip * N_STATS + lane) * a.n_frames + t0 + f] = r;
          }
        } else {
          // Work item = H adjacent mel rows; lane (fp, j) accumulates row item*H + j for the frame pair
          // (fp, fp + FP) over that row's padded band (host-built MelRow table: the rows of an item share
          // one trip count, start bins follow the bank rule of MelLayout, weights are zero padded and 16-byte
          // aligned).  One 16-byte weight fetch and one 16-byte power fetch per frame feed eight FMAs; no
          // cross-lane reduction.  The items of a tile are dealt to the warps round-robin in row order by the host
          // (a.mel_order): neighbouring rows, whose bands overlap in shared memory, run on warps at the same time.
          constexpr int FP = ML::FP;
          constexpr bool PAIR = ML::PAIR;
          const int hwarp = htid >> 5, lane = htid & 31;
          const int fp = lane & (FP - 1), j = lane / FP;
          const bool ok_a = (t0 + fp) < a.n_frames;
          const bool ok_b = PAIR && (t0 + fp + FP) < a.n_frames;
          float wmax = -INFINITY;
          const float* pbase = s_p + fp * RS;
          // output row stride / base: the public [clip][mel][frame] layout, or the tiled mfcc scratch whose
          // 64-frame tiles are contiguous 32 KB blocks for dct_clamp4_kernel (t0 + fp and t0 + fp + FP share a tile)
          const long long orow = a.out_tiled ? 64 : a.n_frames;
          float* obase = a.out_tiled
                             ? a.out_r + ((long long)clip * ((a.n_frames + 63) >> 6) + (t0 >> 6)) * a.n_mels * 64 + (t0 & 63) + fp
                             : a.out_r + (long long)clip * a.n_mels * a.n_frames + t0 + fp;
          // the item index and its row record are fetched one item ahead: two dependent shared-memory loads that
          // would otherwise sit in front of every (short) row with four warps per scheduler to hide them
          int item_nx = a.mel_list_len > 0 ? s_order[hwarp] : 0xffff;
          MelRow row_nx = s_row[(item_nx == 0xffff ? 0 : item_nx * H) + j];
          for (int li = 0; li < a.mel_list_len; ++li) {
            const int item = item_nx;
            if (item == 0xffff) break;
            const int m = item * H + j;
            const MelRow row = row_nx;
            item_nx = li + 1 < a.mel_list_len ? s_order[(li + 1) * HW + hwarp] : 0xffff;
            row_nx = s_row[(item_nx == 0xffff ? 0 : item_nx * H) + j];
            const float4* wp = reinterpret_cast<const float4*>(s_melw + row.off);
            const float4* pa = reinterpret_cast<const float4*>(pbase + row.lo);
            const float4* wend = wp + row.quads;
            float a0 = 0.0f, a1 = 0.0f, b0 = 0.0f, b1 = 0.0f;
            if constexpr (PAIR) {
              const float4* pb = pa + (FP * RS) / 4;
#pragma unroll 2
              for (; wp != wend; ++wp, ++pa, ++pb) {
                const float4 w = *wp, x = *pa, y = *pb;
                a0 = fmaf(w.x, x.x, a0);
                b0 = fmaf(w.x, y.x, b0);
                a1 = fmaf(w.y, x.y, a1);
                b1 = fmaf(w.y, y.y, b1);
                a0 = fmaf(w.z, x.z, a0);
                b0 = fmaf(w.z, y.z, b0);
                a1 = fmaf(w.w, x.w, a1);
                b1 = fmaf(w.w, y.w, b1);
              }
            } else {
#pragma unroll 2
              for (; wp != wend; ++wp, ++pa) {
                const float4 w = *wp, x = *pa;
                a0 = fmaf(w.x, x.x, a0);
                a1 = fmaf(w.y, x.y, a1);
                a0 = fmaf(w.z, x.z, a0);
                a1 = fmaf(w.w, x.w, a1);
              }
            }
            float va = a0 + a1, vb = b0 + b1;
            if (m < a.n_mels) {
              if (a.log_mode) {
                va = db10(fmaxf(a.amin, va)) - a.db_sub;
                if (ok_a) wmax = fmaxf(wmax, va);
                if constexpr (PAIR) {
                  vb = db10(fmaxf(a.amin, vb)) - a.db_sub;
                  if (ok_b) wmax = fmaxf(wmax, vb);
                }
              }
              float* o = obase + (long long)m * orow;
              if (ok_a) o[0] = va;
              if (ok_b) o[FP] = vb;
            }
          }
          if (a.log_mode) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
            if (lane == 0 && wmax > -INFINITY) atomicMax(a.clip_max + clip, float_to_key(wmax));
          }
        }
        // (the next tile's barrier before its first exchange write orders these P reads)
      }
    }
    cur = nxt;
  }
  if constexpr (TM) {
    tmem_fence_before_sync();
    __syncthreads();
    if (tid < 32) {
      tmem_fence_after_sync();
      tmem_free<Tab::NCOLS>(tab.taddr);   // warp 0 sits in quarter 0: its address is the allocation base
    }
  }
}

}  // namespace b2l
