// emulate.cu -- runs the fused kernels' device code on the CPU, thread by thread and phase by phase
// (the code in tilefft.cuh / twopass_kernels.cuh is __host__ __device__), and checks the result
// against a double-precision FFT.  There is no GPU in the build container, so this is how index maps,
// twiddle tables and shared-memory layouts are verified before a kernel ever runs on the B200.
// It also reports shared-memory bank conflicts of the exchange (64-bit/128-bit access model).
// Build: nvcc -std=c++17 -O1 --expt-relaxed-constexpr -I fourier_b200/csrc tools/emulate.cu \
//             fourier_b200/csrc/plan.cu ... (host only, never run on the device)
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "cta_kernels.cuh"
#include "dist_kernels.cuh"
#include "fused_kernels.cuh"
#include "onchip_kernels.cuh"
#include "outer_kernels.cuh"
#include "twopass_kernels.cuh"

#ifndef FB_PAD16
#define FB_PAD16 8
#endif
#ifndef FB_PADX
#define FB_PADX 8
#endif
using namespace fb200;
using namespace fb200::twopass;

template <typename T> static void fill(std::vector<cpx<T>>& x, unsigned seed) {
  unsigned long long s = seed * 2654435761ull + 12345;
  for (auto& v : x) {
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    v.x = (T)((double)(s >> 11) / 9007199254740992.0 * 2 - 1);
    s = s * 6364136223846793005ull + 1442695040888963407ull;
    v.y = (T)((double)(s >> 11) / 9007199254740992.0 * 2 - 1);
  }
}

// worst-case bank conflict degree of one warp-wide shared access, element size B bytes:
// lanes are served in groups of 128 bytes worth of lanes (half-warp for 8 B, quarter-warp for 16 B)
template <int B> static int conflict_degree(const std::vector<long>& elem_index) {
  const int group = 128 / B;
  int worst = 1;
  for (size_t g = 0; g + group <= elem_index.size(); g += group) {
    int count[32] = {0};
    // distinct addresses in the same bank conflict; identical addresses broadcast
    std::vector<long> seen;
    for (int l = 0; l < group; ++l) {
      long e = elem_index[g + l];
      bool dup = false;
      for (long s : seen) dup |= (s == e);
      if (dup) continue;
      seen.push_back(e);
      int bank = (int)((e * B / 4) % 32);
      worst = std::max(worst, ++count[bank]);
    }
  }
  return worst;
}

// Runs one tile body (both phases) for `blocks` CTAs on the CPU.
template <class Body, class Tile, class LAY>
static void run_body(const typename Body::Args& a, long blocks) {
  using V = typename Tile::V;
  std::vector<V> smem(Tile::template smem_elems<LAY>());
  std::vector<Tile> thr(Tile::THREADS);
  for (long b = 0; b < blocks; ++b) {
    for (int t = 0; t < Tile::THREADS; ++t) Body::phase1(thr[t], a, b, t, smem.data());
    for (int t = 0; t < Tile::THREADS; ++t) Body::phase2(thr[t], a, b, t, smem.data());
  }
}

// Bank-conflict report for the exchange of a tile: scatter with mapping UF_A, gather with col-fast.
template <class Tile, class LAY, int UF_A, int UF_B = 0>
static void report_conflicts(const char* name) {
  using V = typename Tile::V;
  constexpr int B = (int)sizeof(V);
  int worst_w = 1, worst_r = 1;
  for (int warp = 0; warp < Tile::THREADS / 32; ++warp) {
    for (int a = 0; a < Tile::NA; ++a)
      for (int p = 0; p < Tile::RA; ++p) {
        std::vector<long> idx;
        for (int l = 0; l < 32; ++l) {
          const int t = warp * 32 + l;
          idx.push_back((long)(Tile::template u_of<UF_A>(t) + Tile::TP * a) * LAY::SJ + (long)p * LAY::SP +
                        (long)Tile::template col_of<UF_A>(t) * LAY::SC);
        }
        worst_w = std::max(worst_w, conflict_degree<B>(idx));
      }
    for (int c = 0; c < Tile::NB; ++c)
      for (int j = 0; j < Tile::RB; ++j) {
        std::vector<long> idx;
        for (int l = 0; l < 32; ++l) {
          const int t = warp * 32 + l;
          idx.push_back((long)j * LAY::SJ + (long)(Tile::template u_of<UF_B>(t) + Tile::TP * c) * LAY::SP +
                        (long)Tile::template col_of<UF_B>(t) * LAY::SC);
        }
        worst_r = std::max(worst_r, conflict_degree<B>(idx));
      }
  }
  printf("  %-8s threads %4d smem %6zu B  exchange conflicts: write x%d, read x%d\n", name, Tile::THREADS,
         sizeof(V) * Tile::template smem_elems<LAY>(), worst_w, worst_r);
}

template <typename T, class Cfg>
static int check(const char* name, double tol) {
  const long N = Cfg::N, N1 = Cfg::N1, N2 = Cfg::N2;
  const int batch = 2;
  printf("%s: N=%ld = %ld x %ld\n", name, N, N1, N2);
  report_conflicts<typename Cfg::template Tile1<true>, typename Cfg::Lay1, false>("pass 1");
  report_conflicts<typename Cfg::template Tile2<true>, typename Cfg::Lay2, true>("pass 2");
  int bad = 0;
  for (int fwd = 1; fwd >= 0; --fwd) {
    std::vector<cpx<T>> x((size_t)N * batch), scratch((size_t)N * batch), out((size_t)N * batch);
    fill<T>(x, 7 + fwd);
    const auto* ops = Cfg::ops();
    auto twa1 = make_twa<T>(ops->ra1, ops->rb1), twa2 = make_twa<T>(ops->ra2, ops->rb2);
    std::vector<cpx<T>> tw2(N);
    for (long k1 = 0; k1 < N1; ++k1)
      for (long c = 0; c < N2; ++c) {
        double re, im;
        host_twiddle((size_t)(k1 * c), (size_t)N, &re, &im);
        tw2[k1 * N2 + c] = mk<T>((T)re, (T)im);
      }
    const T scale = (T)0.5;
    if (fwd) {
      run_body<typename Cfg::template Body1<true>, typename Cfg::template Tile1<true>, typename Cfg::Lay1>(
          Cfg::template args1<true>(x.data(), scratch.data(), twa1.data(), tw2.data()), batch * (N2 / Cfg::template Tile1<true>::C));
      run_body<typename Cfg::template Body2<true>, typename Cfg::template Tile2<true>, typename Cfg::Lay2>(
          Cfg::template args2<true>(scratch.data(), out.data(), twa2.data(), scale, true), batch * (N1 / Cfg::template Tile2<true>::C));
    } else {
      run_body<typename Cfg::template Body1<false>, typename Cfg::template Tile1<false>, typename Cfg::Lay1>(
          Cfg::template args1<false>(x.data(), scratch.data(), twa1.data(), tw2.data()), batch * (N2 / Cfg::template Tile1<false>::C));
      run_body<typename Cfg::template Body2<false>, typename Cfg::template Tile2<false>, typename Cfg::Lay2>(
          Cfg::template args2<false>(scratch.data(), out.data(), twa2.data(), scale, true), batch * (N1 / Cfg::template Tile2<false>::C));
    }
    double worst = 0;
    for (int b = 0; b < batch; ++b) {
      std::vector<double> re(N), im(N);
      for (long i = 0; i < N; ++i) { re[i] = x[(size_t)b * N + i].x; im[i] = x[(size_t)b * N + i].y; }
      host_fft_pow2(re, im, !fwd);
      double maxref = 0, maxerr = 0;
      for (long i = 0; i < N; ++i) {
        const double rr = re[i] * 0.5, ii = im[i] * 0.5;
        maxref = std::max(maxref, std::hypot(rr, ii));
        maxerr = std::max(maxerr, std::hypot(out[(size_t)b * N + i].x - rr, out[(size_t)b * N + i].y - ii));
      }
      worst = std::max(worst, maxerr / maxref);
    }
    printf("  %s: max rel err vs f64 FFT %.3e (tol %.1e) %s\n", fwd ? "forward" : "inverse", worst, tol,
           worst < tol ? "OK" : "FAIL");
    bad += !(worst < tol);
  }
  return bad;
}

// ---- on-chip kernels (onchip_kernels.cuh) -------------------------------------------------------------------------
template <typename T, int RA, int RB, int E, int WARPS>
static int check_onchip(const char* name, double tol) {
  int bad = 0;
  for (int fwd = 1; fwd >= 0; --fwd) {
    const long L = RA * RB, batch = 5;   // 5 is not a multiple of the transforms per CTA: exercises the tail
    std::vector<cpx<T>> x((size_t)L * batch), out((size_t)L * batch);
    fill<T>(x, 21 + fwd);
    auto twa = make_twa<T>(RA, RB);
    auto run = [&](auto cfg_tag) {
      using Cfg = decltype(cfg_tag);
      using Body = onchip::FftBody<Cfg>;
      typename Body::Args a = {x.data(), out.data(), twa.data(), batch, (T)0.5, 1};
      std::vector<cpx<T>> smem(Cfg::Tile::template smem_elems<typename Cfg::Lay>());
      std::vector<typename Cfg::Tile> thr(Cfg::THREADS);
      const long groups = (batch + Cfg::C - 1) / Cfg::C;
      for (long g = 0; g < groups; ++g) {
        for (int t = 0; t < Cfg::THREADS; ++t) Body::phase1(thr[t], a, g, t, smem.data(), twa.data());
        for (int t = 0; t < Cfg::THREADS; ++t) Body::phase2(thr[t], a, g, t, smem.data());
      }
      report_conflicts<typename Cfg::Tile, typename Cfg::Lay, true, true>("exchange");
    };
    if (fwd) run(onchip::OnChipCfg<T, RA, RB, E, WARPS, true>{}); else run(onchip::OnChipCfg<T, RA, RB, E, WARPS, false>{});
    double worst = 0;
    for (long b = 0; b < batch; ++b) {
      std::vector<double> re(L), im(L);
      for (long i = 0; i < L; ++i) { re[i] = x[b * L + i].x; im[i] = x[b * L + i].y; }
      host_fft_pow2(re, im, !fwd);
      double mr = 0, me = 0;
      for (long i = 0; i < L; ++i) {
        mr = std::max(mr, std::hypot(re[i], im[i]) * 0.5);
        me = std::max(me, std::hypot(out[b * L + i].x - 0.5 * re[i], out[b * L + i].y - 0.5 * im[i]));
      }
      worst = std::max(worst, me / mr);
    }
    printf("%s L=%d %s: max rel err %.3e %s\n", name, RA * RB, fwd ? "forward" : "inverse", worst, worst < tol ? "OK" : "FAIL");
    bad += !(worst < tol);
  }
  return bad;
}

template <typename T, int R, int WARPS>
static int check_bluestein(const char* name, long n, double tol) {
  using Cfg = onchip::OnChipCfg<T, R, R, R, WARPS, true>;
  using Body = onchip::BluesteinBody<Cfg>;
  using V = cpx<T>;
  const long L = R * R, M = 2 * L, batch = 3;
  int bad = 0;
  for (int inverse = 0; inverse < 2; ++inverse) {
    // tables exactly as Plan<T>::init_bluestein / init_bluestein_fused build them
    std::vector<double> cr(n), ci(n), wr(M, 0.0), wi(M, 0.0);
    for (long i = 0; i < n; ++i) {
      const size_t idx = (size_t)(((unsigned __int128)i * i) % (2 * (unsigned __int128)n));
      host_twiddle(idx, 2 * n, &cr[i], &ci[i]);
      wr[i] = cr[i]; wi[i] = -ci[i];
      if (i) { wr[M - i] = cr[i]; wi[M - i] = -ci[i]; }
    }
    host_fft_pow2(wr, wi, false);
    const double sgn = inverse ? -1.0 : 1.0;
    std::vector<V> chirp(L, mk<T>(0, 0)), wm(L), wce(L), wco(L);
    for (long i = 0; i < L; ++i) {
      if (i < n) chirp[i] = mk<T>((T)cr[i], (T)(sgn * ci[i]));
      double re, im;
      host_twiddle(i, M, &re, &im);
      wm[i] = mk<T>((T)re, (T)im);
      wce[i] = mk<T>((T)wr[2 * i], (T)(-sgn * wi[2 * i]));
      wco[i] = mk<T>((T)wr[2 * i + 1], (T)(-sgn * wi[2 * i + 1]));
    }
    auto twa = make_twa<T>(R, R);
    std::vector<V> x((size_t)n * batch), out((size_t)n * batch);
    fill<T>(x, 31 + inverse);
    typename Body::Args a = {x.data(), out.data(), twa.data(), chirp.data(), wm.data(), wce.data(), wco.data(), n, batch,
                             (T)(1.0 / M)};
    std::vector<V> exch(Cfg::Tile::template smem_elems<typename Cfg::Lay>());
    std::vector<V> stash((size_t)R * Cfg::THREADS);
    std::vector<typename Cfg::Tile> thr(Cfg::THREADS);
    const long groups = (batch + Cfg::C - 1) / Cfg::C;
    auto all = [&](auto fn) { for (int t = 0; t < Cfg::THREADS; ++t) fn(t); };
    for (long g = 0; g < groups; ++g) {
      auto bidx = [&](int t) { long b = g * Cfg::C + Cfg::Tile::template col_of<true>(t); return b; };
      auto bcl = [&](int t) { long b = bidx(t); return b < batch ? b : batch - 1; };
      for (int odd = 0; odd < 2; ++odd) {
        all([&](int t) { if (odd) Body::template load_half<true>(thr[t], a, bcl(t), t, exch.data(), twa.data(), chirp.data(), wm.data());
                         else Body::template load_half<false>(thr[t], a, bcl(t), t, exch.data(), twa.data(), chirp.data(), wm.data()); });
        all([&](int t) { Body::middle(thr[t], t, exch.data(), odd ? wco.data() : wce.data()); });
        all([&](int t) { Body::second_fft_start(thr[t], t, exch.data(), twa.data()); });
        all([&](int t) { Body::second_fft_finish(thr[t], t, exch.data()); });
        if (!odd) all([&](int t) { Body::stash_even(thr[t], t, stash.data()); });
      }
      all([&](int t) { if (bidx(t) < batch) Body::combine_store(stash.data(), thr[t], a, bcl(t), t, chirp.data(), wm.data()); });
    }
    double worst = 0;
    for (long b = 0; b < batch; ++b) {
      double mr = 0, me = 0;
      for (long k = 0; k < n; ++k) {
        double sr = 0, si = 0;
        for (long j = 0; j < n; ++j) {
          double re, im;
          host_twiddle((size_t)((k * j) % n), (size_t)n, &re, &im);
          if (inverse) im = -im;
          sr += x[b * n + j].x * re - x[b * n + j].y * im;
          si += x[b * n + j].x * im + x[b * n + j].y * re;
        }
        mr = std::max(mr, std::hypot(sr, si));
        me = std::max(me, std::hypot(out[b * n + k].x - sr, out[b * n + k].y - si));
      }
      worst = std::max(worst, me / mr);
    }
    printf("%s N=%ld (L=%ld) %s: max rel err vs naive f64 DFT %.3e %s\n", name, n, L, inverse ? "inverse" : "forward", worst,
           worst < tol ? "OK" : "FAIL");
    bad += !(worst < tol);
  }
  return bad;
}

// ---- persistent kernel: the consumer arithmetic (fused::FusedMath) with the producer / TMA side replaced by
// plain copies: staging = what the TMA box (pass 1) or the bulk copy (pass 2) would deliver --------------------------
template <class Cfg>
static int check_fused(const char* name, double tol) {
  using T = typename Cfg::T;
  using V = cpx<T>;
  constexpr long N = Cfg::N, N1 = Cfg::N1, N2 = Cfg::N2;
  constexpr int C = Cfg::C, C1 = Cfg::C1, GT = Cfg::GT;
  printf("%s: persistent-kernel arithmetic, N=%ld = %ld x %ld, blocked intermediate%s\n", name, N, N1, N2, Cfg::DIRECT ? ", direct loads" : "");
  report_conflicts<typename Cfg::template Tile1<true>, typename Cfg::Lay1, kMapCF>("pass 1");
  report_conflicts<typename Cfg::template Tile2<true>, typename Cfg::Lay2, fused::FusedMath<Cfg, true>::kMap2>("pass 2");
  {  // staging reads of pass 2 (the other staging / table reads are contiguous by construction)
    using Tile = typename Cfg::template Tile2<true>;
    int worst = 1;
    for (int warp = 0; warp < GT / 32; ++warp)
      for (int i = 0; i < Tile::RA; ++i) {
        std::vector<long> idx;
        for (int l = 0; l < 32; ++l) {
          const int t = warp * 32 + l;
          constexpr int M = fused::FusedMath<Cfg, true>::kMap2;
          const long u = Tile::template u_of<M>(t), col = Tile::template col_of<M>(t), n = u + (long)Tile::RB * i;
          idx.push_back((n / 8) * 64 + col * 8 + n % 8);
        }
        worst = std::max(worst, conflict_degree<(int)sizeof(V)>(idx));
      }
    printf("  pass 2 staging reads: conflicts x%d %s\n", worst, worst == 1 ? "" : "FAIL");
    if (worst != 1) return 1;
  }
  {  // LSU cost model of the two accesses the blocked layout changes: 128-byte lines touched by one warp-wide
     // pass-1 store, and different stage twiddles one warp loads in pass 2 (identical addresses broadcast)
    using Tile = typename Cfg::template Tile1<true>;
    using TileB = typename Cfg::template Tile2<true>;
    constexpr int M = fused::FusedMath<Cfg, true>::kMap2;
    long lines = 0, twiddles = 0;
    for (int warp = 0; warp < GT / 32; ++warp) {
      std::vector<long> seen_l, seen_t;
      for (int l = 0; l < 32; ++l) {
        const int t = warp * 32 + l;
        const long col = Tile::template col_of<kMapCF>(t), p = Tile::template u_of<kMapCF>(t);
        const long e = (p >> 3) * (N2 * 8) + (col >> 3) * 64 + (p & 7) * 8 + (col & 7);   // output r = 0
        const long line = e * (long)sizeof(V) / 128, tw = TileB::template u_of<M>(t);
        if (std::find(seen_l.begin(), seen_l.end(), line) == seen_l.end()) seen_l.push_back(line);
        if (std::find(seen_t.begin(), seen_t.end(), tw) == seen_t.end()) seen_t.push_back(tw);
      }
      lines += (long)seen_l.size();
      twiddles += (long)seen_t.size();
    }
    printf("  per warp: %.1f lines of 128 B per pass-1 store instruction (%d B stored), %.1f different pass-2 stage twiddles\n",
           (double)lines / (GT / 32), 32 * (int)sizeof(V), (double)twiddles / (GT / 32));
  }
  auto twa_pairs = make_twa<T>(Cfg::RA, Cfg::RB), twa2_pairs = make_twa<T>(Cfg::RA2, Cfg::RB2);
  std::vector<TwPair<T>> twa(twa_pairs.size()), twa2(twa2_pairs.size());     // the kernel re-lays the tables out in 8-byte planes
  for (int i = 0; i < (int)twa_pairs.size(); ++i) fused::FusedMath<Cfg, true>::relayout_twa(twa.data(), twa_pairs.data(), i, (int)twa_pairs.size());
  for (int i = 0; i < (int)twa2_pairs.size(); ++i) fused::FusedMath<Cfg, true>::relayout_twa(twa2.data(), twa2_pairs.data(), i, (int)twa2_pairs.size());
  std::vector<V> tbase, tstep;
  make_factored_twiddles<T>((size_t)N, (size_t)N2, Cfg::RA, Cfg::RB, C1, tbase, tstep, true);
  int bad = 0;
  for (int fwd = 1; fwd >= 0; --fwd) {
    std::vector<V> x(N), scratch(N), out(N), staging(std::max((size_t)C1 * N1, (size_t)C * N2)), tab((size_t)Cfg::TAB_ELEMS);
    std::vector<V> exch(Cfg::EX_ELEMS);
    fill<T>(x, 41 + fwd);
    const T scale = (T)0.5;
    auto run_tile = [&](auto fwd_tag, auto pass_tag, int tile) {
      constexpr bool FWD = decltype(fwd_tag)::value;
      constexpr int PASS = decltype(pass_tag)::value;
      using Math = fused::FusedMath<Cfg, FWD>;
      using P = typename Math::template Pass<PASS>;
      std::vector<typename P::Tile> thr(GT);
      // direct mode: the threads read global memory themselves (same pointers as the kernel computes)
      const V* src = !Cfg::DIRECT ? staging.data() : PASS == 1 ? x.data() + (size_t)tile * C1
                                                                : scratch.data() + (size_t)tile * C * N2;
      for (int t = 0; t < GT; ++t) { P::load(thr[t], t, src); P::stage_a(thr[t], t, PASS == 1 ? twa.data() : twa2.data()); }
      for (int t = 0; t < GT; ++t) P::scatter(thr[t], t, exch.data());
      for (int t = 0; t < GT; ++t) {
        P::gather(thr[t], t, exch.data());
        thr[t].stage_b();
        if constexpr (PASS == 1) Math::store1(thr[t], t, scratch.data(), tile, tab.data(), tab.data() + Cfg::TAB_BASE);
        else Math::store2(thr[t], t, out.data(), tile, true, scale);
      }
    };
    using One = std::integral_constant<int, 1>;
    using Two = std::integral_constant<int, 2>;
    for (int tile = 0; tile < Cfg::T1; ++tile) {        // pass 1: TMA box = rows n1, columns tile*C .. +C
      for (long r = 0; r < N1; ++r)
        for (int c = 0; c < C1; ++c) staging[r * C1 + c] = x[r * N2 + (long)tile * C1 + c];
      for (int i = 0; i < Cfg::TAB_BASE; ++i) tab[i] = tbase[(size_t)tile * Cfg::TAB_BASE + i];
      for (int i = 0; i < Cfg::TAB_STEP; ++i) tab[Cfg::TAB_BASE + i] = tstep[(size_t)tile * Cfg::TAB_STEP + i];
      if (fwd) run_tile(std::true_type{}, One{}, tile); else run_tile(std::false_type{}, One{}, tile);
    }
    for (int tile = 0; tile < Cfg::T2; ++tile) {        // pass 2: bulk copy of C*N2 contiguous samples
      for (long i = 0; i < (long)C * N2; ++i) staging[i] = scratch[(size_t)tile * C * N2 + i];
      if (fwd) run_tile(std::true_type{}, Two{}, tile); else run_tile(std::false_type{}, Two{}, tile);
    }
    std::vector<double> re(N), im(N);
    for (long i = 0; i < N; ++i) { re[i] = x[i].x; im[i] = x[i].y; }
    host_fft_pow2(re, im, !fwd);
    double maxref = 0, maxerr = 0;
    for (long i = 0; i < N; ++i) {
      maxref = std::max(maxref, std::hypot(re[i], im[i]) * 0.5);
      maxerr = std::max(maxerr, std::hypot(out[i].x - 0.5 * re[i], out[i].y - 0.5 * im[i]));
    }
    printf("  %s: max rel err vs f64 FFT %.3e (tol %.1e) %s\n", fwd ? "forward" : "inverse", maxerr / maxref, tol,
           maxerr / maxref < tol ? "OK" : "FAIL");
    bad += !(maxerr / maxref < tol);
  }
  return bad;
}

// ---- work queue of the fused kernel: order and dependency properties ---------------------------------------------
static int check_queue() {
  int bad = 0;
  const int t1 = 128, t2 = 128;
  for (int batch : {1, 2, 3, 5, 8, 17, 64}) {
    for (int lag : {1, 2, 3, 4, 7}) {
      for (int ring : {lag + 1, 2 * lag + 2}) {
        const long total = (long)batch * (t1 + t2);
        std::vector<long> pos1((size_t)batch * t1, -1), pos2((size_t)batch * t2, -1);
        bool ok = true;
        for (long w = 0; w < total; ++w) {
          const fused::WorkItem it = fused::decode_work(w, batch, lag, t1, t2);
          if (it.pass == 1 && it.b >= 0 && it.b < batch && it.tile >= 0 && it.tile < t1 && pos1[(size_t)it.b * t1 + it.tile] < 0)
            pos1[(size_t)it.b * t1 + it.tile] = w;
          else if (it.pass == 2 && it.b >= 0 && it.b < batch && it.tile >= 0 && it.tile < t2 && pos2[(size_t)it.b * t2 + it.tile] < 0)
            pos2[(size_t)it.b * t2 + it.tile] = w;
          else ok = false;   // out of range or duplicate
        }
        ok = ok && fused::decode_work(total, batch, lag, t1, t2).pass < 0;   // exhausted marker
        for (int b = 0; b < batch && ok; ++b) {
          long last1 = 0, first2 = total, last2 = 0, first1 = total;
          for (int t = 0; t < t1; ++t) { last1 = std::max(last1, pos1[(size_t)b * t1 + t]); first1 = std::min(first1, pos1[(size_t)b * t1 + t]); }
          for (int t = 0; t < t2; ++t) { first2 = std::min(first2, pos2[(size_t)b * t2 + t]); last2 = std::max(last2, pos2[(size_t)b * t2 + t]); }
          if (first1 < 0 || first2 < 0) ok = false;                     // every tile appears
          if (!(last1 < first2)) ok = false;                            // pass 2 of b only depends on earlier items
          if (b + ring < batch) {                                       // slot reuse: pass 1 of b+ring after pass 2 of b
            long f = total;
            for (int t = 0; t < t1; ++t) f = std::min(f, pos1[(size_t)(b + ring) * t1 + t]);
            if (!(last2 < f)) ok = false;
          }
        }
        if (!ok) { printf("queue order FAILED batch=%d lag=%d ring=%d\n", batch, lag, ring); ++bad; }
      }
    }
  }
  printf("fused work queue: permutation / dependency-order properties %s\n", bad ? "FAILED" : "OK");
  return bad;
}

// ---- CTA-level shared-memory Stockham kernel (cta_kernels.cuh): every step for every thread, barrier = loop end ----
template <typename T>
static int check_cta(const char* name, int n, bool chirp_mode, double tol) {
  using V = cpx<T>;
  int len = n;
  if (chirp_mode) { len = 1; while (len < 2 * n - 1) len *= 2; }
  cta::Args<T> a;
  if (!cta::factorize((size_t)len, a.st)) { printf("%s N=%d: cannot factorize\n", name, n); return 1; }
  const int group = std::max(1, (int)(32768 / sizeof(V)) / len), batch = group + 1;   // a full and a partial group
  std::vector<V> wtab = cta::make_stage_twiddles<T>((size_t)len, a.st, host_twiddle);
  std::vector<V> chirp(n), wf(len), x((size_t)batch * n), out((size_t)batch * n);
  if (chirp_mode) {
    std::vector<double> wr(len, 0.0), wi(len, 0.0);
    for (int i = 0; i < n; ++i) {
      double re, im;
      host_twiddle((size_t)(((unsigned long long)i * i) % (2ull * n)), 2 * (size_t)n, &re, &im);
      chirp[i] = mk<T>((T)re, (T)im);
      wr[i] = re; wi[i] = -im;
      if (i) { wr[len - i] = re; wi[len - i] = -im; }
    }
    host_fft_pow2(wr, wi, false);
    for (int i = 0; i < len; ++i) wf[i] = mk<T>((T)wr[i], (T)wi[i]);
  }
  fill<T>(x, 77 + n);
  a.in = x.data(); a.out = out.data(); a.wtab = wtab.data(); a.chirp = chirp.data(); a.wf = wf.data();
  a.batch = batch; a.n = n; a.len = len; a.group = group; a.pad = a.st.radix[0] % 2 == 0 ? 1 : 0;
  printf("%s N=%d%s: on-chip length %d, stages", name, n, chirp_mode ? " (chirp-z)" : "", len);
  for (int i = 0; i < a.st.count; ++i) printf(" %d", a.st.radix[i]);
  printf(", %d transforms per CTA iteration\n", group);
  // bank conflicts of the shared-memory accesses, worst warp-wide instruction per stage
  {
    int sub = len, stride = 1;
    for (int sidx = 0; sidx < a.st.count; ++sidx) {
      const int R = a.st.radix[sidx], per = len / R, m = sub / R;
      int worst_r = 1, worst_w = 1;
      for (int warp = 0; warp < std::min(cta::kThreads, group * per) / 32; ++warp)
        for (int k = 0; k < R; ++k) {
          std::vector<long> ri, wi2;
          for (int l = 0; l < 32; ++l) {
            const int g = warp * 32 + l, tl = g / per, q = g - tl * per, i = q / stride, j = q - i * stride;
            const int er = tl * len + (k * m + i) * stride + j, ew = tl * len + (i * R + k) * stride + j;
            ri.push_back(a.pad ? cta::padded(er) : er);
            wi2.push_back(a.pad ? cta::padded(ew) : ew);
          }
          worst_r = std::max(worst_r, conflict_degree<(int)sizeof(V)>(ri));
          worst_w = std::max(worst_w, conflict_degree<(int)sizeof(V)>(wi2));
        }
      printf("  stage %d (radix %2d, stride %5d): shared read conflicts x%d, write x%d\n", sidx, R, stride, worst_r, worst_w);
      sub /= R; stride *= R;
    }
  }
  int bad = 0;
  std::vector<V> buf0((size_t)cta::padded(group * len) + 1), buf1(buf0.size());
  for (int dir = 1; dir >= 0; --dir) {
    a.scale = (T)(chirp_mode ? 0.5 / len : 0.5);
    for (long first = 0; first < batch; first += group) {
      const int cnt = (int)std::min<long>(group, batch - first);
      auto run = [&](auto D, auto Cm) {
        using P = cta::Program<T, decltype(D)::value, decltype(Cm)::value>;
        for (int st = 0; st < P::steps(a); ++st)
          for (int tid = 0; tid < cta::kThreads; ++tid) P::step(a, st, tid, cta::kThreads, first, cnt, buf0.data(), buf1.data());
      };
      if (dir && chirp_mode) run(std::true_type{}, std::true_type{});
      else if (dir) run(std::true_type{}, std::false_type{});
      else if (chirp_mode) run(std::false_type{}, std::true_type{});
      else run(std::false_type{}, std::false_type{});
    }
    double worst = 0;
    for (int b = 0; b < batch; ++b) {
      double me = 0, mr = 0;
      for (int k = 0; k < n; ++k) {
        double sr = 0, si = 0;
        for (int j = 0; j < n; ++j) {
          double re, im;
          host_twiddle((size_t)(((unsigned long long)j * k) % n), (size_t)n, &re, &im);
          if (!dir) im = -im;
          const double xr = x[(size_t)b * n + j].x, xi = x[(size_t)b * n + j].y;
          sr += xr * re - xi * im; si += xr * im + xi * re;
        }
        sr *= 0.5; si *= 0.5;
        me = std::max(me, std::hypot(out[(size_t)b * n + k].x - sr, out[(size_t)b * n + k].y - si));
        mr = std::max(mr, std::hypot(sr, si));
      }
      worst = std::max(worst, me / mr);
    }
    printf("  %s: max rel err vs naive f64 DFT %.3e %s\n", dir ? "forward" : "inverse", worst, worst < tol ? "OK" : "FAIL");
    bad += !(worst < tol);
  }
  return bad;
}

// ---- row FFTs with the exchange folded into the store of pass 2 (dist_kernels.cuh) -----------------------------
// pass 1 of the configuration as it is, then RowsExchangeBody with P destination buffers in host memory; reference:
// dst_q[c * out_ld + out_off + r] = FFT(row r)[q * cb + c] * w_Ntot^{(row0 + r) * (q * cb + c)}
// SW: shape of the tile (default: the configuration's pass-2 shape; dist_fft.cu also uses tiles of twice as many
// transforms, WideShape)
template <typename T, class Cfg, int TW, class SW = typename Cfg::Shape2>
static int check_rows_exchange(const char* name, int P, double tol) {
  constexpr bool FWD = TW != 2;
  const long N = Cfg::N, N1 = Cfg::N1, N2 = Cfg::N2;
  using Tile = TileFFT<T, SW::RA, SW::RB, SW::E, SW::C, FWD>;
  using LayX = ExLayout<SW::RA * SW::C + SW::PAD, SW::C, 1>;
  report_conflicts<Tile, LayX, true>("exchange tile");
  using Body = dist::RowsExchangeBody<Tile, LayX, Cfg::N1, Cfg::N2, TW>;
  const long rows = 2 * Tile::C, cb = N / P;
  const unsigned long long row0 = 12345, n_total = (unsigned long long)N * 4096, out_off = 3 * rows, out_ld = 5 * rows;
  std::vector<cpx<T>> x((size_t)N * rows), scratch((size_t)N * rows);
  fill<T>(x, 21 + TW);
  const auto* ops = Cfg::ops();
  auto twa1 = make_twa<T>(ops->ra1, ops->rb1), twa2 = make_twa<T>(ops->ra2, ops->rb2);
  std::vector<cpx<T>> tw2(N);
  for (long k1 = 0; k1 < N1; ++k1)
    for (long c = 0; c < N2; ++c) {
      double re, im;
      host_twiddle((size_t)(k1 * c), (size_t)N, &re, &im);
      tw2[k1 * N2 + c] = mk<T>((T)re, (T)im);
    }
  run_body<typename Cfg::template Body1<FWD>, typename Cfg::template Tile1<FWD>, typename Cfg::Lay1>(
      Cfg::template args1<FWD>(x.data(), scratch.data(), twa1.data(), tw2.data()), rows * (N2 / Cfg::template Tile1<FWD>::C));
  std::vector<std::vector<cpx<T>>> dst(P, std::vector<cpx<T>>((size_t)cb * out_ld, mk<T>((T)777, (T)777)));
  typename Body::Args a;
  a.scratch = scratch.data(); a.twa = twa2.data();
  for (int q = 0; q < kMaxPeers; ++q) a.outs.p[q] = q < P ? dst[q].data() : nullptr;
  a.out_ld = out_ld; a.out_off = out_off; a.row0 = row0; a.n_total = n_total; a.groups = (unsigned)(rows / Tile::C);
  a.r0 = 0; a.out_bs = 0; a.rb_shift = 63; a.rpb = 0; a.rows_valid = ~0ull;
  a.cb_shift = 0;
  while ((1L << a.cb_shift) < cb) ++a.cb_shift;
  run_body<Body, Tile, LayX>(a, (long)a.groups * N1);
  double worst = 0, maxref = 0;
  for (long r = 0; r < rows; ++r) {
    std::vector<double> re(N), im(N);
    for (long i = 0; i < N; ++i) { re[i] = x[(size_t)r * N + i].x; im[i] = x[(size_t)r * N + i].y; }
    host_fft_pow2(re, im, !FWD);
    for (long k = 0; k < N; ++k) {
      double wr = 1, wi = 0;
      if (TW) {
        const unsigned long long m = (row0 + r) * (unsigned long long)k % n_total;
        const double ang = 2 * M_PI * (double)m / (double)n_total;
        wr = std::cos(ang); wi = TW == 1 ? -std::sin(ang) : std::sin(ang);
      }
      const double rr = re[k] * wr - im[k] * wi, ii = re[k] * wi + im[k] * wr;
      const cpx<T> got = dst[k / cb][(size_t)(k % cb) * out_ld + out_off + r];
      maxref = std::max(maxref, std::hypot(rr, ii));
      worst = std::max(worst, std::hypot(got.x - rr, got.y - ii));
    }
  }
  // nothing outside the chunk's columns may be written
  long stray = 0;
  for (int q = 0; q < P; ++q)
    for (long c = 0; c < cb; ++c)
      for (long j = 0; j < (long)out_ld; ++j)
        if ((j < (long)out_off || j >= (long)out_off + rows) && dst[q][(size_t)c * out_ld + j].x != (T)777) ++stray;
  const double rel = worst / maxref;
  printf("%s rows+exchange (P=%d, twiddle %d): max rel err %.3e (tol %.1e), stray stores %ld %s\n", name, P, TW, rel, tol, stray,
         rel < tol && stray == 0 ? "OK" : "FAIL");
  return !(rel < tol && stray == 0);
}

// ---- three-pass path (bigpow2.cu): outer column pass + two-pass rows with the transposed store ---------------------
template <typename T, class SO, class Cfg, bool FWD>
static int check_threepass(const char* name, double tol) {
  const long Na = SO::L, Nb = Cfg::N, N = Na * Nb;
  using TileO = TileFFT<T, SO::RA, SO::RB, SO::E, SO::C, FWD>;
  using LayO = ExLayout<SO::RA * SO::C + SO::PAD, SO::C, 1>;
  using BodyO = outer::ColumnBody<TileO, LayO>;
  const long B = 2;   // two long transforms in one call
  std::vector<cpx<T>> x(B * N), work(B * N), scratch(B * N), out(B * N);
  fill<T>(x, 31 + FWD);
  auto twao = make_twa<T>(SO::RA, SO::RB);
  typename BodyO::Args ao;
  ao.in = x.data(); ao.out = work.data(); ao.twa = twao.data(); ao.nb = Nb; ao.n_total = N; ao.tiles = (unsigned)(Nb / SO::C);
  ao.scale = (T)0.5;
  run_body<BodyO, TileO, LayO>(ao, B * (Nb / SO::C));
  const auto* ops = Cfg::ops();
  auto twa1 = make_twa<T>(ops->ra1, ops->rb1), twa2 = make_twa<T>(ops->ra2, ops->rb2);
  std::vector<cpx<T>> tw2(Nb);
  for (long k1 = 0; k1 < Cfg::N1; ++k1)
    for (long c = 0; c < Cfg::N2; ++c) {
      double re, im;
      host_twiddle((size_t)(k1 * c), (size_t)Nb, &re, &im);
      tw2[k1 * Cfg::N2 + c] = mk<T>((T)re, (T)im);
    }
  run_body<typename Cfg::template Body1<FWD>, typename Cfg::template Tile1<FWD>, typename Cfg::Lay1>(
      Cfg::template args1<FWD>(work.data(), scratch.data(), twa1.data(), tw2.data()), B * Na * (Cfg::N2 / Cfg::template Tile1<FWD>::C));
  using Tile = typename Cfg::template Tile2<FWD>;
  using Body = dist::RowsExchangeBody<Tile, typename Cfg::Lay2, Cfg::N1, Cfg::N2, 0>;
  typename Body::Args a;
  a.scratch = scratch.data(); a.twa = twa2.data();
  for (int q = 0; q < kMaxPeers; ++q) a.outs.p[q] = q == 0 ? out.data() : nullptr;
  a.out_ld = Na; a.out_off = 0; a.row0 = 0; a.n_total = 0; a.groups = (unsigned)(B * Na / Tile::C);
  a.r0 = 0; a.out_bs = N; a.rb_shift = 0; a.rpb = 0; a.rows_valid = ~0ull;
  while ((1L << a.rb_shift) < Na) ++a.rb_shift;
  a.cb_shift = 0;
  while ((1L << a.cb_shift) < Nb) ++a.cb_shift;
  run_body<Body, Tile, typename Cfg::Lay2>(a, (long)a.groups * Cfg::N1);
  double maxref = 0, maxerr = 0;
  for (long bb = 0; bb < B; ++bb) {
    std::vector<double> re(N), im(N);
    for (long i = 0; i < N; ++i) { re[i] = x[bb * N + i].x; im[i] = x[bb * N + i].y; }
    host_fft_pow2(re, im, !FWD);
    for (long i = 0; i < N; ++i) {
      maxref = std::max(maxref, std::hypot(re[i] * 0.5, im[i] * 0.5));
      maxerr = std::max(maxerr, std::hypot(out[bb * N + i].x - re[i] * 0.5, out[bb * N + i].y - im[i] * 0.5));
    }
  }
  printf("%s three-pass %ld x %ld (%s): max rel err %.3e (tol %.1e) %s\n", name, Na, Nb, FWD ? "forward" : "inverse",
         maxerr / maxref, tol, maxerr / maxref < tol ? "OK" : "FAIL");
  return !(maxerr / maxref < tol);
}

// ---- three-pass path with an outer radix-3 / 9 / 27 pass (N = 3^b * 2^k, bigpow2.cu) ---------------------------------
template <typename T, int B, class Cfg, bool FWD>
static int check_threepass_radix3(const char* name, double tol) {
  const long Nb = Cfg::N, N = B * Nb, BATCH = 2;
  using Tile = typename Cfg::template Tile2<FWD>;
  const long rows = BATCH * B, rows_pad = (rows + Tile::C - 1) / Tile::C * Tile::C;
  std::vector<cpx<T>> x(BATCH * N), work(rows_pad * Nb, mk<T>((T)NAN, (T)NAN)), scratch(rows_pad * Nb), out(BATCH * N, mk<T>((T)777, (T)777));
  fill<T>(x, 41 + B);
  using BodyO = outer::Radix3ColumnBody<T, B, FWD>;
  typename BodyO::Args ao;
  ao.in = x.data(); ao.out = work.data(); ao.nb = Nb; ao.n_total = N; ao.count = BATCH * Nb; ao.scale = (T)0.5;
  for (long i = 0; i < BATCH * Nb + 7; ++i) BodyO::run(ao, i);          // a few threads beyond the end, as the grid has
  const auto* ops = Cfg::ops();
  auto twa1 = make_twa<T>(ops->ra1, ops->rb1), twa2 = make_twa<T>(ops->ra2, ops->rb2);
  std::vector<cpx<T>> tw2(Nb);
  for (long k1 = 0; k1 < Cfg::N1; ++k1)
    for (long c = 0; c < Cfg::N2; ++c) {
      double re, im;
      host_twiddle((size_t)(k1 * c), (size_t)Nb, &re, &im);
      tw2[k1 * Cfg::N2 + c] = mk<T>((T)re, (T)im);
    }
  run_body<typename Cfg::template Body1<FWD>, typename Cfg::template Tile1<FWD>, typename Cfg::Lay1>(
      Cfg::template args1<FWD>(work.data(), scratch.data(), twa1.data(), tw2.data()), rows_pad * (Cfg::N2 / Cfg::template Tile1<FWD>::C));
  using Body = dist::RowsExchangeBody<Tile, typename Cfg::Lay2, Cfg::N1, Cfg::N2, 0>;
  typename Body::Args a;
  a.scratch = scratch.data(); a.twa = twa2.data();
  for (int q = 0; q < kMaxPeers; ++q) a.outs.p[q] = q == 0 ? out.data() : nullptr;
  a.out_ld = B; a.out_off = 0; a.row0 = 0; a.n_total = 0; a.groups = (unsigned)(rows_pad / Tile::C);
  a.r0 = 0; a.out_bs = N; a.rb_shift = 63; a.rpb = B; a.rows_valid = rows;
  a.cb_shift = 0;
  while ((1L << a.cb_shift) < Nb) ++a.cb_shift;
  run_body<Body, Tile, typename Cfg::Lay2>(a, (long)a.groups * Cfg::N1);
  double maxref = 0, maxerr = 0;
  for (long bb = 0; bb < BATCH; ++bb) {                                   // naive DFT of a few outputs + an FFT-free check
    std::vector<double> re(N), im(N);
    for (long i = 0; i < N; ++i) { re[i] = x[bb * N + i].x; im[i] = x[bb * N + i].y; }
    for (long k = 0; k < N; k += (k < 40 ? 1 : N / 97 + 1)) {
      double sr = 0, si = 0;
      for (long n = 0; n < N; ++n) {
        const double ang = (FWD ? -2.0 : 2.0) * M_PI * (double)((k * n) % N) / (double)N;
        sr += re[n] * std::cos(ang) - im[n] * std::sin(ang);
        si += re[n] * std::sin(ang) + im[n] * std::cos(ang);
      }
      maxref = std::max(maxref, std::hypot(sr * 0.5, si * 0.5));
      maxerr = std::max(maxerr, std::hypot(out[bb * N + k].x - sr * 0.5, out[bb * N + k].y - si * 0.5));
    }
  }
  long untouched = 0, nans = 0;
  for (auto& v : out) { untouched += v.x == (T)777; nans += std::isnan(v.x); }
  printf("%s three-pass %d x %ld (%s): max rel err %.3e (tol %.1e), unwritten %ld, nan %ld %s\n", name, B, Nb, FWD ? "forward" : "inverse",
         maxerr / maxref, tol, untouched, nans, maxerr / maxref < tol && untouched == 0 && nans == 0 ? "OK" : "FAIL");
  return !(maxerr / maxref < tol && untouched == 0 && nans == 0);
}

int main() {
  int bad = 0;
  bad += check_threepass_radix3<float, 3, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, true>("f32 3*2^11", 2e-6);
  bad += check_threepass_radix3<float, 9, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, false>("f32 9*2^11", 2e-6);
  bad += check_threepass_radix3<float, 27, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, true>("f32 27*2^11", 2e-6);
  bad += check_threepass_radix3<double, 27, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, false>("f64 27*2^9", 1e-14);
  bad += check_threepass_radix3<double, 3, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, true>("f64 3*2^9", 1e-14);
  bad += check_threepass<float, Shape<4, 8, 8, 32, 0>, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, true>("f32 2^16", 2e-6);
  bad += check_threepass<float, Shape<8, 16, 16, 16, 0>, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, false>("f32 2^18", 2e-6);
  bad += check_threepass<double, Shape<4, 4, 4, 16, 0>, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, true>("f64 2^13", 5e-15);
  bad += check_threepass<double, Shape<8, 16, 16, 8, 4>, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, false>("f64 2^16", 5e-15);
  // the remaining outer-pass shapes of bigpow2.cu's column_lookup
  bad += check_threepass<float, Shape<8, 8, 8, 32, 0>, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, true>("f32 2^17", 2e-6);
  bad += check_threepass<float, Shape<16, 16, 16, 16, 0>, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, true>("f32 2^19", 2e-6);
  bad += check_threepass<float, Shape<16, 32, 32, 8, 8>, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, false>("f32 2^20", 2e-6);
  bad += check_threepass<float, Shape<32, 32, 32, 8, 8>, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, true>("f32 2^21", 2e-6);
  bad += check_threepass<double, Shape<4, 8, 8, 16, 0>, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, true>("f64 2^14", 5e-15);
  bad += check_threepass<double, Shape<8, 8, 8, 16, 0>, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, false>("f64 2^15", 5e-15);
  bad += check_threepass<double, Shape<16, 16, 16, 8, 4>, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, true>("f64 2^17", 5e-15);
  bad += check_rows_exchange<float, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>, 1>("f32 2^11", 4, 2e-6);
  bad += check_rows_exchange<float, TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<8, 16, 16, 16, 2>, 4, 4>, 1>("f32 2^14", 8, 2e-6);
  bad += check_rows_exchange<float, TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<8, 16, 16, 16, 2>, 4, 4>, 2>("f32 2^14", 2, 2e-6);
  bad += check_rows_exchange<float, TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<16, 16, 16, 16, 1>, 4, 2>, 0>("f32 2^15", 8, 2e-6);
  bad += check_rows_exchange<float, TwoPass<float, 16, 16, 16, 16, 0, 2, 2>, 1>("f32 2^16", 1, 2e-6);
  bad += check_rows_exchange<double, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>, 1>("f64 2^9", 4, 5e-15);
  bad += check_rows_exchange<double, TwoPass<double, 8, 8, 16, 16, 0, 4, 4>, 2>("f64 2^12", 16, 5e-15);
  // tiles of twice as many transforms (256-byte store runs), as dist_fft.cu's WideShape selects them
  bad += check_rows_exchange<float, TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<8, 16, 16, 16, 2>, 4, 4>, 1, Shape<8, 16, 16, 32, 2>>("f32 2^14 wide", 8, 2e-6);
  bad += check_rows_exchange<float, TwoPass<float, 16, 16, 16, 16, 0, 2, 2>, 2, Shape<16, 16, 16, 32, 1>>("f32 2^16 wide", 4, 2e-6);
  bad += check_rows_exchange<double, TwoPassG<double, Shape<8, 8, 8, 16, 0>, Shape<8, 16, 16, 8, 1>, 4, 2>, 1, Shape<8, 16, 16, 16, 1>>("f64 2^13 wide", 2, 5e-15);
  bad += check_rows_exchange<double, TwoPass<double, 16, 16, 8, 8, 4, 2, 2>, 0, Shape<16, 16, 16, 16, 1>>("f64 2^16 wide", 8, 5e-15);
  bad += check_cta<float>("cta f32", 243, false, 2e-6);
  bad += check_cta<float>("cta f32", 729, false, 2e-6);
  bad += check_cta<float>("cta f32", 2187, false, 3e-6);
  bad += check_cta<float>("cta f32", 96, false, 2e-6);
  bad += check_cta<float>("cta f32", 1536, false, 2e-6);
  bad += check_cta<float>("cta f32", 2048, false, 2e-6);
  bad += check_cta<float>("cta f32", 6, false, 2e-6);
  bad += check_cta<float>("cta f32", 9, false, 2e-6);
  bad += check_cta<double>("cta f64", 768, false, 5e-15);
  bad += check_cta<double>("cta f64", 81, false, 5e-15);
  bad += check_cta<double>("cta f64", 1458, false, 5e-15);
  bad += check_cta<float>("cta f32", 1418, true, 3e-6);
  bad += check_cta<float>("cta f32", 3125, true, 4e-6);
  bad += check_cta<double>("cta f64", 1009, true, 1e-13);
  bad += check_cta<double>("cta f64", 5, true, 1e-13);
  bad += check<float, TwoPass<float, 32, 32, 8, 8, 8, 2, 2>>("f32 2^20 (C=8)", 2e-6);
  bad += check<float, TwoPass<float, 16, 16, 16, 16, 0, 2, 2>>("f32 2^16", 2e-6);
  bad += check<float, TwoPass<float, 16, 32, 16, 8, 0, 2, 2>>("f32 2^18", 2e-6);
  bad += check<float, TwoPassG<float, Shape<4, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>>("f32 2^11", 2e-6);
  bad += check<double, TwoPassG<double, Shape<4, 4, 4, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>>("f64 2^9", 5e-15);
  bad += check<double, TwoPassG<double, Shape<4, 8, 8, 16, 0>, Shape<4, 8, 8, 16, 2>, 4, 4>>("f64 2^10", 5e-15);
  bad += check<double, TwoPassG<double, Shape<4, 8, 8, 16, 0>, Shape<8, 8, 8, 16, 1>, 4, 4>>("f64 2^11", 5e-15);
  bad += check<float, TwoPassG<float, Shape<8, 8, 8, 32, 0>, Shape<8, 8, 8, 32, 2>, 4, 4>>("f32 2^12", 2e-6);
  bad += check<float, TwoPassG<float, Shape<8, 8, 8, 32, 0>, Shape<8, 16, 16, 16, 2>, 4, 4>>("f32 2^13", 2e-6);
  bad += check<float, TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<8, 16, 16, 16, 2>, 4, 4>>("f32 2^14", 2e-6);
  bad += check<float, TwoPassG<float, Shape<8, 16, 16, 16, 0>, Shape<16, 16, 16, 16, 1>, 4, 2>>("f32 2^15", 2e-6);
  bad += check<float, TwoPassG<float, Shape<16, 16, 16, 16, 0>, Shape<16, 32, 32, 8, 1>, 2, 2>>("f32 2^17", 2e-6);
  bad += check<float, TwoPassG<float, Shape<16, 32, 32, 8, 8>, Shape<32, 32, 32, 8, 1>, 2, 2>>("f32 2^19", 2e-6);
  bad += check<double, TwoPassG<double, Shape<8, 8, 8, 16, 0>, Shape<8, 16, 16, 8, 1>, 4, 2>>("f64 2^13", 5e-15);
  bad += check<double, TwoPassG<double, Shape<8, 16, 16, 8, 4>, Shape<16, 16, 16, 8, 1>, 2, 2>>("f64 2^15", 5e-15);
  bad += check<double, TwoPass<double, 16, 16, 8, 8, 4, 2, 2>>("f64 2^16", 5e-15);
  bad += check<double, TwoPass<double, 8, 8, 16, 16, 0, 4, 4>>("f64 2^12", 5e-15);
  bad += check<double, TwoPass<double, 8, 16, 16, 8, 0, 4, 2>>("f64 2^14", 5e-15);
  bad += check_onchip<float, 8, 8, 8, 8>("onchip f32", 2e-6);
  bad += check_onchip<float, 8, 16, 16, 8>("onchip f32", 2e-6);
  bad += check_onchip<float, 16, 16, 16, 8>("onchip f32", 2e-6);
  bad += check_onchip<float, 16, 32, 32, 8>("onchip f32", 2e-6);
  bad += check_onchip<float, 32, 32, 32, 8>("onchip f32", 2e-6);
  bad += check_onchip<double, 8, 8, 8, 8>("onchip f64", 5e-15);
  bad += check_onchip<double, 8, 16, 16, 8>("onchip f64", 5e-15);
  bad += check_onchip<double, 16, 16, 16, 8>("onchip f64", 5e-15);
  bad += check_bluestein<float, 32, 11>("bluestein f32", 1009, 3e-6);
  bad += check_bluestein<float, 32, 11>("bluestein f32", 513, 3e-6);
  bad += check_bluestein<float, 16, 8>("bluestein f32", 255, 3e-6);
  bad += check_bluestein<float, 8, 8>("bluestein f32", 37, 3e-6);
  bad += check_bluestein<double, 16, 8>("bluestein f64", 191, 1e-13);
  bad += check_bluestein<double, 8, 8>("bluestein f64", 61, 1e-13);
  bad += check_fused<fused::FusedCfg<float, 32, 8, 2, 8, 1>>("fused f32 2^20", 2e-6);
  bad += check_fused<fused::FusedCfg<double, 16, 8, 3, 4, 3>>("fused f64 2^16", 5e-15);
  bad += check_fused<fused::FusedCfg<double, 8, 8, 8, 4, 8, true>>("fused f64 2^12", 5e-15);
  // <T, RA, C, G, PAD1, EXB, DIRECT, RB, RA2, RB2, E1, E2, C1>
  bad += check_fused<fused::FusedCfg<float, 32, 8, 2, 0, 1, false, 16, 32, 32, 32, 32, 16, true>>("fused f32 2^19", 2e-6);
  bad += check_fused<fused::FusedCfg<float, 16, 8, 6, 8, 6, false, 8, 16, 16, 16, 32>>("fused f32 2^15", 2e-6);
  bad += check_fused<fused::FusedCfg<float, 8, 8, 8, 8, 8, false, 8, 16, 8, 8, 16>>("fused f32 2^13", 2e-6);
  bad += check_fused<fused::FusedCfg<float, 16, 8, 3, 8, 3, false, 16, 32, 16, 16, 32>>("fused f32 2^17", 2e-6);
  bad += check_fused<fused::FusedCfg<double, 8, 8, 8, 4, 8, true, 8, 16, 8, 8, 16>>("fused f64 2^13", 5e-15);
  bad += check_fused<fused::FusedCfg<float, 32, 8, 3, 8, 3, false, 16>>("fused f32 2^18", 2e-6);
  bad += check_fused<fused::FusedCfg<float, 16, 8, 8, 8, 8, false, 8>>("fused f32 2^14", 2e-6);
  bad += check_fused<fused::FusedCfg<double, 16, 8, 4, 4, 4, false, 8>>("fused f64 2^14", 5e-15);
  bad += check_fused<fused::FusedCfg<float, 16, 8, 4, FB_PAD16, 4>>("fused f32 2^16", 2e-6);
  bad += check_queue();
  printf(bad ? "EMULATION FAILED (%d)\n" : "EMULATION OK\n", bad);
  return bad ? 1 : 0;
}
