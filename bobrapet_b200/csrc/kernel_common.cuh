// kernel_common.cuh — PTX / bit-plane helpers shared by the frontier kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/bobrafrontier.h"
#include "device_record.h"

namespace bf {

#define DI __device__ __forceinline__
constexpr uint32_t FULL = 0xffffffffu;

// ------------------------------------------------------------------ PTX helpers
DI uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
DI void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
DI void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
DI uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
DI void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier.
DI void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// 16 bytes global -> shared through the L2 (src_bytes = 0: the destination is zero-filled and nothing is read);
// complete for the issuing thread after cp_async_wait_all
DI void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
DI void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
// shared-memory fetch-and-add.  An atomic on a warp-uniform address under a lane predicate, atomicAdd or inline PTX alike,
// is compiled to a warp-aggregated atomic (lane id, vote, FLO, two POPC and a shuffle around the one ATOMS); a caller that
// means ONE thread passes an address that depends on the lane (e.g. + lane * 4, zero for the lane that executes it).
DI uint32_t atoms_add_u32(uint32_t a, uint32_t v) {
  uint32_t r;
  asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(r) : "r"(a), "r"(v) : "memory");
  return r;
}
DI void sts_zero16(uint32_t a) { asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a), "r"(0u) : "memory"); }
DI void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

template <int IMM>
DI uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t r;
  asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(c), "n"(IMM));
  return r;
}
// 16-entry boolean table over a bit-sliced 4-bit code: 3 LOP3 for 32 steps.
template <uint32_t T16>
DI uint32_t plut(uint32_t p0, uint32_t p1, uint32_t p2, uint32_t p3) {
  const uint32_t lo = lop3<(T16 & 0xFF)>(p2, p1, p0);
  const uint32_t hi = lop3<((T16 >> 8) & 0xFF)>(p2, p1, p0);
  return lop3<0xCA>(p3, hi, lo);  // p3 ? hi : lo
}
// set the code of the steps in mask m to the constant CODE
template <int CODE>
DI void pset(uint32_t m, uint32_t& p0, uint32_t& p1, uint32_t& p2, uint32_t& p3) {
  p0 = (CODE & 1) ? (p0 | m) : (p0 & ~m);
  p1 = (CODE & 2) ? (p1 | m) : (p1 & ~m);
  p2 = (CODE & 4) ? (p2 | m) : (p2 & ~m);
  p3 = (CODE & 8) ? (p3 | m) : (p3 & ~m);
}
DI uint32_t squeeze4(uint32_t x) {  // bits 0,4,..,28 -> low byte
  x = (x | (x >> 3)) & 0x03030303u;
  x = (x | (x >> 6)) & 0x000F000Fu;
  x = (x | (x >> 12)) & 0xFFu;
  return x;
}
DI uint32_t squeeze2(uint32_t x) {  // bits 0,2,..,30 -> low half
  x = (x | (x >> 1)) & 0x33333333u;
  x = (x | (x >> 2)) & 0x0F0F0F0Fu;
  x = (x | (x >> 4)) & 0x00FF00FFu;
  x = (x | (x >> 8)) & 0xFFFFu;
  return x;
}
DI uint32_t spread4(uint32_t x) {  // inverse of squeeze4
  x = (x | (x << 12)) & 0x000F000Fu;
  x = (x | (x << 6)) & 0x03030303u;
  x = (x | (x << 3)) & 0x11111111u;
  return x;
}
DI uint32_t bits4_to_bytes(uint32_t nib) { return (nib * 0x00204081u) & 0x01010101u; }  // 4 bits -> 4 0/1 bytes
// byte permute with the full PTX selector: bit 3 of a selector nibble replicates the sign of the chosen byte
DI uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
  return r;
}
DI uint32_t get_nibble(const uint8_t* base, uint32_t i) {
  const uint32_t v = (base[i >> 1] >> ((i & 1u) * 4u)) & 0xFu;
  return v == 15u ? 0u : v;
}
DI uint32_t redux_or(uint32_t v) { return __reduce_or_sync(FULL, v); }
DI uint32_t redux_add(uint32_t v) { return __reduce_add_sync(FULL, v); }

DI uint32_t bmsk_clamp(uint32_t pos, uint32_t width) {
  uint32_t r;
  asm("bmsk.clamp.b32 %0, %1, %2;" : "=r"(r) : "r"(pos), "r"(width));
  return r;
}

// ---- shared-space accessors on 32-bit addresses (keeps the walk's address math in 32 bits) ----
DI uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
DI uint32_t lds_u16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
DI uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
// polling load of a word another warp publishes: volatile at the PTX level and a compiler barrier (a plain asm-volatile load
// in an empty loop was dropped by the compiler together with the loop)
DI uint32_t lds_poll_u32(uint32_t a) { uint32_t v; asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
DI uint4 lds_v4(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
DI void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
DI void sts_v4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
DI void red_or_shared(uint32_t a, uint32_t v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
DI void sts_v2(uint32_t a, uint32_t x, uint32_t y) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory"); }
// generic pointer of a shared-window address (rare paths only: parallel join, in-loop failure fix-up)
DI const uint8_t* gptr(uint32_t a) { return static_cast<const uint8_t*>(__cvta_shared_to_generic(a)); }
// keep a loop-invariant value in a register instead of letting the compiler rematerialise it from constants
DI uint32_t pin(uint32_t v) { asm volatile("" : "+r"(v)); return v; }

// ------------------------------------------------------------------ stage D: the dependency walk
// findReadySteps' inner loop (dag.go:2711-2733): one step per lane over the `needs` row of every candidate step,
// visiting only the 32-step words that hold a candidate.  Status byte of a dependency: bit0 = not satisfied,
// bit1 = failed dependency; the byte at index PAD = 32*W (just past the last step word) is always 0.
//
// Row formats (device_record.h), a compile-time parameter of the hot walks:
//   FMT_CSR4   CSR, no row longer than 4: the first four entries are fetched branch-free and clamp-free (col_idx carries
//              four zero entries of padding, so whatever lies past a short row is a valid step index; the verdict is
//              masked with the row length)
//   FMT_CSRL   CSR with longer rows: the same plus a tail loop
//   FMT_ELL2 / FMT_ELL4   fixed-width rows of 2 / 4 entries, unused entries = PAD: no row_ptr, no mask
//   FMT_ELL2B / FMT_ELL4B the same with BYTE entries (S <= 256): a row is ONE 16- / 32-bit load; short rows repeat their
//              first entry, rows without needs are kept out of the walk by the NODEP plane (device_record.h)
//   FMT_ELL4P  four 10-BIT entries (S > 512, the one-run-per-warp kernel only): one 32-bit load + one byte load per row; the
//              `rp_addr` argument of the walks carries the address of the block's high-byte array (there is no row_ptr)
enum : int { FMT_CSR4 = 0, FMT_CSRL = 1, FMT_ELL2 = 2, FMT_ELL4 = 4, FMT_ELL2B = 0x102, FMT_ELL4B = 0x104, FMT_ELL4P = 0x204 };
template <int FMT> struct fmt_traits {
  static constexpr bool byte_rows = (FMT & 0x100) != 0;
  static constexpr bool packed10 = (FMT & 0x200) != 0;
  static constexpr bool fixed = FMT >= 2;
  static constexpr uint32_t row_bytes = packed10 ? 4u : (byte_rows ? (uint32_t)(FMT & 0xFF) : 2u * (uint32_t)(FMT & 0xFF));  // fixed formats (10-bit: the lo words)
};

DI int fmt_of(uint32_t ell, uint32_t max_deg) { return ell ? (int)ell : (max_deg > 4 ? FMT_CSRL : FMT_CSR4); }

// phase 1 of an item: where the row of step `i` starts (shared address) and, for CSR, its length
template <int FMT>
DI void row_locate(bool cand, uint32_t i, uint32_t rp_addr, uint32_t col_addr, uint32_t& p, uint32_t& n) {
  if (fmt_traits<FMT>::packed10) { p = col_addr + i * 4u; n = rp_addr + i; }   // n carries the address of the row's high byte
  else if (fmt_traits<FMT>::fixed) { p = col_addr + i * fmt_traits<FMT>::row_bytes; n = (uint32_t)(FMT & 0xFF); }  // rows exist for every step of the word (padded to 32*W)
  else {
    uint32_t e0 = 0;
    n = 0;
    if (cand) { const uint32_t a = rp_addr + i * 2u; e0 = lds_u16(a); n = lds_u16(a + 2u) - e0; }
    p = col_addr + e0 * 2u;
  }
}
// phase 2: the first entries of the row (may run past a short CSR row: valid indices, masked in phase 3)
template <int FMT>
DI void row_fetch(uint32_t p, uint32_t n, uint32_t (&x)[4]) {
  if (FMT == FMT_ELL4P) {
    const uint32_t lo = lds_u32(p), hi = lds_u8(n);
    x[0] = lo & 0x3FFu; x[1] = (lo >> 10) & 0x3FFu; x[2] = (lo >> 20) & 0x3FFu; x[3] = (lo >> 30) | (hi << 2);
    return;
  }
  if (FMT == FMT_ELL4B) {
    const uint32_t r = lds_u32(p);
    x[0] = r & 0xFFu; x[1] = (r >> 8) & 0xFFu; x[2] = (r >> 16) & 0xFFu; x[3] = r >> 24;
    return;
  }
  if (FMT == FMT_ELL2B) {
    const uint32_t r = lds_u16(p);
    x[0] = r & 0xFFu; x[1] = r >> 8;
    return;
  }
  x[0] = lds_u16(p); x[1] = lds_u16(p + 2u);
  if (FMT != FMT_ELL2) { x[2] = lds_u16(p + 4u); x[3] = lds_u16(p + 6u); }
}
// phase 3: OR of the status bytes of the row's dependencies (CSR: one byte lane per entry, masked by the row length)
template <int FMT>
DI uint32_t row_status(uint32_t p, uint32_t n, const uint32_t (&x)[4], uint32_t st_addr) {
  if (FMT == FMT_ELL2 || FMT == FMT_ELL2B) return lds_u8(st_addr + x[0]) | lds_u8(st_addr + x[1]);
  const uint32_t s0 = lds_u8(st_addr + x[0]), s1 = lds_u8(st_addr + x[1]), s2 = lds_u8(st_addr + x[2]), s3 = lds_u8(st_addr + x[3]);
  if (FMT == FMT_ELL4 || FMT == FMT_ELL4B || FMT == FMT_ELL4P) return s0 | s1 | s2 | s3;
  uint32_t w = (((s3 * 256u + s2) * 256u + s1) * 256u + s0) & bmsk_clamp(0u, n * 8u);
  if (FMT == FMT_CSRL)
    for (uint32_t q = 4; q < n; ++q) w |= lds_u8(st_addr + lds_u16(p + q * 2u));
  return w;
}

// ---- one run per warp (frontier_kernel.cu): K candidate words at once = K independent load chains in flight.
// All K words exist (the driver below only calls it with at least K left).
template <int K, int FMT, bool NEED_FD>
DI void walk_group(uint32_t lane, uint32_t CAND, uint32_t& todo, uint32_t rp_addr, uint32_t col_addr, uint32_t st_addr,
                   uint32_t& met_w, uint32_t& fd_w) {
  uint32_t j[K], p[K], n[K], w[K], cw[K], x[K][4];
  bool c[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    j[k] = __ffs(todo) - 1;
    todo &= todo - 1;
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    cw[k] = __shfl_sync(FULL, CAND, j[k]);
    c[k] = (cw[k] >> lane) & 1u;
    row_locate<FMT>(c[k], j[k] * 32u + lane, rp_addr, col_addr, p[k], n[k]);
  }
#pragma unroll
  for (int k = 0; k < K; ++k) row_fetch<FMT>(p[k], n[k], x[k]);
#pragma unroll
  for (int k = 0; k < K; ++k) w[k] = row_status<FMT>(p[k], n[k], x[k], st_addr);
#pragma unroll
  for (int k = 0; k < K; ++k) {
    if (fmt_traits<FMT>::fixed) {   // every lane holds a real row: the (lane-uniform) candidate word masks the ballot
      const uint32_t m = __ballot_sync(FULL, (w[k] & 0x01010101u) == 0) & cw[k];
      if (lane == j[k]) met_w = m;
      if (NEED_FD) {
        const uint32_t f = __ballot_sync(FULL, (w[k] & 0x02020202u) != 0) & cw[k];
        if (lane == j[k]) fd_w = f;
      }
    } else {
      const uint32_t m = __ballot_sync(FULL, c[k] && (w[k] & 0x01010101u) == 0);
      if (lane == j[k]) met_w = m;
      if (NEED_FD) {
        const uint32_t f = __ballot_sync(FULL, c[k] && (w[k] & 0x02020202u) != 0);
        if (lane == j[k]) fd_w = f;
      }
    }
  }
}

// Stage D driver: the candidate words of a run, KMAX at a time while that many are left, then 2, then 1.
// KMAX = 1 is the plain walk; 2 pays at two CTAs per SM (+2 %), 4 where one CTA per SM leaves little else to hide
// latency (S = 1024: +10 %).  Measured on B200, see DESIGN.md section 5.
template <int KMAX, int FMT, bool NEED_FD>
DI void walk_words(uint32_t lane, uint32_t CAND, uint32_t rp_addr, uint32_t col_addr, uint32_t st_addr, uint32_t& met_w,
                   uint32_t& fd_w) {
  met_w = 0;
  fd_w = 0;
  uint32_t todo = __ballot_sync(FULL, CAND != 0);  // words with at least one candidate step
  if (KMAX >= 4)
    while (__popc(todo) >= 4) walk_group<4, FMT, NEED_FD>(lane, CAND, todo, rp_addr, col_addr, st_addr, met_w, fd_w);
  if (KMAX >= 2) {
    if (KMAX >= 4) {
      if (__popc(todo) >= 2) walk_group<2, FMT, NEED_FD>(lane, CAND, todo, rp_addr, col_addr, st_addr, met_w, fd_w);
    } else {
      while (__popc(todo) >= 2) walk_group<2, FMT, NEED_FD>(lane, CAND, todo, rp_addr, col_addr, st_addr, met_w, fd_w);
    }
  }
  if (KMAX >= 2) {
    if (todo) walk_group<1, FMT, NEED_FD>(lane, CAND, todo, rp_addr, col_addr, st_addr, met_w, fd_w);
  } else {
    while (todo) walk_group<1, FMT, NEED_FD>(lane, CAND, todo, rp_addr, col_addr, st_addr, met_w, fd_w);
  }
}

template <int KMAX, bool NEED_FD>
DI void walk_words_fmt(int fmt, uint32_t lane, uint32_t CAND, uint32_t rp_addr, uint32_t col_addr, uint32_t st_addr,
                       uint32_t& met_w, uint32_t& fd_w) {  // fmt is warp-uniform
  if (fmt == FMT_ELL4P) walk_words<KMAX, FMT_ELL4P, NEED_FD>(lane, CAND, rp_addr, col_addr, st_addr, met_w, fd_w);
  else if (fmt == FMT_ELL4B) walk_words<KMAX, FMT_ELL4B, NEED_FD>(lane, CAND, rp_addr, col_addr, st_addr, met_w, fd_w);
  else if (fmt == FMT_ELL4) walk_words<KMAX, FMT_ELL4, NEED_FD>(lane, CAND, rp_addr, col_addr, st_addr, met_w, fd_w);
  else if (fmt == FMT_ELL2B) walk_words<KMAX, FMT_ELL2B, NEED_FD>(lane, CAND, rp_addr, col_addr, st_addr, met_w, fd_w);
  else if (fmt == FMT_CSR4) walk_words<KMAX, FMT_CSR4, NEED_FD>(lane, CAND, rp_addr, col_addr, st_addr, met_w, fd_w);
  else if (fmt == FMT_ELL2) walk_words<KMAX, FMT_ELL2, NEED_FD>(lane, CAND, rp_addr, col_addr, st_addr, met_w, fd_w);
  else walk_words<KMAX, FMT_CSRL, NEED_FD>(lane, CAND, rp_addr, col_addr, st_addr, met_w, fd_w);
}

// ---- the fix-up walk (rare): a step set Failed earlier in this same loop (dag.go:2744/2810 mutate stepStates while
// `completed` stays as built at :497) is visible to LATER steps of the list only.  Plain loop over every entry of the
// row, any format.  The item (word j of the run whose CAND word is held by lane `owner`) is given by the caller.
DI void fixup_item(uint32_t lane, uint32_t candw, uint32_t j, uint32_t ell, uint32_t rp_addr, uint32_t col_addr, uint32_t st_addr,
                   uint32_t mfail_addr, uint32_t failed_class, uint32_t& metb, uint32_t& fdb) {
  const bool cand = (candw >> lane) & 1u;
  const uint32_t i = j * 32u + lane;
  uint32_t acc = 0;
  if (cand) {
    uint32_t p, n;
    const uint32_t eb = (ell & ELL_BYTE) ? 1u : 2u;   // bytes per entry (the caller keeps NODEP steps out of candw)
    uint32_t lo10 = 0, hi10 = 0;
    if (ell & ELL_PACK10) { n = 4u; p = 0; lo10 = lds_u32(col_addr + i * 4u); hi10 = lds_u8(rp_addr + i); }  // rp_addr: the high-byte array
    else if (ell) { n = ell_k(ell); p = col_addr + i * n * eb; }
    else { const uint32_t a = rp_addr + i * 2u; const uint32_t e0 = lds_u16(a); n = lds_u16(a + 2u) - e0; p = col_addr + e0 * 2u; }
    for (uint32_t e = 0; e < n; ++e) {
      const uint32_t d = (ell & ELL_PACK10) ? (e < 3u ? (lo10 >> (10u * e)) & 0x3FFu : (lo10 >> 30) | (hi10 << 2))
                                            : (eb == 1u ? lds_u8(p + e) : lds_u16(p + e * 2u));
      uint32_t sb = lds_u8(st_addr + d);
      if (d < i && ((lds_u32(mfail_addr + (d >> 5) * 4u) >> (d & 31u)) & 1u)) sb = failed_class;  // PAD >= i: never
      acc |= sb;
    }
  }
  fdb = __ballot_sync(FULL, cand && (acc & 2u) != 0);
  metb = __ballot_sync(FULL, cand && (acc & 1u) == 0);
}

}  // namespace bf
