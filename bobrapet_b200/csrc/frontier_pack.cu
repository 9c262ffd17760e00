// frontier_pack.cu — packed-lanes frontier pass: one warp evaluates a GROUP of R = 32 / Wq StoryRuns per trip
// (Wq = words per run rounded up to a power of two; R = 4 at S = 256, 16 at S = 64).  It is the default kernel of
// single-pass batches whose runs have at most 512 steps; frontier_kernel.cu (one run per warp) covers S > 512,
// the device fixpoint and, as a second tier, the runs whose topology has `parallel` steps.
//
// Why: at S = 256 the one-run-per-warp kernel spends ~290 of its 440 warp instructions per run on per-word work that
// keeps 8 of 32 lanes busy and is bound by instruction issue (72 % of the issue slots at 75 % of the HBM roofline).
// Here lane l = g * Wq + w holds word w (32 steps) of run g of the group, so every bit-plane stage (gate / sleep /
// wait rewrite dag.go:1455-1547, buildStateMaps :3358-3391, fail-fast / compensation marking and group selection
// :422-511, cond masking :2741-2843, result words) runs on all 32 lanes and its instructions are shared by R runs;
// per-run reductions are sub-warp redux / ballots.  Only the dependency walk (dag.go:2711-2733, one step per lane
// over a `needs` row) stays per (run, word).
//
// Data movement: the CTA (one per SM, persistent) owns a ring of NG slot groups in shared memory, each holding the R
// state records (adjacent in HBM: ONE bulk copy) and R topology records (one bulk copy each) of a group, guarded by
// one mbarrier per slot group.  The ring is shared by all warps of the CTA: groups are consumed in ticket order (a free
// warp draws the CTA's next group from a shared counter), and the warp that finishes group t re-arms the slot group it
// just read with the copies of group t + NG, which whichever warp draws that ticket will consume — so the number of
// groups in flight adapts by itself (a warp waiting at a barrier IS a group in flight), and a CTA keeps 24 warps fed
// from 33 slot groups where a private double-buffered ring per warp would allow only 16 warps.  The chain run ->
// slot id -> slot entry of group t + NG is fetched by the R lanes that own its runs while the warp works on group t
// (first link before the barrier wait, second after stage C, landing in shared memory so that it holds no registers through
// the walk), and those lanes issue the copies.
// A dead / oversized slot is marked by a zero header written before the arrive, a run deferred to the general kernel by
// an all-ones header word.
//
// Start-up and tail: a cold CTA needs three dependent DRAM round trips (slot id, slot entry, bulk copy: ~3.6 - 6.6 us
// measured with tools/trace_probe.py) before its first group can be evaluated, and the CTAs of a grid finish 4 - 5 us
// apart.  BF_EVAL_PIPELINED (a caller's promise that consecutive passes are independent) launches the pass as a
// programmatic dependent of the preceding kernel: its CTAs take the SMs that kernel has already left, so start-up,
// launch gap and tail overlap (cfg3: 45.8 -> 40.1 us per pass); griddepcontrol.wait sits in front of the counters.
//
// All shared-memory traffic goes through 32-bit shared-window addresses.  Integer only; no tensor cores.
#include "kernel_common.cuh"

namespace bf {

extern __shared__ __align__(128) uint8_t smem_p[];

#ifndef WALK_K
#define WALK_K 4   // (run, word) items walked at once: independent load chains per warp (measured: 2: 50.9 us, 3: 50.0, 4: 49.5)
#endif
#ifndef PACK_MAX_WARPS
#define PACK_MAX_WARPS 24   // warps per CTA the kernel is compiled for (registers: 65536 / (32 * PACK_MAX_WARPS) per thread = 80).
#endif                      // Measured at cfg3 with byte-entry rows (ring of 33 slot groups): 16: 48.2 us, 20: 47.1, 24: 45.6, 28: 47.9, 32: 49.4

#ifdef PACK_TRACE   // timeline probe (tools/trace_probe.py, lib_ab builds only): per launch and CTA {start, first group landed, last group done, end}
__device__ unsigned long long g_trace[8][160][4];
__device__ unsigned int g_launch;
DI unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#endif

// ---- stage D over the (run, word) items of a group.
// Where the rows and status bytes of run g live: CSR formats read the per-run table {col_a, rp_a, st_a, max_deg | ell << 16}
// written in stage C; fixed-width rows always start 32 bytes into the run's topology buffer, so their addresses are
// computed (two multiply-adds, no dependent shared-memory load in front of the row fetch).
struct WalkCtx {
  uint32_t tab_a;      // per-run table (16 B entries)
  uint32_t col0;       // fixed-width formats: col_idx of run 0 of the group (topology buffer 0 + 32)
  uint32_t topo_buf;   // bytes between the topology buffers of consecutive runs
  uint32_t st0;        // status bytes of run 0
  uint32_t st_stride;  // bytes between the status areas of consecutive runs
};

// K items at once (independent load chains); FMT as in kernel_common.cuh — the caller guarantees that every live run
// of the group has this row format (else it takes walk_items_any).  Items are taken from the highest lane down (one FLO
// per item); every item delivers to its own lane, so the order does not matter.
// Fixed-width rows exist for every step of a word, so all 32 lanes fetch and ballot; the ballots are not masked here — the
// owner lane masks its two words with its own candidate word once, after the walk (walk_items).  For every byte a fixed-width
// row can name (a step < S, col_idx is validated at upload, or PAD) the status byte is 0, 1 or 3 (FD is a subset of U below S,
// and PAD is 0), so the OR of a row's bytes is 0 when every need is met and above 1 when one has failed.
// AL (byte-entry rows of four, 8 words per run): the owner lane of an item publishes `own` = (its row base << 14) | (its run's
// status base >> 8) (walk_items); one shuffle gives every lane both.  The status bytes of a run start on a 256-byte boundary,
// so the address of a dependency's status byte is ONE byte permute: byte k of the row word, then bytes 0 and 1 of `own`
// (status base bits 8 .. 17; bits 14 and 15 of `own` are row-base bits 0 and 1, zero for a 4-byte aligned row), then the
// sign of byte 1 (bit 15 = 0) as the zero top byte.
template <int K, int FMT, bool NEED_FD, bool AL = false>
DI void walk_items_k(uint32_t lane, uint32_t CAND, uint32_t own, uint32_t& todo, uint32_t lg, const WalkCtx& C, uint32_t& met_w,
                     uint32_t& fd_w) {
  const uint32_t wmask = (1u << lg) - 1u;
  uint32_t L[K], p[K], n[K], wv[K], st[K], x[K][4];
  bool c[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    L[k] = 31u - __clz(todo);
    todo &= bmsk_clamp(0u, L[k]);   // clears bit L and above
  }
  if (AL && FMT == FMT_ELL4B) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      st[k] = __shfl_sync(FULL, own, L[k]);
      n[k] = lds_u32((st[k] >> 14) + lane * 4u);   // the row of step (L & 7) * 32 + lane: four byte entries
    }
#pragma unroll
    for (int k = 0; k < K; ++k)
      wv[k] = lds_u8(prmt(n[k], st[k], 0xD540u)) | lds_u8(prmt(n[k], st[k], 0xD541u)) | lds_u8(prmt(n[k], st[k], 0xD542u)) |
              lds_u8(prmt(n[k], st[k], 0xD543u));
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const uint32_t m = __ballot_sync(FULL, wv[k] == 0);
      const uint32_t f = NEED_FD ? __ballot_sync(FULL, wv[k] > 1u) : 0u;
      if (lane == L[k]) {
        met_w = m;
        if (NEED_FD) fd_w = f;
      }
    }
    return;
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const uint32_t g = L[k] >> lg, i = (L[k] & wmask) * 32u + lane;
    if (fmt_traits<FMT>::fixed) {
      st[k] = C.st0 + g * C.st_stride;
      p[k] = C.col0 + g * C.topo_buf + i * fmt_traits<FMT>::row_bytes;   // rows exist for every step of the word (device_record.h)
      n[k] = (uint32_t)(FMT & 0xFF);
    } else {
      c[k] = (__shfl_sync(FULL, CAND, L[k]) >> lane) & 1u;
      const uint4 t = lds_v4(C.tab_a + g * 16u);
      st[k] = t.z;
      row_locate<FMT>(c[k], i, t.y, t.x, p[k], n[k]);
    }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) row_fetch<FMT>(p[k], n[k], x[k]);
#pragma unroll
  for (int k = 0; k < K; ++k) wv[k] = row_status<FMT>(p[k], n[k], x[k], st[k]);
#pragma unroll
  for (int k = 0; k < K; ++k) {
    if (fmt_traits<FMT>::fixed) {   // wv = OR of the row's status bytes (0, 1 or 3)
      const uint32_t m = __ballot_sync(FULL, wv[k] == 0);
      const uint32_t f = NEED_FD ? __ballot_sync(FULL, wv[k] > 1u) : 0u;
      if (lane == L[k]) {
        met_w = m;
        if (NEED_FD) fd_w = f;
      }
    } else {
      const uint32_t m = __ballot_sync(FULL, c[k] && (wv[k] & 0x01010101u) == 0);
      if (lane == L[k]) met_w = m;
      if (NEED_FD) {
        const uint32_t f = __ballot_sync(FULL, c[k] && (wv[k] & 0x02020202u) != 0);
        if (lane == L[k]) fd_w = f;
      }
    }
  }
}

template <int FMT, bool NEED_FD, bool AL = false>
DI void walk_items(uint32_t lane, uint32_t CAND, uint32_t lg, const WalkCtx& C, uint32_t& met_w, uint32_t& fd_w) {
  met_w = 0;
  fd_w = 0;
  uint32_t own = 0;
  if (AL) {   // Wq = 8: lane = g * 8 + w; shared-window addresses are below 2^18 (at most 227 KB of shared memory per block)
    const uint32_t g = lane >> 3, w = lane & 7u;
    own = ((C.col0 + g * C.topo_buf + w * 128u) << 14) | ((C.st0 + g * 256u) >> 8);
  }
  uint32_t todo = __ballot_sync(FULL, CAND != 0);  // (run, word) pairs with at least one candidate step
  while (__popc(todo) >= WALK_K) walk_items_k<WALK_K, FMT, NEED_FD, AL>(lane, CAND, own, todo, lg, C, met_w, fd_w);
  if (WALK_K > 2)
    if (__popc(todo) >= 2) walk_items_k<2, FMT, NEED_FD, AL>(lane, CAND, own, todo, lg, C, met_w, fd_w);
  if (todo) walk_items_k<1, FMT, NEED_FD, AL>(lane, CAND, own, todo, lg, C, met_w, fd_w);
  met_w &= CAND;   // the fixed-width ballots cover all 32 steps of a word
  fd_w &= CAND;
}

// mixed row formats inside one group (rare): one item at a time, format read from the item's table entry
template <bool NEED_FD>
DI void walk_items_any(uint32_t lane, uint32_t CAND, uint32_t lg, const WalkCtx& C, uint32_t& met_w, uint32_t& fd_w) {
  met_w = 0;
  fd_w = 0;
  for (uint32_t todo = __ballot_sync(FULL, CAND != 0); todo;) {
    const uint32_t L = __ffs(todo) - 1;
    const uint32_t meta = lds_u32(C.tab_a + (L >> lg) * 16u + 12u);
    const int fmt = fmt_of(meta >> 16, meta & 0xFFFFu);  // warp-uniform
    uint32_t one = todo & (0u - todo);
    todo ^= one;
    if (fmt == FMT_ELL4B) walk_items_k<1, FMT_ELL4B, NEED_FD>(lane, CAND, 0u, one, lg, C, met_w, fd_w);
    else if (fmt == FMT_ELL2B) walk_items_k<1, FMT_ELL2B, NEED_FD>(lane, CAND, 0u, one, lg, C, met_w, fd_w);
    else if (fmt == FMT_ELL4) walk_items_k<1, FMT_ELL4, NEED_FD>(lane, CAND, 0u, one, lg, C, met_w, fd_w);
    else if (fmt == FMT_CSR4) walk_items_k<1, FMT_CSR4, NEED_FD>(lane, CAND, 0u, one, lg, C, met_w, fd_w);
    else if (fmt == FMT_ELL2) walk_items_k<1, FMT_ELL2, NEED_FD>(lane, CAND, 0u, one, lg, C, met_w, fd_w);
    else walk_items_k<1, FMT_CSRL, NEED_FD>(lane, CAND, 0u, one, lg, C, met_w, fd_w);
  }
  met_w &= CAND;
  fd_w &= CAND;
}

// CD: cond and/or decision codes present   XO: any of fail/needs_cond/skip_dep/phase_out requested
template <bool CD, bool XO>
#ifndef PACK_MIN_BLOCKS
#define PACK_MIN_BLOCKS 1   // resident CTAs per SM the build is compiled for (BF_PACK_CTAS experiments)
#endif
__global__ void __launch_bounds__(32 * PACK_MAX_WARPS, PACK_MIN_BLOCKS) frontier_pack_kernel(const KParams P) {
  // BF_EVAL_PIPELINED: let the next kernel of the stream (launched as a programmatic dependent) take the SMs this grid leaves
  // as its CTAs run out of groups; a no-op otherwise
  if (P.flags & BF_EVAL_PIPELINED) asm volatile("griddepcontrol.launch_dependents;");
  const uint32_t lane = pin(threadIdx.x & 31u);  // pinned: otherwise rematerialised from S2R inside the loop
  const uint32_t warp = __shfl_sync(FULL, threadIdx.x >> 5, 0);  // through a shuffle: the compiler then treats it as warp-uniform
  const uint32_t NW = P.warps_per_block, NG = P.slot_groups;
  const uint32_t Wq = P.wq, lg = P.wq_log2, R = 32u >> lg;
  const uint32_t g = pin(lane >> lg), w = pin(lane & (Wq - 1u));
  const uint32_t gmask = (Wq == 32u ? FULL : ((1u << Wq) - 1u)) << (g << lg);

#ifdef PACK_TRACE
  const unsigned long long tr_start = gtime();
  const unsigned int tr_launch = *((volatile unsigned int*)&g_launch) & 7u;
  unsigned long long tr_first = 0, tr_last = 0;
#endif
  // ---- shared memory carve-up: [block counters 128 B][mbarriers, one per slot group][NG slot groups][warp scratch]
  // slot group: R state records (contiguous, as in HBM) then R topology buffers of topo_buf_bytes each.
  // The mbarriers sit in one block AWAY from the TMA destinations (a barrier next to a record tail cost 9 %).
  unsigned long long* blk_counts = reinterpret_cast<unsigned long long*>(smem_p);
  const uint32_t smem_base = smem_u32(smem_p);
  const uint32_t bars = pin(smem_base + 128u);
  const uint32_t armed_a = bars + NG * 8u;                        // u32 per slot group: uses armed so far (see the wait below)
  const uint32_t bars_bytes = (NG * 12u + 127u) & ~127u;
  const uint32_t group_bytes = R * (P.state_stride + P.topo_buf_bytes);
  const uint32_t groups_a = pin(smem_base + 128u + bars_bytes);
  // scratch (per warp, 256-byte aligned, work_bytes a multiple of 256): [status bytes: R x st_stride][fix-up fail words 128 B]
  // [walk table: R x 16 B].  st_stride = 32*Wq + 16 (the PAD byte of a full-width run with u16 rows lives in the + 16) except at
  // Wq = 8, where it is 256 so that every run's status bytes start on a 256-byte boundary (walk_items_k, AL; no topology of
  // 8 words has u16 fixed-width rows: plan_record, abi.cu)
  const uint32_t st_stride = Wq == 8u ? 256u : 32u * Wq + 16u;
  const uint32_t scratch_a = ((groups_a + NG * group_bytes + 255u) & ~255u) + warp * P.work_bytes;
  const uint32_t st0_a = scratch_a;
  const uint32_t mfail_a = st0_a + R * st_stride;
  const uint32_t tab_a = mfail_a + 128u;

  if (threadIdx.x < 5) blk_counts[threadIdx.x] = 0ull;   // four counters + the group ticket
  if (threadIdx.x < NG) {
    mbar_init(bars + 8u * threadIdx.x, R);
    sts_u32(armed_a + 4u * threadIdx.x, 0u);
    fence_barrier_init();
  }
  for (uint32_t x = lane * 4u; x < P.work_bytes; x += 128u) sts_u32(scratch_a + x, 0u);  // PAD bytes start as 0 and stay 0
  __syncthreads();

  // ---- the CTA's groups: global group id = blockIdx.x + t * gridDim.x, runs R * gid .. R * gid + R - 1
  const uint32_t N = P.n_runs;
  const uint32_t n_groups = (N + R - 1) >> (5 - lg);
  const uint32_t T = blockIdx.x < n_groups ? (n_groups - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  // Schedule: groups are CONSUMED in ticket order — a warp that is free takes the next group of the CTA from a shared
  // counter (a static t -> warp map left the warps with one group more than the others running alone at the end: 8 against
  // 7.04 groups per warp at the headline size).  Group t lives in slot group t % NG, use number t / NG; groups t < NG are
  // issued in the prologue (by warp t % NW), group t >= NG by the warp that consumed t - NG and thereby freed the slot.
  const uint32_t n_pro = warp < NG ? (NG - warp + NW - 1) / NW : 0;   // my prologue issues: t = warp + q * NW < NG

  // ---- producer side: the chain run -> slot id -> slot entry of a group is fetched by the R lanes that own its runs.
  // Prologue: lane l holds (issue q0 + l / R, run l % R) of a batch of GB = 32 / R issues; steady state: the lanes of
  // issue 0 (lq == 0) hold the group my warp will issue when it is done with the current one.
  const uint32_t GB = 32u >> (5 - lg);        // = Wq: issues per prologue batch
  const uint32_t lq = lane >> (5 - lg), lr = lane & (R - 1u);   // my pair inside a batch: issue lq, run lr
  uint32_t pf_sid = 0xFFFFFFFFu;
  auto load_sid = [&](uint32_t t, bool mine) {   // first link: my run's topology slot id (the head word of its state record)
    pf_sid = 0xFFFFFFFFu;
    if (mine && t < T) {
      const uint32_t r = ((blockIdx.x + t * gridDim.x) << (5 - lg)) + lr;
      if (r < N) pf_sid = __ldg(reinterpret_cast<const uint32_t*>(P.state + (size_t)r * P.state_stride));
    }
  };
  // issue the copies of group t into slot group `sg`, which thereby starts its use number `use`; `mine`: my lane owns a run of
  // it; `ent`: my run's slot entry (address, bytes, meta), all zero for a slot id out of range
  auto issue = [&](uint32_t t, uint32_t sg, uint32_t use, bool mine, const uint4 ent) {
    if (t < T && mine) {
      const uint32_t buf = groups_a + sg * group_bytes;
      const uint32_t bar = bars + 8u * sg;
      const uint32_t tb = buf + R * P.state_stride + lr * P.topo_buf_bytes;   // my run's topology buffer
      const uint32_t first = (blockIdx.x + t * gridDim.x) << (5 - lg);
      const bool valid = first + lr < N;
      const bool dfr = valid && P.defer_list != nullptr && (ent.w >> 16) != 0;  // topology with parallel steps
      const bool ok = valid && !dfr && (ent.x | ent.y) != 0 && ent.z <= P.topo_buf_bytes;
      if (!ok) sts_v4(tb, dfr ? 0xFFFFFFFFu : 0u, 0u, 0u, 0u);   // marker header (W = 0: dead, all-ones: deferred)
      uint32_t sbytes = 0;
      if (lr == 0) {
        sbytes = min(R, N - first) * P.state_stride;   // the group's state records are adjacent: one copy
        sts_u32(armed_a + 4u * sg, use + 1u);          // published before my arrive: the previous use is over, this one is armed
      }
      mbar_expect_tx(bar, (ok ? ent.z : 0u) + sbytes);
      if (lr == 0) bulk_g2s(buf, P.state + (size_t)first * P.state_stride, sbytes, bar);
      if (ok) bulk_g2s(tb, reinterpret_cast<const void*>((uint64_t)ent.x | ((uint64_t)ent.y << 32)), ent.z, bar);
    }
  };
  for (uint32_t q0 = 0; q0 < n_pro; q0 += GB) {      // prologue: GB of my issues at a time (both links of all of them in flight together)
    const bool in_pro = q0 + lq < n_pro;
    load_sid(warp + (q0 + lq) * NW, in_pro);
    const uint4 ent = pf_sid < P.n_slots ? __ldg(reinterpret_cast<const uint4*>(P.slots + pf_sid)) : make_uint4(0u, 0u, 0u, 0u);
    for (uint32_t k = 0; k < GB && q0 + k < n_pro; ++k) {
      const uint32_t t = warp + (q0 + k) * NW;       // < NG: its slot group is t itself, use 0
      issue(t, t, 0u, lq == k, ent);
    }
  }

  const uint32_t Wmax = P.words;
  const bool has_cond = CD && P.off_cond != BF_OFF_NONE;
  const bool has_dec = CD && P.off_decision != BF_OFF_NONE;
  uint32_t lane_ready = 0, lane_skip = 0, lane_evals = 0;  // per-lane running totals, reduced once at the end

  // the next group to consume: a CTA-wide ticket counter behind the four block counters (smem_p + 32)
  const uint32_t ng_magic = NG > 1u ? (uint32_t)(0x100000000ull / NG) + 1u : 0u;   // t / NG = umulhi(t, ng_magic), exact for t < 2^32 / NG (NG = 1: T <= 1, t = 0)
  for (;;) {
    uint32_t t = 0;
    const uint32_t lane4 = pin(lane * 4u);   // outside the branch (inside it lane is known to be 0): a single-lane atomic
    if (lane == 0) t = atoms_add_u32(smem_base + 32u + lane4, 1u);
    t = __shfl_sync(FULL, t, 0);
    if (t >= T) break;
    const uint32_t cur_use = __umulhi(t, ng_magic), cur_sg = t - cur_use * NG;   // t / NG, t % NG
    load_sid(t + NG, lq == 0);   // first link of the group I shall issue into this slot group when I am done with it
    // The slot group is shared between warps: its use `cur_use` is armed by the warp that consumed the previous use.
    // A parity wait alone cannot tell "use u - 1 still pending" from "use u complete" (the parity then names the phase
    // before), so first wait until the arming warp has published use u; from then on the barrier is in phase u.
    while ((int32_t)(lds_poll_u32(armed_a + 4u * cur_sg) - (cur_use + 1u)) < 0) __nanosleep(32);
    mbar_wait(bars + 8u * cur_sg, cur_use & 1u);
#ifdef PACK_TRACE
    if (t == 0) tr_first = gtime();
#endif

    const uint32_t gid = blockIdx.x + t * gridDim.x;
    const uint32_t r = (gid << (5 - lg)) + g;                 // my run
    uint8_t* const rr = P.result + (size_t)r * P.result_stride;
    const uint32_t grp_a = groups_a + cur_sg * group_bytes;
    const uint32_t sr_a = grp_a + g * P.state_stride;                                   // my run's state record
    const uint32_t tr_a = grp_a + R * P.state_stride + g * P.topo_buf_bytes;            // my run's topology record

    const bool in_batch = r < N;
    const uint4 h0 = lds_v4(tr_a);
    const uint4 h1 = lds_v4(tr_a + 16);
    const bool deferred = in_batch && h0.x == 0xFFFFFFFFu;
    uint32_t S = h0.x & 0xFFFFu, Wt = h0.x >> 16;
    const uint32_t max_deg = h0.y & 0xFFFFu;
    uint32_t n_main = h0.z & 0xFFFFu, n_comp = h0.z >> 16, n_final = h0.w & 0xFFFFu;
    const bool live = in_batch && Wt - 1u < Wmax;  // group-uniform (a marker header has W = 0 or 0xFFFF)
    if (!live) { S = 0; Wt = 0; n_main = n_comp = n_final = 0; }
    const uint32_t ell = live ? (h1.x >> 16) : 0u;
    const uint32_t rflags = live ? lds_u8(sr_a + 4) : (uint32_t)BF_RF_HOST_GROUP | (BF_GROUP_DONE << BF_RF_HOST_GROUP_SHIFT);

    // ---------------- planes of my word ----------------
    const bool act = w < Wt;
    uint32_t AF = 0, TS = 0, HASIF = 0, G1 = 0, G2 = 0, VALID = 0, SYNC_T = 0, NODEP = 0;
    uint32_t c0 = 0, c1 = 0, d0 = 0, d1 = 0;
    uint32_t p0 = 0, p1 = 0, p2 = 0, p3 = 0;
    if (act) {
      const uint32_t sp = tr_a + h1.y + w * 4u, ps = Wt * 4u;   // static planes: my word, plane stride
      AF = lds_u32(sp + PL_AF * ps);
      G1 = lds_u32(sp + PL_G1 * ps); G2 = lds_u32(sp + PL_G2 * ps);
      if (XO) HASIF = lds_u32(sp + PL_HASIF * ps);
      if (ell_has_nodep(ell)) NODEP = lds_u32(sp + PL_NODEP * ps);   // byte-entry rows: steps without needs stay out of the walk
      VALID = bmsk_clamp(0u, S - w * 32u);
      const uint32_t pw = sr_a + P.off_phase + w * 4u, ds = Wmax * 4u;  // dynamic planes: stride of the layout
      p0 = lds_u32(pw); p1 = lds_u32(pw + ds); p2 = lds_u32(pw + 2u * ds); p3 = lds_u32(pw + 3u * ds);
      const uint32_t keep = VALID & ~(p0 & p1 & p2 & p3);  // steps >= S and the reserved code 15 read as 0
      p0 &= keep; p1 &= keep; p2 &= keep; p3 &= keep;
      if (CD) {
        if (has_cond) { const uint32_t cw = sr_a + P.off_cond + w * 4u; c0 = lds_u32(cw); c1 = lds_u32(cw + ds); }
        if (has_dec) {
          const uint32_t dw = sr_a + P.off_decision + w * 4u; d0 = lds_u32(dw); d1 = lds_u32(dw + ds);
          const uint32_t t0 = lds_u32(sp + PL_T0 * ps), t1 = lds_u32(sp + PL_T1 * ps), t2 = lds_u32(sp + PL_T2 * ps);
          TS = lds_u32(sp + PL_TS * ps);
          SYNC_T = t0 & (t1 | t2);  // sleep(3) | wait(5) | gate(7)
        }
      }
    }
    const uint32_t q0 = p0, q1 = p1, q2 = p2, q3 = p3;
    const uint32_t GM = VALID & ~G1 & ~G2;
    const bool fail_fast = rflags & BF_RF_FAIL_FAST;
    const bool realtime = rflags & BF_RF_REALTIME;
    const bool topo_term = rflags & BF_RF_TOPOLOGY_TERMINATED;
    const bool host_group = rflags & BF_RF_HOST_GROUP;
    bool marked = false;  // group-uniform

    // ---------------- stage G: gate / sleep / wait sync (dag.go:1469-1533, 1235-1277, 1327-1437) ----------------
    if (CD) {
      if (has_dec) {
        const uint32_t syn = SYNC_T & plut<BF_LUT_RUNNING>(p0, p1, p2, p3);
        const uint32_t n0 = d0;
        const uint32_t n1 = d0 & ~(d1 & TS);
        const uint32_t n2 = d1 & (~d0 | TS);
        const uint32_t n3 = ~(d0 ^ d1);
        p0 = (p0 & ~syn) | (n0 & syn);
        p1 = (p1 & ~syn) | (n1 & syn);
        p2 = (p2 & ~syn) | (n2 & syn);
        p3 = (p3 & ~syn) | (n3 & syn);
      }
    }

    // ---------------- stage B: classification (dag.go:3377-3388, 2020-2033) ----------------
    uint32_t TERM = plut<BF_LUT_TERMINAL>(p0, p1, p2, p3);
    uint32_t COMPL = plut<BF_LUT_COMPLETED0>(p0, p1, p2, p3) | (TERM & AF);
    uint32_t RUNQ = plut<BF_LUT_RUNNING_Q>(p0, p1, p2, p3);
    uint32_t FAILED = TERM & ~COMPL;
    uint32_t group, sum = 0;
    // ---------------- stage I (dag.go:422-495): per-run reductions = one sub-warp redux.or ----------------
    // A group none of whose runs has a compensation or finally step, nor takes the realtime + topology-terminated branch
    // (host-group runs never do), needs only the main-group facts: every fact about G1 / G2 is empty, so the general code
    // below would mark nothing there and find compensation and finally done and not failed.
    const bool main_only = __all_sync(FULL, (G1 | G2) == 0u && !(realtime && topo_term && !host_group));
    const uint32_t DONE = COMPL | FAILED;
    const uint32_t mark_ff = GM & ~COMPL & ~RUNQ & ~TERM;             // markFailFastSkipped candidates (:3289-3312)
    if (main_only) {
      const uint32_t bits = __reduce_or_sync(gmask, ((FAILED & GM) != 0 ? 1u : 0u) | ((GM & ~DONE) != 0 ? 2u : 0u) |
                                                        ((GM & ~DONE & ~mark_ff) != 0 ? 4u : 0u) | (mark_ff != 0 ? 8u : 0u));
      const bool amf = bits & 1u;
      const bool do_ff = !host_group && fail_fast && amf;
      if (do_ff) {
        marked = bits & 8u;
        pset<BF_PHASE_SKIPPED>(mark_ff, p0, p1, p2, p3);
        TERM |= mark_ff; COMPL |= mark_ff;
      }
      const bool main_done = n_main == 0 || !(bits & (do_ff ? 4u : 2u));
      group = main_done ? BF_GROUP_DONE : BF_GROUP_MAIN;
      sum = (main_done ? BF_SUM_MAIN_DONE : 0u) | (amf ? BF_SUM_MAIN_FAILED : 0u) | BF_SUM_COMP_DONE | BF_SUM_FINAL_DONE;
    } else {
      uint32_t RUN = plut<BF_LUT_RUNNING>(p0, p1, p2, p3);
      const uint32_t mark_cs = G1 & ~COMPL & ~RUN & ~FAILED & ~TERM;   // markCompensationsSkipped candidates (:3314-3342)
      uint32_t bits = ((FAILED & GM) != 0 ? 1u : 0u) | ((GM & ~DONE) != 0 ? 2u : 0u) | ((GM & ~DONE & ~mark_ff) != 0 ? 4u : 0u) |
                      ((G1 & ~DONE) != 0 ? 8u : 0u) | ((G1 & ~DONE & ~mark_cs) != 0 ? 16u : 0u) | ((G2 & ~DONE) != 0 ? 32u : 0u) |
                      ((FAILED & G1) != 0 ? 64u : 0u) | ((FAILED & G2) != 0 ? 128u : 0u) | (mark_ff != 0 ? 256u : 0u) |
                      (mark_cs != 0 ? 512u : 0u);
      bits = __reduce_or_sync(gmask, bits);
      // no collective may sit under a per-run branch: host-group runs (tier K1) take part in every
      // vote below and simply never qualify for a marking
      const bool auto_group = !host_group;
      bool amf = bits & 1u;
      const bool do_ff = auto_group && fail_fast && amf;
      if (do_ff) {
        marked = marked || (bits & 256u);
        pset<BF_PHASE_SKIPPED>(mark_ff, p0, p1, p2, p3);
        TERM |= mark_ff; COMPL |= mark_ff; RUN &= ~mark_ff;
      }
      bool main_done = n_main == 0 || !(bits & (do_ff ? 4u : 2u));
      const bool acf = bits & 64u;
      // dag.go:436-464 (rare)
      const bool tt = auto_group && !main_done && realtime && topo_term;
      if (__any_sync(FULL, tt)) {
        const uint32_t mtt = tt ? (GM & (p0 | p1 | p2 | p3) & ~TERM) : 0u;
        pset<BF_PHASE_FAILED>(mtt, p0, p1, p2, p3);
        TERM |= mtt; COMPL |= mtt & AF; FAILED |= mtt & ~AF; RUN &= ~mtt; RUNQ &= ~mtt;
        const uint32_t b2 = __reduce_or_sync(gmask, (mtt != 0 ? 1u : 0u) | ((FAILED & GM) != 0 ? 2u : 0u));
        if (tt) {
          marked = marked || (b2 & 1u);
          main_done = true;
          amf = b2 & 2u;
        }
      }
      bool comp_done;
      if (auto_group && main_done && !amf && n_comp != 0) {
        marked = marked || (bits & 512u);
        pset<BF_PHASE_SKIPPED>(mark_cs, p0, p1, p2, p3);
        TERM |= mark_cs; COMPL |= mark_cs;
        comp_done = !(bits & 16u);
      } else {
        comp_done = n_comp == 0 || !(bits & 8u);
      }
      const bool final_done = n_final == 0 || !(bits & 32u);
      const bool aff = bits & 128u;
      if (!main_done) group = BF_GROUP_MAIN;
      else if (amf && n_comp != 0 && !comp_done) group = BF_GROUP_COMPENSATION;
      else if (n_final != 0 && !final_done) group = BF_GROUP_FINALLY;
      else group = BF_GROUP_DONE;
      sum = (main_done ? BF_SUM_MAIN_DONE : 0u) | (amf ? BF_SUM_MAIN_FAILED : 0u) | (comp_done ? BF_SUM_COMP_DONE : 0u) |
            (final_done ? BF_SUM_FINAL_DONE : 0u) | (acf ? BF_SUM_COMP_FAILED : 0u) | (aff ? BF_SUM_FINAL_FAILED : 0u);
    }
    if (host_group) {
      group = (rflags >> BF_RF_HOST_GROUP_SHIFT) & 3u;
      sum = 0;
    }
    uint32_t summary = sum | group;

    // ------------- D-prep: dependency classes under this pass's policy (dag.go:499-502) -------------
    const bool evaluate = group != BF_GROUP_DONE;
    const bool allow_failed = group != BF_GROUP_MAIN;
    const bool skip_on_failed = group == BF_GROUP_MAIN && !fail_fast;
    const uint32_t GSEL = group == BF_GROUP_MAIN ? GM : (group == BF_GROUP_COMPENSATION ? G1 : G2);
    const uint32_t SAT = COMPL | (realtime ? plut<BF_LUT_RT_SAT>(p0, p1, p2, p3) : 0u) | (allow_failed ? TERM : 0u);
    const uint32_t U = VALID & ~SAT;   // & VALID: bytes past the last step (the PAD byte of a narrower run) read "satisfied"
    const uint32_t FD = skip_on_failed ? (TERM & ~SAT) : 0u;
    const uint32_t CAND0 = evaluate ? (GSEL & ~COMPL & ~RUNQ & ~TERM) : 0u;
    const uint32_t FREE = CAND0 & NODEP;   // candidates without needs: met by definition (byte-entry rows only)
    const uint32_t CAND = CAND0 & ~NODEP;  // the candidates whose rows are walked
    // ------------- stage C: one status byte per step (bit0 unmet, bit1 failed-dep), all R runs -------------
    const bool any_fd = __any_sync(FULL, skip_on_failed);              // some run of the group has a failed-dependency class
    const int my_fmt = fmt_of(ell, max_deg);
    const int fmt0 = __shfl_sync(FULL, live ? my_fmt : -1, __ffs(__ballot_sync(FULL, live) | 0x80000000u) - 1);  // format of the first live run
    const bool mixed = __any_sync(FULL, live && my_fmt != fmt0);
    const uint32_t my_st = st0_a + g * st_stride;
    __syncwarp();
    {
      // every lane writes the 32 bytes of its own word, 16 steps per store; the half a lane stores first follows lane bit 2,
      // so that at Wq = 8 (words 32 bytes apart) the 8 lanes of each store phase cover all 32 banks
      const uint32_t hs = lane & 4u ? 16u : 0u;
      const uint32_t u = __funnelshift_r(U, U, hs), f = __funnelshift_r(FD, FD, hs);   // step hs + j at bit j
#pragma unroll
      for (uint32_t it = 0; it < 2; ++it) {
        const uint32_t s = it * 16u;
        uint32_t v0 = bits4_to_bytes((u >> s) & 0xFu), v1 = bits4_to_bytes((u >> (s + 4u)) & 0xFu);
        uint32_t v2 = bits4_to_bytes((u >> (s + 8u)) & 0xFu), v3 = bits4_to_bytes((u >> (s + 12u)) & 0xFu);
        if (any_fd) {  // warp-uniform
          v0 |= bits4_to_bytes((f >> s) & 0xFu) << 1; v1 |= bits4_to_bytes((f >> (s + 4u)) & 0xFu) << 1;
          v2 |= bits4_to_bytes((f >> (s + 8u)) & 0xFu) << 1; v3 |= bits4_to_bytes((f >> (s + 12u)) & 0xFu) << 1;
        }
        sts_v4(my_st + w * 32u + (hs ^ s), v0, v1, v2, v3);
      }
    }
    // per-run walk entry: CSR / row bases, status base, longest row and row format
    const uint32_t col_a = tr_a + (h1.x & 0xFFFFu);
    if (w == 0) sts_v4(tab_a + g * 16u, col_a, tr_a + (uint32_t)sizeof(TopoHeader), my_st, max_deg | (ell << 16));
    __syncwarp();
    // second link of the group I shall issue (its slot id, requested when I drew my ticket, has arrived by now — asking for
    // it right behind the barrier wait stalled every trip for a DRAM round trip); consumed by issue() at the end of the trip.
    // The entry lands in shared memory, not in registers that would stay live through the walk: in the head of state record
    // lr of this slot group, which nothing reads once the planes above are loaded (the __syncwarp orders those reads first)
    // and which the re-arm overwrites only after issue() has read the entry back.
    const uint32_t ent_a = grp_a + lr * P.state_stride;
    if (lq == 0) cp_async16(ent_a, P.slots + (pf_sid < P.n_slots ? pf_sid : 0u), pf_sid < P.n_slots ? 16u : 0u);
    // ------------- stage D: walk the needs rows (dag.go:2711-2733) -------------
    uint32_t met_w, fd_w;
    const WalkCtx wctx{tab_a, grp_a + R * P.state_stride + (uint32_t)sizeof(TopoHeader), P.topo_buf_bytes, st0_a, st_stride};
    if (mixed) {
      if (any_fd) walk_items_any<true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items_any<false>(lane, CAND, lg, wctx, met_w, fd_w);
    } else if (fmt0 == FMT_ELL4B && Wq == 8u) {   // 129 .. 256 steps: status bytes on 256-byte boundaries
      if (any_fd) walk_items<FMT_ELL4B, true, true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items<FMT_ELL4B, false, true>(lane, CAND, lg, wctx, met_w, fd_w);
    } else if (fmt0 == FMT_ELL4B) {
      if (any_fd) walk_items<FMT_ELL4B, true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items<FMT_ELL4B, false>(lane, CAND, lg, wctx, met_w, fd_w);
    } else if (fmt0 == FMT_ELL2B) {
      if (any_fd) walk_items<FMT_ELL2B, true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items<FMT_ELL2B, false>(lane, CAND, lg, wctx, met_w, fd_w);
    } else if (fmt0 == FMT_ELL4) {
      if (any_fd) walk_items<FMT_ELL4, true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items<FMT_ELL4, false>(lane, CAND, lg, wctx, met_w, fd_w);
    } else if (fmt0 == FMT_CSR4) {
      if (any_fd) walk_items<FMT_CSR4, true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items<FMT_CSR4, false>(lane, CAND, lg, wctx, met_w, fd_w);
    } else if (fmt0 == FMT_ELL2) {
      if (any_fd) walk_items<FMT_ELL2, true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items<FMT_ELL2, false>(lane, CAND, lg, wctx, met_w, fd_w);
    } else {
      if (any_fd) walk_items<FMT_CSRL, true>(lane, CAND, lg, wctx, met_w, fd_w);
      else walk_items<FMT_CSRL, false>(lane, CAND, lg, wctx, met_w, fd_w);
    }
    met_w |= FREE;
    uint32_t ready_w = met_w, skipc_w = 0, fail_w = 0;
    if (CD) {
      ready_w = met_w & ~c0 & ~c1;   // BF_COND_PASS
      skipc_w = met_w & c0 & ~c1;    // BF_COND_SKIP
      fail_w = met_w & c0 & c1;      // BF_COND_FAIL
      if (__any_sync(FULL, fail_w != 0)) {
        // a step set Failed inside the loop is visible to LATER steps of the list only (dag.go:2745, :497)
        const uint32_t fclass = allow_failed ? 0u : (skip_on_failed ? 3u : 1u);
        const uint32_t wmask = (1u << lg) - 1u;
        for (uint32_t round = 0; round <= 32u * Wmax; ++round) {
          __syncwarp();
          sts_u32(mfail_a + lane * 4u, fail_w);
          __syncwarp();
          met_w = 0; fd_w = 0;
          for (uint32_t todo = __ballot_sync(FULL, CAND != 0); todo; todo &= todo - 1) {
            const uint32_t L = __ffs(todo) - 1;
            const uint4 te = lds_v4(tab_a + (L >> lg) * 16u);
            uint32_t mb, fb;
            fixup_item(lane, __shfl_sync(FULL, CAND, L), L & wmask, te.w >> 16, te.y, te.x, te.z, mfail_a + ((L >> lg) << lg) * 4u,
                       __shfl_sync(FULL, fclass, L), mb, fb);
            if (lane == L) { met_w = mb; fd_w = fb; }
          }
          met_w |= FREE;
          const uint32_t nf = met_w & c0 & c1;
          const bool same = !__any_sync(FULL, nf != fail_w);
          fail_w = nf;
          if (same) break;
        }
        ready_w = met_w & ~c0 & ~c1;
        skipc_w = met_w & c0 & ~c1;
      }
      pset<BF_PHASE_FAILED>(fail_w, p0, p1, p2, p3);  // dag.go:2745-2747, 2810-2812
    }
    const uint32_t acc_ready = ready_w, acc_skip = fd_w | skipc_w;

    // ---------------- stage E: result records ----------------
    const uint32_t cnt = __reduce_add_sync(gmask, (uint32_t)__popc(acc_ready) | ((uint32_t)__popc(acc_skip) << 16));
    bool changed = marked;
    if (CD) changed = (__ballot_sync(FULL, ((p0 ^ q0) | (p1 ^ q1) | (p2 ^ q2) | (p3 ^ q3)) != 0) & gmask) != 0;
    // fused compaction head (compact.cu): events of the run = steps with a bit in any result mask the layout carries
    uint32_t n_events = 0;
    if (P.head) {
      uint32_t u = acc_ready | acc_skip;
      if (XO) {
        if (P.off_fail != BF_OFF_NONE) u |= fail_w;
        if (P.off_needs_cond != BF_OFF_NONE) u |= realtime ? 0u : (met_w & HASIF);
        if (P.off_skip_dep != BF_OFF_NONE) u |= fd_w;
      }
      n_events = __reduce_add_sync(gmask, (uint32_t)__popc(u));
    }
    if (deferred) {
      if (w == 0) P.defer_list[atomicAdd(P.defer_count, 1u)] = r;  // the general kernel writes this run's record
    } else if (in_batch) {
      if (w == 0) {
        summary = live ? (summary | (changed ? BF_SUM_PHASE_CHANGED : 0u) | (1u << BF_SUM_ITER_SHIFT)) : 0xFFFFFFFFu;
        *reinterpret_cast<uint4*>(rr) = make_uint4(summary, cnt & 0xFFFFu, cnt >> 16, 0u);
        if (P.exp_counts) P.exp_counts[r] = 0;
        if (P.head) {
          P.head[r] = live ? ((summary & BF_HEAD_SUMMARY_MASK) | BF_HEAD_LISTED | (n_events << BF_HEAD_COUNT_SHIFT)) : (BF_HEAD_DEAD | BF_HEAD_LISTED);
          if (live && n_events) atomicAdd(&P.head_sums[r >> 9], (unsigned long long)n_events);
        }
      }
      if (w < Wmax) {
        reinterpret_cast<uint32_t*>(rr + P.off_ready)[w] = acc_ready;
        reinterpret_cast<uint32_t*>(rr + P.off_skip)[w] = acc_skip;
        if (XO) {
          if (P.off_fail != BF_OFF_NONE) reinterpret_cast<uint32_t*>(rr + P.off_fail)[w] = fail_w;
          if (P.off_needs_cond != BF_OFF_NONE) reinterpret_cast<uint32_t*>(rr + P.off_needs_cond)[w] = realtime ? 0u : (met_w & HASIF);
          if (P.off_skip_dep != BF_OFF_NONE) reinterpret_cast<uint32_t*>(rr + P.off_skip_dep)[w] = fd_w;
          if (P.off_phase_out != BF_OFF_NONE) {
            uint32_t* po = reinterpret_cast<uint32_t*>(rr + P.off_phase_out) + w;
            po[0] = p0; po[Wmax] = p1; po[2 * Wmax] = p2; po[3 * Wmax] = p3;
          }
        }
      }
      if (P.result_tail != P.result_stride)
        for (uint32_t x = P.result_tail / 4 + w; x < P.result_stride / 4; x += Wq) reinterpret_cast<uint32_t*>(rr)[x] = 0u;
    }
    lane_ready += (uint32_t)__popc(acc_ready);
    lane_skip += (uint32_t)__popc(acc_skip);
    lane_evals += (w == 0 && live) ? S : 0u;

    __syncwarp();  // every lane is done with this slot group's buffers
    uint4 ent = make_uint4(0u, 0u, 0u, 0u);
    if (lq == 0) {
      cp_async_wait_all();
      ent = lds_v4(ent_a);
    }
    issue(t + NG, cur_sg, cur_use + 1u, lq == 0, ent);  // re-arm it with group t + NG (consumed by whichever warp draws that ticket)
#ifdef PACK_TRACE
    if (t == 0 && lane == 0 && blockIdx.x < 160) g_trace[tr_launch][blockIdx.x][1] = tr_first;
    tr_last = gtime();
#endif
  }
#ifdef PACK_TRACE
  if (lane == 0 && blockIdx.x < 160) atomicMax(&g_trace[tr_launch][blockIdx.x][2], tr_last);
#endif

  // ---- BF_EVAL_PIPELINED: this grid may have started before the preceding kernel of the stream ended (it reads and writes
  // nothing of that kernel's); from here on it touches the counts and then completes, so that kernel must be complete.
  if (P.flags & BF_EVAL_PIPELINED) asm volatile("griddepcontrol.wait;" ::: "memory");
  // ---- counters: lane -> warp (redux) -> block (shared atomics) -> one global atomic per block ----
  if (P.counts) {
    const uint32_t wr = redux_add(lane_ready), ws = redux_add(lane_skip), we = redux_add(lane_evals);
    if (lane == 0) {
      atomicAdd(&blk_counts[0], (unsigned long long)wr);
      atomicAdd(&blk_counts[1], (unsigned long long)ws);
      atomicAdd(&blk_counts[3], (unsigned long long)we);
    }
    __syncthreads();
    if (P.acc == nullptr) {
      if (threadIdx.x < 4 && blk_counts[threadIdx.x] != 0ull) atomicAdd(&P.counts[threadIdx.x], blk_counts[threadIdx.x]);
    } else {
      // BF_EVAL_COUNTS_SET: totals gathered in this launch's block of the ctx scratch ring; the last CTA out writes them to
      // `counts` and clears the block for the launch that gets it next
      if (threadIdx.x < 4 && blk_counts[threadIdx.x] != 0ull) atomicAdd(&P.acc[threadIdx.x], blk_counts[threadIdx.x]);
      __threadfence();
      __syncthreads();
      volatile unsigned int* last_out = reinterpret_cast<volatile unsigned int*>(smem_p + 40);   // free word of the counter block
      if (threadIdx.x == 0) *last_out = atomicAdd(reinterpret_cast<unsigned int*>(&P.acc[4]), 1u) == gridDim.x - 1u;
      __syncthreads();
      if (*last_out) {
        __threadfence();
        if (threadIdx.x < 4) P.counts[threadIdx.x] = atomicExch(&P.acc[threadIdx.x], 0ull);
        if (threadIdx.x == 4) P.acc[4] = 0ull;
      }
    }
  }
#ifdef PACK_TRACE
  __syncthreads();
  if (threadIdx.x == 0 && blockIdx.x < 160) {
    g_trace[tr_launch][blockIdx.x][0] = tr_start;
    g_trace[tr_launch][blockIdx.x][3] = gtime();
    __threadfence();
    if (atomicAdd(reinterpret_cast<unsigned int*>(&g_trace[tr_launch][159][0]), 1u) == gridDim.x - 1) {   // last CTA out
      *reinterpret_cast<unsigned int*>(&g_trace[tr_launch][159][0]) = 0u;
      atomicAdd(&g_launch, 1u);
      for (int b = 0; b < 160; ++b) g_trace[(tr_launch + 1) & 7u][b][2] = 0ull;   // next launch's atomicMax cells
    }
  }
#endif
}

typedef void (*PackFn)(const KParams);
static PackFn pick_pack(const KParams& P) {
  const bool cd = P.off_cond != BF_OFF_NONE || P.off_decision != BF_OFF_NONE;
  const bool xo = P.off_fail != BF_OFF_NONE || P.off_needs_cond != BF_OFF_NONE || P.off_skip_dep != BF_OFF_NONE ||
                  P.off_phase_out != BF_OFF_NONE;
  if (cd) return xo ? frontier_pack_kernel<true, true> : frontier_pack_kernel<true, false>;
  return xo ? frontier_pack_kernel<false, true> : frontier_pack_kernel<false, false>;
}

uint32_t frontier_pack_max_warps() { return PACK_MAX_WARPS; }
#ifdef PACK_TRACE
extern "C" int bf_debug_pack_trace(unsigned long long* out, unsigned int* launch) {
  cudaDeviceSynchronize();
  if (cudaMemcpyFromSymbol(out, g_trace, sizeof(g_trace)) != cudaSuccess) return -1;
  return cudaMemcpyFromSymbol(launch, g_launch, sizeof(unsigned int)) == cudaSuccess ? 0 : -1;
}
#endif

cudaError_t launch_frontier_pack(const KParams& P, uint32_t grid, uint32_t smem_bytes, cudaStream_t stream) {
  PackFn fn = pick_pack(P);
  static PackFn configured[8][4] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  bool known = false;
  if (dev >= 0 && dev < 8)
    for (int i = 0; i < 4; ++i) known = known || configured[dev][i] == fn;
  if (!known) {
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 8)
      for (int i = 0; i < 4; ++i)
        if (configured[dev][i] == nullptr) { configured[dev][i] = fn; break; }
  }
  if (P.flags & BF_EVAL_PIPELINED) {   // programmatic dependent launch: may start while the preceding kernel drains
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(P.warps_per_block * 32); cfg.dynamicSmemBytes = smem_bytes; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, fn, P);
  }
  fn<<<grid, P.warps_per_block * 32, smem_bytes, stream>>>(P);
  return cudaGetLastError();
}

}  // namespace bf
