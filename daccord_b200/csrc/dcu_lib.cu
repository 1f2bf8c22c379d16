// dcu_lib.cu -- sm_100a kernel wrapper and C-ABI (include/daccord_b200.h) of the window-consensus engine.
// One persistent launch per batch: every warp pulls window indices from a global ticket counter and runs
// dcu::process_window (window_core.cuh) on its private workspace slab.  Windows whose graph does not fit
// the small (tier 0) slab are queued and re-run by a second launch on large (tier 1) slabs -- still on the
// GPU; there is no CPU path in this library.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>
#include <new>
#include <mutex>
#include <chrono>
#include "window_core.cuh"            // namespace dcu : every workspace field in the warp's HBM slab (overflow passes, deep piles)
#define DCU_NS dcus
#define DCU_TIER_SMEM 1
#include "window_core.cuh"            // namespace dcus: hot fields in the warp's shared-memory arena (optional first pass)
#define DCU_NS dcuh
#define DCU_TIER_SMEM 2
#include "window_core.cuh"            // namespace dcuh: only the k-mer table in shared memory, at full occupancy (first pass of deep, clean piles)
#include "host_tables.hpp"
#include "host_caps.hpp"
#include "pile_host.hpp"
#include "vote_host.hpp"
#include "../../include/daccord_b200.h"

static_assert(sizeof(dcu::Slice) == sizeof(dcu_slice) && sizeof(dcu::Window) == sizeof(dcu_window) && sizeof(dcu::Result) == sizeof(dcu_result), "ABI structs");
static_assert(sizeof(dvote::Win) == sizeof(dcu_window) && sizeof(dvote::Res) == sizeof(dcu_result), "ABI structs (vote)");

namespace {

constexpr int WPB = 16;                // warps per block of the HBM passes
constexpr int BPS = 2;                 // resident blocks per SM the HBM kernel is compiled for (64 registers / thread)
constexpr int SWPB = 16;               // most warps per block of the shared-memory pass (one block per SM, 128 registers / thread)

struct KArgs {
  const uint8_t* packed; const dcu::Slice* sl; const dcu::Window* win;
  dcu::Result* res; uint8_t* cons; uint8_t* ops;
  uint8_t* slabs;                      // [total warps][layout bytes]
  const uint32_t* todo;                // window indices to run (nullptr: 0..n-1)
  uint32_t n; uint32_t vs_words;       // vs_words != 0: stage the VS table in dynamic shared memory
  int sync_group;                      // warps per phase-synchronous group (1 = free running)
  int sync_mask;                       // inner stage boundaries that are barriers
  unsigned int* ticket;                // work counter
  unsigned int* ovf_cnt; uint32_t* ovf_list;   // windows that overflowed this pass
  unsigned long long packed_bytes;     // readable bytes of the packed database (staging never reads beyond)
  int stage;                           // shared-memory pass: stage the slices of the next window with cp.async.bulk
  unsigned int launch_seq;             // number of this launch in the context's life (upper half of the forward slot tags: records of earlier launches in the slab are stale)
};

// One persistent launch per pass.  Every warp owns one window at a time and walks it through the stages of window_core.cuh; the
// warps of a group (named barriers) run the same stage at the same time, which keeps the instruction caches effective
// (profiles/r01_summary.md).  NS = dcu (HBM workspace) or dcus (hot fields in shared memory, slices staged by bulk copies).
#define DCU_STAGE_LOOP(NS, FINAL_HOOK)                                                                                          \
    if (G == 1) alldone = idle;                                                                                                 \
    else {                                                                                                                      \
      if (lane == 0) s_done[par][warp] = idle ? 1 : 0;                                                                          \
      gsync();                                                                                                                  \
      alldone = true;                                                                                                           \
      for (int i = 0; i < G; ++i) alldone = alldone && (s_done[par][gfirst + i] != 0);                                          \
    }                                                                                                                           \
    if (alldone) break;                                                                                                         \
    if (st.ph == NS::PH_HASH) NS::st_hash(c, st, lane);                                                                         \
    if (smask & 1) gsync();                                                                                                     \
    if (st.ph == NS::PH_NODES) NS::st_nodes(c, st, lane);                                                                       \
    if (smask & 32) gsync();                                                                                                    \
    if (st.ph == NS::PH_EDGES) NS::st_edges(c, st, lane);                                                                       \
    if (smask & 2) gsync();                                                                                                     \
    if (st.ph == NS::PH_TRAV) NS::st_trav(c, st, lane);                                                                         \
    if (smask & 16) gsync();                                                                                                    \
    if (st.ph == NS::PH_POS) NS::st_pos(c, st, lane);                                                                           \
    if (smask & 4) gsync();                                                                                                     \
    if (st.ph == NS::PH_RPATH) NS::st_rpath(c, st, lane);                                                                       \
    if (smask & 64) gsync();                                                                                                    \
    if (st.ph == NS::PH_SEARCH) NS::st_search(c, st, lane);                                                                     \
    if (smask & 128) gsync();                                                                                                   \
    if (st.ph == NS::PH_SCORE) NS::st_score(c, st, lane);                                                                       \
    if (smask & 8) gsync();                                                                                                     \
    if (st.ph == NS::PH_FINAL) { FINAL_HOOK; NS::st_final(c, st, a.cons + (size_t)wi * DCU_CONS_STRIDE, a.ops + (size_t)wi * DCU_OPS_STRIDE, lane); } \
    if (st.ph == NS::PH_END && !idle) { publish(); __syncwarp(); }

// ---- HBM build: layout, capacities, table descriptors and parameters in __constant__ memory (dcu::c_*), set per launch
// W warps per block, two blocks per SM: W = 16 gives 64 registers per thread, W = 12 (DCU_WPB=12, measurement knob) 85 at 24 warps per SM
template <int W, int B = BPS> __global__ void __launch_bounds__(W * 32, B) dcu_window_kernel(const __grid_constant__ KArgs a) {
  extern __shared__ unsigned long long s_vs[];          // block-shared copy of the transposed VS table (when it fits)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (a.vs_words) { for (uint32_t i = threadIdx.x; i < a.vs_words; i += blockDim.x) s_vs[i] = dcu::c_T.VSq[i]; __syncthreads(); }
  dcu::Ctx c;
  c.ws.base = a.slabs + ((size_t)blockIdx.x * W + warp) * (size_t)dcu::c_layout.bytes;
  c.vsq = a.vs_words ? s_vs : dcu::c_T.VSq; c.vs_sm = a.vs_words ? 1 : 0; c.epoch = (unsigned long long)a.launch_seq << 32;
  c.packed = a.packed; c.sl = a.sl;
  __shared__ int s_done[2][W];                         // double buffered: with a single barrier per round a fast warp must not overwrite what a slow one still reads
  const int G = a.sync_group, grp = warp / G, gfirst = grp * G;
  auto gsync = [&]() { if (G > 1) asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "r"(G * 32) : "memory"); };
  const int smask = a.sync_mask;                       // which of the inner stage boundaries are barriers (bit 0: hash|nodes, 5: nodes|edges, 1: edges|trav, 4: trav|pos, 2: pos|rpath, 6: rpath|search, 7: search|score, 3: score|final)
  dcu::WinState st; st.ph = dcu::PH_END;
  uint32_t wi = 0; bool nomore = false; int par = 0;
  auto publish = [&]() {
    if (lane == 0) {
      a.res[wi] = st.res;
      if (st.res.status == dcu::ST_OVERFLOW) { unsigned int o = atomicAdd(a.ovf_cnt, 1u); a.ovf_list[o] = wi; }
    }
  };
  for (;; par ^= 1) {
    while (!nomore && st.ph == dcu::PH_END) {          // finish / fetch
      unsigned int t = 0;
      if (lane == 0) t = atomicAdd(a.ticket, 1u);
      t = __shfl_sync(0xffffffffu, t, 0);
      if (t >= a.n) { nomore = true; break; }
      wi = a.todo ? a.todo[t] : t;
      const dcu::Window wd = a.win[wi];
      dcu::st_begin(c, st, wd, lane, nullptr);
      if (st.ph == dcu::PH_END) publish();             // skipped or overflowed right away
    }
    const bool idle = st.ph == dcu::PH_END;
    bool alldone;
    DCU_STAGE_LOOP(dcu, (void)0)
  }
}

// ---- hybrid build: as dcu_window_kernel, plus a 5 KB arena per warp behind the VS table that holds the window's k-mer table
__global__ void __launch_bounds__(WPB * 32, BPS) dcuh_window_kernel(const __grid_constant__ KArgs a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t vs_bytes = (a.vs_words * 8u + 127u) & ~127u;
  if (a.vs_words) { unsigned long long* s_vs = (unsigned long long*)dcuh::dcu_smem; for (uint32_t i = threadIdx.x; i < a.vs_words; i += blockDim.x) s_vs[i] = dcuh::c_T.VSq[i]; __syncthreads(); }
  dcuh::Ctx c;
  c.ws.base = a.slabs + ((size_t)blockIdx.x * WPB + warp) * (size_t)dcuh::c_layout.bytes;
  c.ws.sm = vs_bytes + (uint32_t)warp * dcuh::c_layout.sbytes;
  c.vsq = a.vs_words ? (const unsigned long long*)dcuh::dcu_smem : dcuh::c_T.VSq; c.vs_sm = a.vs_words ? 1 : 0; c.epoch = (unsigned long long)a.launch_seq << 32;
  c.packed = a.packed; c.sl = a.sl;
  __shared__ int s_done[2][WPB];
  const int G = a.sync_group, grp = warp / G, gfirst = grp * G;
  auto gsync = [&]() { if (G > 1) asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "r"(G * 32) : "memory"); };
  const int smask = a.sync_mask;
  dcuh::WinState st; st.ph = dcuh::PH_END;
  uint32_t wi = 0; bool nomore = false; int par = 0;
  auto publish = [&]() {
    if (lane == 0) {
      a.res[wi] = st.res;
      if (st.res.status == dcuh::ST_OVERFLOW) { unsigned int o = atomicAdd(a.ovf_cnt, 1u); a.ovf_list[o] = wi; }
    }
  };
  for (;; par ^= 1) {
    while (!nomore && st.ph == dcuh::PH_END) {         // finish / fetch
      unsigned int t = 0;
      if (lane == 0) t = atomicAdd(a.ticket, 1u);
      t = __shfl_sync(0xffffffffu, t, 0);
      if (t >= a.n) { nomore = true; break; }
      wi = a.todo ? a.todo[t] : t;
      const dcu::Window wd = a.win[wi];
      dcuh::st_begin(c, st, wd, lane, nullptr);
      if (st.ph == dcuh::PH_END) publish();
    }
    const bool idle = st.ph == dcuh::PH_END;
    bool alldone;
    DCU_STAGE_LOOP(dcuh, (void)0)
  }
}

// ---- shared-memory build: dynamic shared memory = [transposed VS table | one arena per warp]; the packed bytes of the next
// window's slices are copied into the (then idle) pre-filter bitmap region of the arena by cp.async.bulk, completion on a
// per-warp mbarrier, while the current window is placed
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__global__ void __launch_bounds__(SWPB * 32, 1) dcus_window_kernel(const __grid_constant__ KArgs a) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t vs_bytes = (a.vs_words * 8u + 127u) & ~127u;
  {
    unsigned long long* s_vs = (unsigned long long*)dcus::dcu_smem;
    for (uint32_t i = threadIdx.x; i < a.vs_words; i += blockDim.x) s_vs[i] = dcus::c_T.VSq[i];
  }
  __shared__ int s_done[2][SWPB];
  __shared__ __align__(8) unsigned long long s_mbar[SWPB];
  if (lane == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s_mbar[warp])) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  dcus::Ctx c;
  c.ws.base = a.slabs + ((size_t)blockIdx.x * (blockDim.x >> 5) + warp) * (size_t)dcus::c_layout.bytes;
  c.ws.sm = vs_bytes + (uint32_t)warp * dcus::c_layout.sbytes;
  c.vsq = a.vs_words ? (const unsigned long long*)dcus::dcu_smem : dcus::c_T.VSq; c.vs_sm = a.vs_words ? 1 : 0; c.epoch = (unsigned long long)a.launch_seq << 32;
  c.packed = a.packed; c.sl = a.sl;
  const int G = a.sync_group, grp = warp / G, gfirst = grp * G;
  auto gsync = [&]() { if (G > 1) asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "r"(G * 32) : "memory"); };
  const int smask = a.sync_mask;
  dcus::WinState st; st.ph = dcus::PH_END;
  uint32_t wi = 0; bool nomore = false; int par = 0;
  // staging state: pf = 0 nothing claimed, 1 window pfwi claimed and its slices in flight / landed, 2 claimed but not staged (direct loads)
  int pf = 0; uint32_t pfwi = 0, mpar = 0;
  uint8_t* const raw = dcus::dcu_smem + c.ws.sm + dcus::c_layout.off[dcus::F_hbA];
  const uint32_t rawcap = dcus::c_layout.off[dcus::F_hstate] - dcus::c_layout.off[dcus::F_hbA];
  const uint32_t mbar = smem_u32(&s_mbar[warp]);
  auto publish = [&]() {
    if (lane == 0) {
      a.res[wi] = st.res;
      if (st.res.status == dcus::ST_OVERFLOW) { unsigned int o = atomicAdd(a.ovf_cnt, 1u); a.ovf_list[o] = wi; }
    }
  };
  // claims the next window and starts the copies of its slices; the chunk offsets are the ones load_window recomputes
  auto claim = [&]() {
    unsigned int t = 0;
    if (lane == 0) t = atomicAdd(a.ticket, 1u);
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t >= a.n) { nomore = true; return; }
    pfwi = a.todo ? a.todo[t] : t;
    pf = 2;
    if (!a.stage) return;
    const dcu::Window W = a.win[pfwi];
    const int n = W.slice_cnt;
    if (n == 0 || n > dcus::c_cap.S) return;
    const dcu::Slice* sl = a.sl + W.slice_begin;
    uint32_t total = 0; bool ok = true;
    for (int base = 0; base < n; base += 32) {
      const int j = base + lane; uint32_t stt = 0, cb = 0;
      if (j < n) { dcus::slice_chunk(sl[j], stt, cb); if ((unsigned long long)stt + cb > a.packed_bytes) ok = false; }
      total += __reduce_add_sync(0xffffffffu, cb);
    }
    if (__ballot_sync(0xffffffffu, !ok) || total == 0 || total > rawcap) return;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the region was last written through the generic proxy (bitmaps)
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%1], %0;" ::"r"(total), "r"(mbar) : "memory");
    __syncwarp();
    uint32_t run = 0;
    for (int base = 0; base < n; base += 32) {
      const int j = base + lane; uint32_t stt = 0, cb = 0;
      if (j < n) dcus::slice_chunk(sl[j], stt, cb);
      const uint32_t inc = dcus::scan_incl(cb, lane);
      if (cb) asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                           ::"r"(smem_u32(raw + run + inc - cb)), "l"(a.packed + stt), "r"(cb), "r"(mbar) : "memory");
      run += __shfl_sync(0xffffffffu, inc, 31);
    }
    pf = 1;
  };
  for (;; par ^= 1) {
    while (st.ph == dcus::PH_END) {                    // finish / fetch
      if (pf == 0) { if (nomore) break; claim(); if (pf == 0) break; }
      const uint8_t* rawp = nullptr;
      if (pf == 1) {                                   // wait for the bytes
        asm volatile("{\n\t.reg .pred P1;\n\tLAB_WAIT:\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t@P1 bra DONE;\n\tbra LAB_WAIT;\n\tDONE:\n\t}" ::"r"(mbar), "r"(mpar) : "memory");
        mpar ^= 1u; rawp = raw;
      }
      pf = 0; wi = pfwi;
      dcu::Window W = a.win[wi];
      dcus::st_begin(c, st, W, lane, rawp);
      if (st.ph == dcus::PH_END) publish();            // skipped or overflowed right away
    }
    const bool idle = st.ph == dcus::PH_END;
    bool alldone;
    DCU_STAGE_LOOP(dcus, if (pf == 0 && !nomore) claim())
  }
}

// ---------------------------------------------------------------- piling kernels (pile_core.cuh), one thread per item
// ---- scan helpers shared by the piling and vote stages: one value per thread, SCAN_TPB threads per block
constexpr int VOTE_TPB = 256;
// block-wide exclusive scan of one value per thread (VOTE_TPB threads); returns the thread's offset, *total = block sum
__device__ __forceinline__ uint32_t block_exscan(uint32_t v, uint32_t* total) {
  __shared__ uint32_t s_w[VOTE_TPB / 32];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  uint32_t x = v;
  for (int d = 1; d < 32; d <<= 1) { uint32_t y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
  if (lane == 31) s_w[wp] = x;
  __syncthreads();
  uint32_t base = 0, tot = 0;
  for (int i = 0; i < VOTE_TPB / 32; ++i) { if (i < wp) base += s_w[i]; tot += s_w[i]; }
  __syncthreads();
  *total = tot;
  return base + x - v;
}
// exclusive scan of the block sums in place (one block); blk[nblk] = grand total
__global__ void __launch_bounds__(VOTE_TPB) vote_kscan(uint64_t* blk, uint64_t nblk) {
  __shared__ uint64_t s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint64_t base = 0; base < nblk; base += VOTE_TPB) {
    const uint64_t i = base + threadIdx.x;
    const uint32_t v = i < nblk ? (uint32_t)blk[i] : 0u;          // a block sum is < 2^32 (<= 127 * VOTE_TPB)
    uint32_t total;
    const uint32_t off = block_exscan(v, &total);
    const uint64_t carry = s_carry;
    if (i < nblk) blk[i] = carry + off;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + total;
    __syncthreads();
  }
  if (threadIdx.x == 0) blk[nblk] = s_carry;
}

__global__ void pile_k0(const dpile::Ovl* ovl, uint64_t novl, const uint16_t* trace, uint32_t* tile_b) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < novl) dpile::pile_tile_starts(ovl[i], trace, tile_b);
}
__global__ void __launch_bounds__(64) pile_k1(const dpile::Ovl* ovl, uint64_t novl, uint64_t ntiles, const dpile::ReadInfo* reads, dpile::Params P, const uint16_t* trace,
                                              const uint32_t* tile_b, const uint8_t* packed, const uint64_t* read_boff, const uint32_t* read_len, uint32_t* bm) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ntiles) return;
  uint64_t a = 0, b = novl;                       // last overlap with tile_off <= t
  while (b - a > 1) { uint64_t mid = (a + b) >> 1; if (ovl[mid].tile_off <= t) a = mid; else b = mid; }
  const dpile::Ovl o = ovl[a];
  const uint32_t l = reads[o.ridx].maxaepos, s0 = l >= P.w ? l - P.w : 0;
  dpile::U128 PV[dpile::PILE_MAXB + 1], MV[dpile::PILE_MAXB + 1], PH[dpile::PILE_MAXB + 1], MH[dpile::PILE_MAXB + 1];
  dpile::pile_align_tile(o, (int)(t - o.tile_off), P, trace, tile_b, packed, read_boff, read_len, s0, l, bm, PV, MV, PH, MH);
}
__global__ void pile_k2a(const dpile::ReadInfo* reads, uint64_t nr, const dpile::Ovl* ovl, const double* minerate, const double* ediv, unsigned long long* keys) {
  uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < nr) dpile::pile_order(reads[r], ovl, minerate[r], ediv[r], keys + reads[r].ovl_begin);
}
// one thread per candidate window.  pass 0 (win == nullptr): slices per candidate (0 = empty pile) and per block the number of
// windows and slices; pass 1: descriptors at the scanned offsets
__global__ void __launch_bounds__(VOTE_TPB) pile_k2(const dpile::ReadInfo* reads, const uint32_t* read_id, uint32_t nr, uint64_t ncand, const dpile::Ovl* ovl, dpile::Params P,
                                                   const uint32_t* bm, const uint64_t* read_boff, const uint32_t* read_len, const unsigned long long* keys,
                                                   uint32_t* cnt, uint64_t* blkw, uint64_t* blks, dpile::Win* win, dpile::Sl* sl, int* err) {
  const uint64_t idx = (uint64_t)blockIdx.x * VOTE_TPB + threadIdx.x;
  uint32_t n = 0, r = 0, y = 0;
  if (idx < ncand) {
    uint32_t a = 0, b = nr;                       // last read with win_off <= idx that has candidates
    while (b - a > 1) { uint32_t mid = (a + b) >> 1; if (reads[mid].win_off <= idx) a = mid; else b = mid; }
    r = a; y = (uint32_t)(idx - reads[r].win_off);
    if (!win) { n = (uint32_t)dpile::pile_window(reads[r], y, ovl, P, bm, read_boff, read_len, keys + reads[r].ovl_begin, read_id[r], nullptr, nullptr, 0u); cnt[idx] = n; }
    else n = cnt[idx];
  }
  uint32_t totw, tots;
  const uint32_t woff = block_exscan(n ? 1u : 0u, &totw);
  const uint32_t soff = block_exscan(n, &tots);
  if (!win) { if (threadIdx.x == 0) { blkw[blockIdx.x] = totw; blks[blockIdx.x] = tots; } return; }
  if (!n) return;
  const uint64_t wo = blkw[blockIdx.x] + woff, so = blks[blockIdx.x] + soff;
  if (dpile::pile_window(reads[r], y, ovl, P, bm, read_boff, read_len, keys + reads[r].ovl_begin, read_id[r], win + wo, sl + so, (uint32_t)so) < 0) atomicExch(err, 2);
}
// per-window pile statistics of a device-built batch: max slice count and max bases of a window
__global__ void pile_k3(const dpile::Win* win, const dpile::Sl* sl, uint64_t nwin, unsigned int* maxS, unsigned int* maxB) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nwin) return;
  const dpile::Win w = win[i]; unsigned int b = 0;
  for (uint32_t j = 0; j < w.slice_cnt; ++j) b += sl[w.slice_begin + j].len;
  atomicMax(maxS, (unsigned int)w.slice_cnt); atomicMax(maxB, b);
}

// ---- pile vote (vote_core.cuh): per window the offset table, per A position the column votes (count pass, then fill pass)
__global__ void vote_k0(const dvote::Res* res, const uint8_t* ops, uint64_t nwin, dvote::Params P, uint16_t* ent, int* err) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nwin || res[i].status != dvote::ST_OK) return;
  if (!dvote::vote_window_table(res[i], ops + i * P.ops_stride, P.w, ent + i * (P.w + 1))) atomicExch(err, 1);
}
// pass 0 (chars == nullptr): per position the character count (bit 7: the pile holds something there) and per block the sum;
// pass 1: the characters at blk_off[block] + in-block offset, and the run boundary records
__global__ void __launch_bounds__(VOTE_TPB) vote_k1(dvote::Ctx c, const dvote::Read* reads, uint32_t nr, uint64_t npos, uint8_t* flag, uint64_t* blk,
                                                   char* chars, dvote::Bound* bound, unsigned int* nbound, unsigned int bound_cap) {
  const uint64_t idx = (uint64_t)blockIdx.x * VOTE_TPB + threadIdx.x;
  uint32_t n = 0; bool present = false; uint32_t r = 0, p = 0;
  if (idx < npos) {
    uint32_t a = 0, b = nr;                       // last read with pos_off <= idx
    while (b - a > 1) { uint32_t mid = (a + b) >> 1; if (reads[mid].pos_off <= idx) a = mid; else b = mid; }
    r = a; p = (uint32_t)(idx - reads[r].pos_off);
    if (!chars) { n = (uint32_t)dvote::vote_position(c, reads[r], p, nullptr, &present); flag[idx] = (uint8_t)(n | (present ? 0x80u : 0u)); }
    else { n = flag[idx] & 0x7Fu; present = (flag[idx] & 0x80u) != 0; }
  }
  uint32_t total;
  const uint32_t off = block_exscan(n, &total);
  if (!chars) { if (threadIdx.x == 0) blk[blockIdx.x] = total; return; }
  if (idx >= npos || !present) return;
  const uint64_t o = blk[blockIdx.x] + off;
  if (n) { bool pr; dvote::vote_position(c, reads[r], p, chars + o, &pr); }
  const bool left = p > 0 && (flag[idx - 1] & 0x80u), right = p + 1 < reads[r].span && (flag[idx + 1] & 0x80u);
  if (!left) { unsigned int q = atomicAdd(nbound, 1u); if (q < bound_cap) bound[q] = dvote::Bound{o, r, p, 0u, 0u}; }
  if (!right) { unsigned int q = atomicAdd(nbound, 1u); if (q < bound_cap) bound[q] = dvote::Bound{o + n, r, p, 1u, 0u}; }
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_); return DCU_ERR_CUDA; } } while (0)

// The launch-wide state of the window kernels (layout, capacities, tables, parameters) lives in __constant__ memory, one copy per
// device and process: the window passes of several dcu_ctx on one device are therefore serialised by this lock (held from the
// constant upload to the end of the last pass).  Everything else -- piling, vote, copies, the host work of a batch -- runs
// concurrently, which is what lets a caller keep several batches in flight (daccord_main.cpp).
std::mutex g_window_pass_lock[64];

// DCU_TIMING=1: host-side lap times of dcu_pile / dcu_vote on stderr (measurement aid)
struct Laps {
  bool on; const char* what; std::chrono::steady_clock::time_point t0, t; std::string s;
  explicit Laps(const char* w) : on(getenv("DCU_TIMING") != nullptr), what(w), t0(std::chrono::steady_clock::now()), t(t0) {}
  void lap(const char* name) { if (!on) return; auto n = std::chrono::steady_clock::now(); char b[64]; snprintf(b, sizeof b, " %s %.1f", name, std::chrono::duration<double, std::milli>(n - t).count()); s += b; t = n; }
  ~Laps() { if (on) fprintf(stderr, "[timing] %s: total %.1f ms:%s\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), s.c_str()); }
};

template <class T> struct DevBuf {
  T* p = nullptr; size_t cap = 0;
  cudaError_t ensure(size_t n, bool zero = false) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = n + n / 4 + 16;
    cudaError_t e = cudaMalloc((void**)&p, want * sizeof(T));
    if (e == cudaSuccess) { cap = want; if (zero) e = cudaMemset(p, 0, want * sizeof(T)); }      // (workspace slabs start zeroed: no slot record carries a tag)
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

}  // namespace

struct dcu_ctx {
  int device = 0;
  dcu_params prm{};
  dcu_host::HostTables HT;
  dcu::Tables T{}; dcu::Params P{}; dcu::Params Pl[2] = {};     // Pl: the per-pass copies handed to the launches
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int num_sms = 0, blocks_per_sm[2] = {BPS, 1}; int sync_group = WPB; int sync_group_env = 0;
  int use_smem = 1; int smem_optin = 0;             // first pass in shared memory (DCU_NO_SMEM=1 turns it off); opt-in shared memory per block
  // tables
  DevBuf<double> dDPn, dDPsq; DevBuf<unsigned long long> dVSq, dklim; DevBuf<uint16_t> dsuplo, dsuphi;
  // database
  DevBuf<uint8_t> dpacked_own; const uint8_t* dpacked = nullptr; uint64_t packed_bytes = 0, packed_padded = 0;     // packed_padded: bytes that may be read (staging copies whole 16-byte chunks)
  // batch
  DevBuf<dcu::Window> dwin; DevBuf<dcu::Slice> dsl; DevBuf<dcu::Result> dres; DevBuf<uint8_t> dcons, dops;
  DevBuf<uint32_t> dovf[3]; DevBuf<unsigned int> dcnt;     // dcnt: [ticket, overflows] of the passes at 0 (HBM first), 2 (HBM large), 8 (shared memory); 4..7 piling / vote
  DevBuf<uint8_t> dslab[3];
  dcu::Caps caps[2]; dcu::Layout lay[2]; int grid[2] = {0, 0};
  dcu::Caps capsS{}; dcus::Layout layS{}; int warpsS = 0;   // shared-memory pass: capacities, layout, warps per block
  dcu::Caps capsH{}; dcuh::Layout layH{}; int use_hybrid = 0, hybrid_ok = 0; DevBuf<uint8_t> dslabH; DevBuf<uint32_t> dovfH;   // hybrid pass (k-mer table in shared memory)
  uint64_t nwin = 0, nsl = 0; int maxS = 0, maxB = 0;
  // piling scratch
  DevBuf<dpile::Ovl> dpo; DevBuf<dpile::ReadInfo> dpr; DevBuf<uint32_t> dprid, dptile, dpbm, dprlen; DevBuf<uint64_t> dpboff; DevBuf<uint16_t> dptrace;
  DevBuf<double> dpmin, dpdiv; DevBuf<unsigned long long> dpact; DevBuf<uint32_t> dpcnt; DevBuf<uint64_t> dpblkw, dpblks;
  // vote scratch and results
  DevBuf<uint16_t> dvent; DevBuf<uint8_t> dvflag; DevBuf<uint64_t> dvblk; DevBuf<char> dvchars; DevBuf<dvote::Read> dvreads; DevBuf<dvote::Bound> dvbound;
  std::vector<dcu_segment> segs; uint64_t nchars = 0; bool results_valid = false;
  dcu_window* hwin = nullptr; uint64_t hwin_cap = 0;      // pinned host copy of the window descriptors (dcu_vote lays out the reads from it)
  unsigned int launch_seq = 0;
  uint64_t launches = 0, hard = 0, second = 0, lost = 0;     // second: windows the shared-memory pass handed on; hard: windows of the large-workspace pass; lost: beyond every capacity
  std::string err;
};

extern "C" {

const char* dcu_strerror(int code) {
  switch (code) {
    case DCU_OK: return "ok";
    case DCU_ERR_PARAM: return "invalid parameter";
    case DCU_ERR_CUDA: return "CUDA error";
    case DCU_ERR_UNSUPPORTED: return "parameter outside the range this build supports";
    case DCU_ERR_OVERFLOW: return "a window exceeded the large-workspace capacities";
    case DCU_ERR_STATE: return "call out of order";
    default: return "unknown";
  }
}
const char* dcu_last_error(dcu_ctx* ctx) { return ctx ? ctx->err.c_str() : "null ctx"; }

int dcu_create(const dcu_params* p, int device, dcu_ctx** out) {
  if (!p || !out) return DCU_ERR_PARAM;
  *out = nullptr;
  if (p->w < 8 || p->w > 59) return DCU_ERR_UNSUPPORTED;               // consensus / A window must fit 64-bit Myers words
  if (p->k_lo < 3 || p->k_hi > 14 || p->k_lo > p->k_hi) return DCU_ERR_UNSUPPORTED;
  if (p->max_ff < p->min_ff || p->min_ff < 0) return DCU_ERR_PARAM;
  if (!(p->p_i >= 0 && p->p_i < 1 && p->p_d >= 0 && p->p_d < 1)) return DCU_ERR_PARAM;
  if (!(p->est_cor >= 0 && p->est_cor <= 1)) return DCU_ERR_PARAM;     // a probability (NaN fails too): the k-mer limits are its binomial quantiles
  dcu_ctx* ctx = new (std::nothrow) dcu_ctx();
  if (!ctx) return DCU_ERR_PARAM;
  ctx->device = device; ctx->prm = *p;
  *out = ctx;
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  ctx->num_sms = prop.multiProcessorCount;
  CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CK(cudaEventCreate(&ctx->ev0)); CK(cudaEventCreate(&ctx->ev1));
  dcu_host::build_tables((int)p->w, p->p_i, p->p_d, p->est_cor, (int)p->k_lo, (int)p->k_hi, 2048, ctx->HT);
  auto& H = ctx->HT;
  CK(ctx->dDPn.ensure(H.DPn.size())); CK(ctx->dDPsq.ensure(H.DPsq.size())); CK(ctx->dVSq.ensure(H.VSq.size()));
  CK(ctx->dklim.ensure(H.klim.size())); CK(ctx->dsuplo.ensure(H.suplo.size())); CK(ctx->dsuphi.ensure(H.suphi.size()));
  CK(cudaMemcpy(ctx->dDPn.p, H.DPn.data(), H.DPn.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ctx->dDPsq.p, H.DPsq.data(), H.DPsq.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ctx->dVSq.p, H.VSq.data(), H.VSq.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ctx->dklim.p, H.klim.data(), H.klim.size() * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ctx->dsuplo.p, H.suplo.data(), H.suplo.size() * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(ctx->dsuphi.p, H.suphi.data(), H.suphi.size() * 2, cudaMemcpyHostToDevice));
  ctx->T.DPn = ctx->dDPn.p; ctx->T.DPsq = ctx->dDPsq.p; ctx->T.VSq = ctx->dVSq.p; ctx->T.klim = ctx->dklim.p;
  ctx->T.suplo = ctx->dsuplo.p; ctx->T.suphi = ctx->dsuphi.p; ctx->T.NP = H.NP; ctx->T.MS = H.MS; ctx->T.KLIMN = H.KLIMN;
  ctx->P.w = (int)p->w; ctx->P.k_lo = (int)p->k_lo; ctx->P.k_hi = (int)p->k_hi; ctx->P.minff = p->min_ff; ctx->P.maxff = p->max_ff;
  ctx->P.mincov = (int)p->min_cov; ctx->P.check = p->est_cor != 0.0; ctx->P.eminrate = p->max_err; ctx->P.defer_ff = 0;
  { const char* e = getenv("DCU_POSCACHE"); ctx->P.poscache = e ? atoi(e) : 1; }
  CK(ctx->dcnt.ensure(16));
  // First pass: the HBM build by default.  The shared-memory build (graph in shared memory, slices staged by bulk copies) is complete and
  // parity-tested but measured slower on B200 (12-16 resident warps per SM against 32: profiles/r02_summary.md); DCU_SMEM=1 selects it.
  { const char* e2 = getenv("DCU_SMEM"); ctx->use_smem = (e2 && atoi(e2)) ? 1 : 0; if (getenv("DCU_NO_SMEM") && atoi(getenv("DCU_NO_SMEM"))) ctx->use_smem = 0; }
  ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
  // (measured: 1.55 against 2.33 M windows/s for the plain HBM first pass -- the 168 KB of table arenas take the L1 the scratch data of the
  //  other stages lives on: L1 hit rate 54 % against 68 %.  Kept as DCU_HYBRID=1 for the record, profiles/r02_summary.md)
  { const char* e3 = getenv("DCU_HYBRID"); ctx->use_hybrid = e3 ? atoi(e3) : 0; }
  const char* e = getenv("DCU_BLOCKS_PER_SM");
  if (e && atoi(e) > 0) ctx->blocks_per_sm[0] = atoi(e);
  e = getenv("DCU_SYNC_GROUP");
  if (e && (atoi(e) == 1 || atoi(e) == 2 || atoi(e) == 4 || atoi(e) == 8 || atoi(e) == 16 || atoi(e) == 32)) ctx->sync_group_env = atoi(e);
  return DCU_OK;
}

void dcu_destroy(dcu_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  ctx->dDPn.release(); ctx->dDPsq.release(); ctx->dVSq.release(); ctx->dklim.release(); ctx->dsuplo.release(); ctx->dsuphi.release();
  ctx->dpacked_own.release(); ctx->dwin.release(); ctx->dsl.release(); ctx->dres.release(); ctx->dcons.release(); ctx->dops.release();
  ctx->dpo.release(); ctx->dpr.release(); ctx->dprid.release(); ctx->dptile.release(); ctx->dpbm.release(); ctx->dprlen.release();
  ctx->dpboff.release(); ctx->dptrace.release(); ctx->dpmin.release(); ctx->dpdiv.release(); ctx->dpact.release(); ctx->dpcnt.release(); ctx->dpblkw.release(); ctx->dpblks.release();
  ctx->dovf[0].release(); ctx->dovf[1].release(); ctx->dovf[2].release(); ctx->dcnt.release(); ctx->dslab[0].release(); ctx->dslab[1].release(); ctx->dslab[2].release();
  ctx->dslabH.release(); ctx->dovfH.release(); ctx->dvent.release(); ctx->dvflag.release(); ctx->dvblk.release(); ctx->dvchars.release(); ctx->dvreads.release(); ctx->dvbound.release();
  if (ctx->hwin) cudaFreeHost(ctx->hwin);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int dcu_set_reads(dcu_ctx* ctx, const uint8_t* packed, uint64_t nbytes) {
  if (!ctx || !packed) return DCU_ERR_PARAM;
  if (nbytes >= (1ull << 30)) { ctx->err = "database larger than 2^32 bases"; return DCU_ERR_UNSUPPORTED; }
  CK(cudaSetDevice(ctx->device));
  CK(ctx->dpacked_own.ensure(nbytes + 64));
  CK(cudaMemcpyAsync(ctx->dpacked_own.p, packed, nbytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->dpacked_own.p + nbytes, 0, 64, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->dpacked = ctx->dpacked_own.p; ctx->packed_bytes = nbytes; ctx->packed_padded = (nbytes + 48) & ~(uint64_t)15;
  return DCU_OK;
}
int dcu_set_reads_device(dcu_ctx* ctx, const void* dpacked, uint64_t nbytes) {
  if (!ctx || !dpacked) return DCU_ERR_PARAM;
  if (nbytes >= (1ull << 30)) { ctx->err = "database larger than 2^32 bases"; return DCU_ERR_UNSUPPORTED; }
  ctx->dpacked = (const uint8_t*)dpacked; ctx->packed_bytes = nbytes; ctx->packed_padded = nbytes & ~(uint64_t)15;     // a caller's buffer: whole 16-byte chunks inside it only
  if (((uintptr_t)dpacked & 15) != 0) ctx->packed_padded = 0;      // unaligned buffer: no staging (direct loads)
  return DCU_OK;
}

int dcu_share_reads(dcu_ctx* ctx, dcu_ctx* owner) {
  if (!ctx || !owner || ctx->device != owner->device) return DCU_ERR_PARAM;
  if (!owner->dpacked) { ctx->err = "owner holds no read database"; return DCU_ERR_STATE; }
  ctx->dpacked = owner->dpacked; ctx->packed_bytes = owner->packed_bytes; ctx->packed_padded = owner->packed_padded;
  return DCU_OK;
}

// sizes the workspaces and result buffers for a batch whose descriptors are (or will be) in ctx->dwin / ctx->dsl
static int finish_batch(dcu_ctx* ctx, int maxS, int maxB, uint64_t totS, uint64_t nwin, uint64_t nsl) {
  if (maxS < 4) maxS = 4;
  if (maxB < 64) maxB = 64;
  // windows beyond what the 16-bit indices of the kernel address (>= KLIMN slices or > 65000 bases) end as DCU_WIN_OVERFLOW in the
  // kernel's own capacity checks (load_window); they do not fail the batch
  if (maxS >= ctx->HT.KLIMN) maxS = ctx->HT.KLIMN - 1;
  if (maxB > 65000) maxB = 65000;
  ctx->maxS = maxS; ctx->maxB = maxB;
  // phase-synchronous group size: deep, homogeneous piles gain from large groups (instruction-cache locality); shallow
  // piles have a heavy tail of windows that need the filterfreq-1 pass, where waiting on the slowest warp costs more
  // than the locality brings (measured: profiles/r01_summary.md).  Results do not depend on it.
  // (round 2: with the leaner stages the whole block in lock step wins at every depth -- 10x: +25 % over free running, 20x: +25 % over groups of 8)
  (void)totS; ctx->sync_group = ctx->sync_group_env ? ctx->sync_group_env : WPB;
  for (int t = 0; t < 2; ++t) { ctx->caps[t] = dcu_host::make_caps(t, (int)ctx->prm.w, maxS, maxB); dcu::make_layout(ctx->caps[t], ctx->lay[t]); }
  { const char* e = getenv("DCU_HEAVY_NN"); if (e) ctx->caps[0].HEAVY = atoi(e); if (ctx->sync_group == 1) ctx->caps[0].HEAVY = 0; }   // free-running batches keep heavy windows in place
  CK(ctx->dwin.ensure(nwin + 1)); CK(ctx->dsl.ensure(nsl + 1)); CK(ctx->dres.ensure(nwin + 1));
  CK(ctx->dcons.ensure((nwin + 1) * DCU_CONS_STRIDE)); CK(ctx->dops.ensure((nwin + 1) * DCU_OPS_STRIDE));
  CK(ctx->dovf[0].ensure(nwin + 1)); CK(ctx->dovf[1].ensure(nwin + 1)); CK(ctx->dovf[2].ensure(nwin + 1));
  {   // shared-memory pass: as many warps per SM as the arenas of this batch's capacities allow
    ctx->capsS = dcu_host::make_caps_smem((int)ctx->prm.w, maxS, maxB); dcus::make_layout(ctx->capsS, ctx->layS);
    size_t vs_bytes = ctx->HT.VSq.size() * sizeof(unsigned long long);
    if (vs_bytes > 40 * 1024) vs_bytes = 0;
    vs_bytes = (vs_bytes + 127) & ~(size_t)127;
    const size_t avail = (size_t)ctx->smem_optin - 1024 - vs_bytes;     // static: barrier flags, mbarriers
    int wps = (int)(avail / ctx->layS.sbytes);
    if (wps > SWPB) wps = SWPB;
    { const char* e = getenv("DCU_S_WARPS"); if (e && atoi(e) > 0 && atoi(e) < wps) wps = atoi(e); }
    ctx->warpsS = wps;
  }
  {   // hybrid pass: worth it where the filter frequency 2 graph usually succeeds (deep, clean piles) and the 15-bit counts cannot overflow
    const double mean = nwin ? (double)totS / (double)nwin : 0.0;
    ctx->capsH = dcu_host::make_caps_hybrid((int)ctx->prm.w, maxS, maxB); dcuh::make_layout(ctx->capsH, ctx->layH);
    size_t vs_bytes = ctx->HT.VSq.size() * sizeof(unsigned long long);
    if (vs_bytes > 40 * 1024) vs_bytes = 0;
    vs_bytes = (vs_bytes + 127) & ~(size_t)127;
    const size_t per_block = vs_bytes + (size_t)WPB * ctx->layH.sbytes + 1536;
    const double mind = getenv("DCU_HYBRID_MIN_DEPTH") ? atof(getenv("DCU_HYBRID_MIN_DEPTH")) : 25.0;
    ctx->hybrid_ok = ctx->use_hybrid && !ctx->use_smem && ctx->prm.max_ff >= 2 && mean >= mind && maxB < 32768 && BPS * per_block <= (size_t)ctx->smem_optin + 1024 && per_block <= (size_t)ctx->smem_optin;
    CK(ctx->dovfH.ensure(nwin + 1));
  }
  ctx->nwin = nwin; ctx->nsl = nsl; ctx->results_valid = false;
  return DCU_OK;
}

int dcu_upload(dcu_ctx* ctx, const dcu_window* win, uint64_t nwin, const dcu_slice* sl, uint64_t nsl) {
  if (!ctx || (!win && nwin) || (!sl && nsl)) return DCU_ERR_PARAM;
  if (!ctx->dpacked) { ctx->err = "dcu_set_reads not called"; return DCU_ERR_STATE; }
  if (nwin >= 0xFFFFFFF0ull || nsl >= 0xFFFFFFF0ull) return DCU_ERR_UNSUPPORTED;
  CK(cudaSetDevice(ctx->device));
  // validate and size the workspaces for this batch
  int maxS = 4, maxB = 64; uint64_t totS = 0;
  const uint64_t nbases = ctx->packed_bytes * 4;
  int bad = 0;                                     // 1 range, 3 slice outside DB, 4 A window length (a slice longer than 255 bases ends its window as DCU_WIN_OVERFLOW in the kernel)
  const uint32_t wlen = ctx->prm.w, mincov = ctx->prm.min_cov;
#pragma omp parallel for schedule(static) reduction(max : maxS, maxB, bad) reduction(+ : totS)
  for (int64_t i = 0; i < (int64_t)nwin; ++i) {
    const dcu_window& W = win[i];
    if ((uint64_t)W.slice_begin + W.slice_cnt > nsl) { bad = std::max(bad, 1); continue; }
    int b = 0;
    for (uint32_t j = 0; j < W.slice_cnt; ++j) {
      const dcu_slice& s = sl[W.slice_begin + j];
      if ((uint64_t)s.gpos + s.len > nbases) bad = std::max(bad, 3);
      b += s.len;
    }
    if (W.slice_cnt && sl[W.slice_begin].len != wlen && W.slice_cnt >= mincov) bad = std::max(bad, 4);
    maxS = std::max<int>(maxS, W.slice_cnt); maxB = std::max(maxB, b); totS += W.slice_cnt;
  }
  if (bad == 1) { ctx->err = "window slice range out of bounds"; return DCU_ERR_PARAM; }
  if (bad == 3) { ctx->err = "slice outside the read database"; return DCU_ERR_PARAM; }
  if (bad == 4) { ctx->err = "slice 0 of a window must be the A window of length w"; return DCU_ERR_PARAM; }
  int rc = finish_batch(ctx, maxS, maxB, totS, nwin, nsl);
  if (rc) return rc;
  if (nwin) CK(cudaMemcpyAsync(ctx->dwin.p, win, nwin * sizeof(dcu_window), cudaMemcpyHostToDevice, ctx->stream));
  if (nsl) CK(cudaMemcpyAsync(ctx->dsl.p, sl, nsl * sizeof(dcu_slice), cudaMemcpyHostToDevice, ctx->stream));
  return DCU_OK;
}

// trace reconstruction + window / slice extraction on the device (pile_core.cuh)
int dcu_pile(dcu_ctx* ctx, const dcu_overlap* ovl, uint64_t novl, const uint16_t* trace, uint64_t ntrace, int32_t tspace,
             const uint64_t* read_boff, const uint32_t* read_len, uint64_t nreads, uint32_t advance, uint64_t maxalign, uint64_t* nwin_out, uint64_t* nsl_out) {
  if (!ctx || (!ovl && novl) || (!trace && ntrace) || !read_boff || !read_len) return DCU_ERR_PARAM;
  if (!ctx->dpacked) { ctx->err = "dcu_set_reads not called"; return DCU_ERR_STATE; }
  CK(cudaSetDevice(ctx->device));
  Laps laps("dcu_pile");
  dpile::Prep P;
  if (!dpile::prepare(ovl, novl, ntrace, tspace, ctx->prm.w, advance, nreads, read_len, P)) { ctx->err = P.err; return DCU_ERR_UNSUPPORTED; }
  laps.lap("prepare");
  int bad = 0;                                   // every B block must lie inside its read and fit the tile aligner
#pragma omp parallel for schedule(static) reduction(max : bad)
  for (int64_t i = 0; i < (int64_t)novl; ++i) {
    uint64_t b = (uint64_t)ovl[i].bbpos; int e = 0;
    for (int32_t t = 1; t < ovl[i].tlen; t += 2) { uint16_t bl = trace[ovl[i].trace_off + t]; if (bl > dpile::PILE_MAXB) e = 3; b += bl; }
    if (b > read_len[ovl[i].bread]) e = std::max(e, 2);
    if ((read_boff[ovl[i].bread] + (read_len[ovl[i].bread] + 3) / 4) > ctx->packed_bytes) e = std::max(e, 1);
    bad = std::max(bad, e);
  }
  laps.lap("validate");
  if (bad == 3) { ctx->err = "trace block longer than 256"; return DCU_ERR_UNSUPPORTED; }
  if (bad == 2) { ctx->err = "trace points run past the B read"; return DCU_ERR_PARAM; }
  if (bad == 1) { ctx->err = "read outside the packed database"; return DCU_ERR_PARAM; }
  const uint64_t nr = P.reads.size();
  dpile::Params prm; prm.tspace = tspace; prm.w = ctx->prm.w; prm.a = advance; prm.maxalign = maxalign;
  CK(ctx->dpo.ensure(novl + 1)); CK(ctx->dpr.ensure(nr + 1)); CK(ctx->dprid.ensure(nr + 1)); CK(ctx->dptile.ensure(P.ntiles + 1)); CK(ctx->dpbm.ensure(P.nbm + 1));
  CK(ctx->dprlen.ensure(nreads + 1)); CK(ctx->dpboff.ensure(nreads + 1)); CK(ctx->dptrace.ensure(ntrace + 1));
  CK(ctx->dpmin.ensure(nr + 1)); CK(ctx->dpdiv.ensure(nr + 1)); CK(ctx->dpact.ensure(novl + 1)); CK(ctx->dcnt.ensure(16));
  cudaStream_t st = ctx->stream;
  laps.lap("ensure");
  if (novl) CK(cudaMemcpyAsync(ctx->dpo.p, P.ovl.data(), novl * sizeof(dpile::Ovl), cudaMemcpyHostToDevice, st));
  if (ntrace) CK(cudaMemcpyAsync(ctx->dptrace.p, trace, ntrace * 2, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->dpboff.p, read_boff, nreads * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->dprlen.p, read_len, nreads * 4, cudaMemcpyHostToDevice, st));
  if (nr) {
    CK(cudaMemcpyAsync(ctx->dpr.p, P.reads.data(), nr * sizeof(dpile::ReadInfo), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->dprid.p, P.read_id.data(), nr * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->dpmin.p, P.minerate.data(), nr * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->dpdiv.p, P.ediv.data(), nr * 8, cudaMemcpyHostToDevice, st));
  }
  uint64_t tw = 0, ts = 0;
  unsigned int mx[2] = {4, 64};
  if (novl) {
    int* derr = (int*)(ctx->dcnt.p + 4);
    const uint64_t ncand = P.ncand, nblk = (ncand + VOTE_TPB - 1) / VOTE_TPB;
    if (nblk >= 0x7FFFFFFFull) { ctx->err = "batch too large"; return DCU_ERR_UNSUPPORTED; }
    CK(ctx->dpcnt.ensure(ncand + 1)); CK(ctx->dpblkw.ensure(nblk + 2)); CK(ctx->dpblks.ensure(nblk + 2));
    CK(cudaMemsetAsync(ctx->dcnt.p + 4, 0, 4 * sizeof(unsigned int), st));
    pile_k0<<<(unsigned)((novl + 127) / 128), 128, 0, st>>>(ctx->dpo.p, novl, ctx->dptrace.p, ctx->dptile.p);
    pile_k1<<<(unsigned)((P.ntiles + 63) / 64), 64, 0, st>>>(ctx->dpo.p, novl, P.ntiles, ctx->dpr.p, prm, ctx->dptrace.p, ctx->dptile.p, ctx->dpacked, ctx->dpboff.p, ctx->dprlen.p, ctx->dpbm.p);
    pile_k2a<<<(unsigned)((nr + 63) / 64), 64, 0, st>>>(ctx->dpr.p, nr, ctx->dpo.p, ctx->dpmin.p, ctx->dpdiv.p, ctx->dpact.p);
    if (ncand) {
      pile_k2<<<(unsigned)nblk, VOTE_TPB, 0, st>>>(ctx->dpr.p, ctx->dprid.p, (uint32_t)nr, ncand, ctx->dpo.p, prm, ctx->dpbm.p, ctx->dpboff.p, ctx->dprlen.p, ctx->dpact.p,
                                                 ctx->dpcnt.p, ctx->dpblkw.p, ctx->dpblks.p, nullptr, nullptr, derr);
      vote_kscan<<<1, VOTE_TPB, 0, st>>>(ctx->dpblkw.p, nblk);
      vote_kscan<<<1, VOTE_TPB, 0, st>>>(ctx->dpblks.p, nblk);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(&tw, ctx->dpblkw.p + nblk, 8, cudaMemcpyDeviceToHost, st));
      CK(cudaMemcpyAsync(&ts, ctx->dpblks.p + nblk, 8, cudaMemcpyDeviceToHost, st));
      laps.lap("enqueue");
      CK(cudaStreamSynchronize(st));
      laps.lap("sync1");
    }
    if (tw >= 0xFFFFFFF0ull || ts >= 0xFFFFFFF0ull) { ctx->err = "batch too large"; return DCU_ERR_UNSUPPORTED; }
    CK(ctx->dwin.ensure(tw + 1)); CK(ctx->dsl.ensure(ts + 1));
    if (tw) pile_k2<<<(unsigned)nblk, VOTE_TPB, 0, st>>>(ctx->dpr.p, ctx->dprid.p, (uint32_t)nr, ncand, ctx->dpo.p, prm, ctx->dpbm.p, ctx->dpboff.p, ctx->dprlen.p, ctx->dpact.p,
                                                       ctx->dpcnt.p, ctx->dpblkw.p, ctx->dpblks.p, (dpile::Win*)ctx->dwin.p, (dpile::Sl*)ctx->dsl.p, derr);
    unsigned int* dmx = ctx->dcnt.p + 6;
    CK(cudaMemcpyAsync(dmx, mx, sizeof(mx), cudaMemcpyHostToDevice, st));
    if (tw) pile_k3<<<(unsigned)((tw + 255) / 256), 256, 0, st>>>((const dpile::Win*)ctx->dwin.p, (const dpile::Sl*)ctx->dsl.p, tw, dmx, dmx + 1);
    CK(cudaGetLastError());
    int herr = 0;
    CK(cudaMemcpyAsync(mx, dmx, sizeof(mx), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&herr, derr, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    laps.lap("pass2+sync");
    if (herr) { ctx->err = "piling failed on the device (slice longer than 65535 bases)"; return DCU_ERR_UNSUPPORTED; }
  }
  if (nwin_out) *nwin_out = tw;
  if (nsl_out) *nsl_out = ts;
  return finish_batch(ctx, (int)mx[0], (int)mx[1], ts, tw, ts);
}

int dcu_get_windows(dcu_ctx* ctx, dcu_window* win, dcu_slice* sl) {
  if (!ctx) return DCU_ERR_PARAM;
  CK(cudaSetDevice(ctx->device));
  if (win && ctx->nwin) CK(cudaMemcpyAsync(win, ctx->dwin.p, ctx->nwin * sizeof(dcu_window), cudaMemcpyDeviceToHost, ctx->stream));
  if (sl && ctx->nsl) CK(cudaMemcpyAsync(sl, ctx->dsl.p, ctx->nsl * sizeof(dcu_slice), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return DCU_OK;
}

static void fill_args(dcu_ctx* ctx, KArgs& a, int cnt_at, int list, const uint32_t* todo, uint32_t n) {
  a.packed = ctx->dpacked; a.sl = ctx->dsl.p; a.win = ctx->dwin.p; a.res = ctx->dres.p; a.cons = ctx->dcons.p; a.ops = ctx->dops.p;
  a.todo = todo; a.n = n;
  a.ticket = ctx->dcnt.p + cnt_at; a.ovf_cnt = ctx->dcnt.p + cnt_at + 1; a.ovf_list = ctx->dovf[list].p;
  a.packed_bytes = ctx->packed_padded; a.stage = 0; a.launch_seq = ++ctx->launch_seq;
  { const char* e = getenv("DCU_SYNC_MASK"); a.sync_mask = e ? atoi(e) : 255; }
}
// HBM passes: tier 0 (first overflow pass, or the first pass when the shared-memory pass is off), tier 1 (large workspaces, free running)
static int launch_tier(dcu_ctx* ctx, int tier, const uint32_t* todo, uint32_t n) {
  int bps = ctx->blocks_per_sm[tier];
  int grid = ctx->num_sms * bps;
  int wpb = WPB;
  { const char* e = getenv("DCU_WPB"); if (e && tier == 0 && (atoi(e) == 12 || atoi(e) == 32)) { wpb = atoi(e); if (wpb == 32) { bps = 1; grid = ctx->num_sms; } } }
  size_t need_blocks = ((size_t)n + wpb - 1) / wpb;
  if ((size_t)grid > need_blocks) grid = (int)std::max<size_t>(1, need_blocks);
  CK(ctx->dslab[tier].ensure((size_t)grid * wpb * ctx->lay[tier].bytes, true));
  KArgs a;
  CK(cudaMemcpyToSymbolAsync(dcu::c_layout, &ctx->lay[tier], sizeof(dcu::Layout), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(dcu::c_cap, &ctx->caps[tier], sizeof(dcu::Caps), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(dcu::c_T, &ctx->T, sizeof(dcu::Tables), 0, cudaMemcpyHostToDevice, ctx->stream));
  {   // experimental: DCU_DEFER_FF=1 queues windows whose first filter frequency fails for the free-running second pass (DESIGN.md section 7)
    dcu::Params& P = ctx->Pl[tier];
    P = ctx->P;
    P.defer_ff = (tier == 0 && ctx->sync_group > 1 && getenv("DCU_DEFER_FF")) ? 1 : 0;
    CK(cudaMemcpyToSymbolAsync(dcu::c_P, &P, sizeof(dcu::Params), 0, cudaMemcpyHostToDevice, ctx->stream));
  }
  fill_args(ctx, a, 2 * tier, tier, todo, n);
  a.slabs = ctx->dslab[tier].p;
  size_t vs_bytes = ctx->HT.VSq.size() * sizeof(unsigned long long);
  if (vs_bytes > 40 * 1024 || getenv("DCU_VS_GLOBAL")) vs_bytes = 0;            // one copy per block (2 blocks / SM); larger tables are read from L2
  a.vs_words = (uint32_t)(vs_bytes / 8);
  a.sync_group = tier ? 1 : ctx->sync_group;       // the large-workspace pass only sees heavy-tailed windows: free running
  while (a.sync_group > 1 && wpb % a.sync_group) --a.sync_group;                       // groups must tile the block
  int pct_used = 0;
  {   // leave as much of the 228 KB as possible to L1: the kernel lives on cached scratch data (measured +5 %, profiles/r01_summary.md)
    int pct = (int)((bps * (vs_bytes + 1024) * 100 + 228 * 1024 - 1) / (228 * 1024)) + 3;
    const char* e = getenv("DCU_CARVEOUT");
    if (e) pct = atoi(e);
    CK(cudaFuncSetAttribute(dcu_window_kernel<16>, cudaFuncAttributePreferredSharedMemoryCarveout, pct > 100 ? 100 : pct));
    CK(cudaFuncSetAttribute(dcu_window_kernel<12>, cudaFuncAttributePreferredSharedMemoryCarveout, pct > 100 ? 100 : pct));
    pct_used = pct > 100 ? 100 : pct;
  }
  if (wpb == 32) { CK(cudaFuncSetAttribute(dcu_window_kernel<32, 1>, cudaFuncAttributePreferredSharedMemoryCarveout, pct_used)); dcu_window_kernel<32, 1><<<grid, 32 * 32, vs_bytes, ctx->stream>>>(a); }
  else if (wpb == 12) dcu_window_kernel<12><<<grid, 12 * 32, vs_bytes, ctx->stream>>>(a);
  else dcu_window_kernel<16><<<grid, WPB * 32, vs_bytes, ctx->stream>>>(a);
  CK(cudaGetLastError());
  ctx->launches++;
  return DCU_OK;
}
// shared-memory pass: one block of warpsS warps per SM, dynamic shared memory = VS table + warpsS arenas
static int launch_smem(dcu_ctx* ctx, uint32_t n) {
  const int wps = ctx->warpsS;
  int grid = ctx->num_sms;
  size_t need_blocks = ((size_t)n + wps - 1) / wps;
  if ((size_t)grid > need_blocks) grid = (int)std::max<size_t>(1, need_blocks);
  CK(ctx->dslab[2].ensure((size_t)grid * wps * ctx->layS.bytes, true));
  CK(cudaMemcpyToSymbolAsync(dcus::c_layout, &ctx->layS, sizeof(dcus::Layout), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(dcus::c_cap, &ctx->capsS, sizeof(dcu::Caps), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(dcus::c_T, &ctx->T, sizeof(dcu::Tables), 0, cudaMemcpyHostToDevice, ctx->stream));
  { dcu::Params P = ctx->P; P.defer_ff = 0; ctx->Pl[0] = P; CK(cudaMemcpyToSymbolAsync(dcus::c_P, &ctx->Pl[0], sizeof(dcu::Params), 0, cudaMemcpyHostToDevice, ctx->stream)); }
  KArgs a;
  fill_args(ctx, a, 8, 2, nullptr, n);
  a.slabs = ctx->dslab[2].p;
  size_t vs_bytes = ctx->HT.VSq.size() * sizeof(unsigned long long);
  if (vs_bytes > 40 * 1024) vs_bytes = 0;
  a.vs_words = (uint32_t)(vs_bytes / 8);
  vs_bytes = (vs_bytes + 127) & ~(size_t)127;
  { int g = ctx->sync_group_env ? ctx->sync_group_env : 4; while (g > 1 && wps % g) --g; a.sync_group = g; }      // groups must tile the block (measured: 4 > 6 > 12 > 2 > 1)
  { const char* e = getenv("DCU_STAGE"); a.stage = e ? atoi(e) : 1; }
  const size_t dyn = vs_bytes + (size_t)wps * ctx->layS.sbytes;
  CK(cudaFuncSetAttribute(dcus_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  dcus_window_kernel<<<grid, wps * 32, dyn, ctx->stream>>>(a);
  CK(cudaGetLastError());
  ctx->launches++;
  return DCU_OK;
}

// hybrid pass: grid and block shape of the HBM first pass, dynamic shared memory = VS table + 16 k-mer table arenas
static int launch_hybrid(dcu_ctx* ctx, uint32_t n) {
  int grid = ctx->num_sms * BPS;
  size_t need_blocks = ((size_t)n + WPB - 1) / WPB;
  if ((size_t)grid > need_blocks) grid = (int)std::max<size_t>(1, need_blocks);
  CK(ctx->dslabH.ensure((size_t)grid * WPB * ctx->layH.bytes, true));
  CK(cudaMemcpyToSymbolAsync(dcuh::c_layout, &ctx->layH, sizeof(dcuh::Layout), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(dcuh::c_cap, &ctx->capsH, sizeof(dcu::Caps), 0, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyToSymbolAsync(dcuh::c_T, &ctx->T, sizeof(dcu::Tables), 0, cudaMemcpyHostToDevice, ctx->stream));
  { dcu::Params P = ctx->P; P.defer_ff = 0; ctx->Pl[0] = P; CK(cudaMemcpyToSymbolAsync(dcuh::c_P, &ctx->Pl[0], sizeof(dcu::Params), 0, cudaMemcpyHostToDevice, ctx->stream)); }
  KArgs a;
  fill_args(ctx, a, 12, 0, nullptr, n);
  a.ovf_list = ctx->dovfH.p;
  a.slabs = ctx->dslabH.p;
  size_t vs_bytes = ctx->HT.VSq.size() * sizeof(unsigned long long);
  if (vs_bytes > 40 * 1024) vs_bytes = 0;
  a.vs_words = (uint32_t)(vs_bytes / 8);
  vs_bytes = (vs_bytes + 127) & ~(size_t)127;
  a.sync_group = ctx->sync_group;
  while (a.sync_group > 1 && WPB % a.sync_group) --a.sync_group;
  const size_t dyn = vs_bytes + (size_t)WPB * ctx->layH.sbytes;
  CK(cudaFuncSetAttribute(dcuh_window_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  CK(cudaFuncSetAttribute(dcuh_window_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  dcuh_window_kernel<<<grid, WPB * 32, dyn, ctx->stream>>>(a);
  CK(cudaGetLastError());
  ctx->launches++;
  return DCU_OK;
}

int dcu_launch(dcu_ctx* ctx, float* kernel_ms) {
  if (!ctx) return DCU_ERR_PARAM;
  CK(cudaSetDevice(ctx->device));
  ctx->launches = 0; ctx->hard = 0; ctx->second = 0; ctx->lost = 0;
  if (kernel_ms) *kernel_ms = 0.f;
  if (!ctx->nwin) return DCU_OK;
  std::lock_guard<std::mutex> pass_lock(g_window_pass_lock[ctx->device & 63]);
  CK(cudaMemsetAsync(ctx->dcnt.p, 0, 4 * sizeof(unsigned int), ctx->stream));
  CK(cudaMemsetAsync(ctx->dcnt.p + 8, 0, 8 * sizeof(unsigned int), ctx->stream));
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  unsigned int cnt[2];
  const uint32_t* todo = nullptr; uint32_t n = (uint32_t)ctx->nwin;
  if (ctx->use_smem && ctx->warpsS >= 2) {           // pass 1: shared-memory workspaces
    int rc = launch_smem(ctx, n);
    if (rc) return rc;
    CK(cudaMemcpyAsync(cnt, ctx->dcnt.p + 8, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->second = cnt[1]; todo = ctx->dovf[2].p; n = cnt[1];
  } else if (ctx->hybrid_ok) {                       // pass 1: k-mer table in shared memory, 32 warps per SM
    int rc = launch_hybrid(ctx, n);
    if (rc) return rc;
    CK(cudaMemcpyAsync(cnt, ctx->dcnt.p + 12, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->second = cnt[1]; todo = ctx->dovfH.p; n = cnt[1];
  }
  if (n) {                                           // HBM workspaces, first-pass capacities
    int rc = launch_tier(ctx, 0, todo, n);
    if (rc) return rc;
    CK(cudaMemcpyAsync(cnt, ctx->dcnt.p, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    n = cnt[1];
    if (n) {                                         // large workspaces
      ctx->hard = n;
      rc = launch_tier(ctx, 1, ctx->dovf[0].p, n);
      if (rc) return rc;
      CK(cudaMemcpyAsync(cnt, ctx->dcnt.p + 2, sizeof(cnt), cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      if (cnt[1]) {
        // beyond every capacity of this build: the windows keep status DCU_WIN_OVERFLOW (the caller treats them like failed windows, as the
        // reference swallows a read's exception, src/daccord.cpp:2466-2478); the batch itself is not an error
        uint32_t wi = 0; dcu::Result r; memset(&r, 0, sizeof(r));
        CK(cudaMemcpy(&wi, ctx->dovf[1].p, sizeof(wi), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(&r, ctx->dres.p + wi, sizeof(r), cudaMemcpyDeviceToHost));
        char b[192]; snprintf(b, sizeof b, "%u windows exceeded the large-workspace capacities (first: window %u, capacity code %u)", cnt[1], wi, r.err);
        ctx->err = b; ctx->lost = cnt[1];
      }
    }
  }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaEventSynchronize(ctx->ev1));
  if (kernel_ms) CK(cudaEventElapsedTime(kernel_ms, ctx->ev0, ctx->ev1));
  ctx->results_valid = true;
  return DCU_OK;
}

int dcu_download(dcu_ctx* ctx, dcu_result* res, uint8_t* cons, uint8_t* ops) {
  if (!ctx) return DCU_ERR_PARAM;
  CK(cudaSetDevice(ctx->device));
  if (!ctx->nwin) return DCU_OK;
  if (res) CK(cudaMemcpyAsync(res, ctx->dres.p, ctx->nwin * sizeof(dcu_result), cudaMemcpyDeviceToHost, ctx->stream));
  if (cons) CK(cudaMemcpyAsync(cons, ctx->dcons.p, ctx->nwin * DCU_CONS_STRIDE, cudaMemcpyDeviceToHost, ctx->stream));
  if (ops) CK(cudaMemcpyAsync(ops, ctx->dops.p, ctx->nwin * DCU_OPS_STRIDE, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return DCU_OK;
}

// pile vote of the resident batch on the device (vote_core.cuh)
int dcu_vote(dcu_ctx* ctx, int producefull, uint64_t minlen, const uint64_t* read_boff, const uint32_t* read_len, uint64_t nreads, uint64_t* nseg, uint64_t* nchars) {
  if (!ctx) return DCU_ERR_PARAM;
  CK(cudaSetDevice(ctx->device));
  ctx->segs.clear(); ctx->nchars = 0;
  if (nseg) *nseg = 0;
  if (nchars) *nchars = 0;
  if (!ctx->nwin) return DCU_OK;
  if (!ctx->results_valid) { ctx->err = "dcu_vote needs the results of dcu_launch"; return DCU_ERR_STATE; }
  if (ctx->prm.w > 127) { ctx->err = "vote tables hold w <= 127"; return DCU_ERR_UNSUPPORTED; }
  cudaStream_t st = ctx->stream;
  const uint64_t nwin = ctx->nwin;
  Laps laps("dcu_vote");
  if (nwin > ctx->hwin_cap) {                        // pinned staging of the window descriptors (a pageable target costs 30 ms per 84 MB instead of 4)
    if (ctx->hwin) cudaFreeHost(ctx->hwin);
    ctx->hwin = nullptr; ctx->hwin_cap = 0;
    CK(cudaMallocHost((void**)&ctx->hwin, (nwin + nwin / 4 + 16) * sizeof(dcu_window)));
    ctx->hwin_cap = nwin + nwin / 4 + 16;
  }
  dcu_window* const hwin_p = ctx->hwin;
  CK(cudaMemcpyAsync(hwin_p, ctx->dwin.p, nwin * sizeof(dcu_window), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  laps.lap("windows_d2h");
  dvote::Layout L;
  if (!dvote::layout_reads(hwin_p, nwin, ctx->prm.w, producefull != 0, read_boff, read_len, nreads, L)) { ctx->err = L.err; return DCU_ERR_PARAM; }
  laps.lap("layout");
  if (producefull) for (auto& R : L.reads) if (R.boff + (R.rlen + 3) / 4 > ctx->packed_bytes) { ctx->err = "read outside the packed database"; return DCU_ERR_PARAM; }
  const uint32_t nr = (uint32_t)L.reads.size();
  const uint64_t npos = L.npos, nblk = (npos + VOTE_TPB - 1) / VOTE_TPB;
  if (nblk >= 0x7FFFFFFFull) { ctx->err = "batch too large for the vote"; return DCU_ERR_UNSUPPORTED; }
  const uint64_t bound_cap = 2 * (nwin + nr) + 16;
  CK(ctx->dvent.ensure(nwin * (ctx->prm.w + 1))); CK(ctx->dvflag.ensure(npos + 1)); CK(ctx->dvblk.ensure(nblk + 2)); CK(ctx->dvreads.ensure(nr + 1));
  CK(ctx->dvbound.ensure(bound_cap)); CK(ctx->dcnt.ensure(16));
  CK(cudaMemcpyAsync(ctx->dvreads.p, L.reads.data(), nr * sizeof(dvote::Read), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(ctx->dcnt.p + 4, 0, 4 * sizeof(unsigned int), st));
  int* derr = (int*)(ctx->dcnt.p + 4); unsigned int* dnb = ctx->dcnt.p + 5;
  dvote::Params vp; vp.w = ctx->prm.w; vp.cons_stride = DCU_CONS_STRIDE; vp.ops_stride = DCU_OPS_STRIDE; vp.producefull = producefull ? 1 : 0;
  dvote::Ctx vc; vc.win = (const dvote::Win*)ctx->dwin.p; vc.res = (const dvote::Res*)ctx->dres.p; vc.cons = ctx->dcons.p; vc.ent = ctx->dvent.p; vc.packed = ctx->dpacked; vc.P = vp;
  vote_k0<<<(unsigned)((nwin + 255) / 256), 256, 0, st>>>((const dvote::Res*)ctx->dres.p, ctx->dops.p, nwin, vp, ctx->dvent.p, derr);
  vote_k1<<<(unsigned)nblk, VOTE_TPB, 0, st>>>(vc, ctx->dvreads.p, nr, npos, ctx->dvflag.p, ctx->dvblk.p, nullptr, nullptr, nullptr, 0u);
  vote_kscan<<<1, VOTE_TPB, 0, st>>>(ctx->dvblk.p, nblk);
  CK(cudaGetLastError());
  uint64_t total = 0; int herr = 0;
  CK(cudaMemcpyAsync(&total, ctx->dvblk.p + nblk, 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&herr, derr, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  laps.lap("count_pass");
  if (herr) { ctx->err = "a placement trace does not cover its window"; return DCU_ERR_STATE; }
  CK(ctx->dvchars.ensure(total + 1));
  vote_k1<<<(unsigned)nblk, VOTE_TPB, 0, st>>>(vc, ctx->dvreads.p, nr, npos, ctx->dvflag.p, ctx->dvblk.p, ctx->dvchars.p, ctx->dvbound.p, dnb, (unsigned int)bound_cap);
  CK(cudaGetLastError());
  unsigned int nb = 0;
  CK(cudaMemcpyAsync(&nb, dnb, 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  if (nb > bound_cap) { ctx->err = "run boundary list overflow"; return DCU_ERR_OVERFLOW; }
  std::vector<dvote::Bound> hb(nb);
  if (nb) CK(cudaMemcpyAsync(hb.data(), ctx->dvbound.p, nb * sizeof(dvote::Bound), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  laps.lap("fill_pass");
  std::string perr;
  if (!dvote::pair_bounds(hb, L, producefull != 0, minlen, ctx->segs, perr)) { ctx->err = perr; return DCU_ERR_STATE; }
  laps.lap("pair_bounds");
  ctx->nchars = total; ctx->launches += 4;
  if (nseg) *nseg = ctx->segs.size();
  if (nchars) *nchars = total;
  return DCU_OK;
}
int dcu_get_corrected(dcu_ctx* ctx, dcu_segment* seg, char* chars) {
  if (!ctx) return DCU_ERR_PARAM;
  CK(cudaSetDevice(ctx->device));
  if (seg && !ctx->segs.empty()) memcpy(seg, ctx->segs.data(), ctx->segs.size() * sizeof(dcu_segment));
  if (chars && ctx->nchars) { CK(cudaMemcpyAsync(chars, ctx->dvchars.p, ctx->nchars, cudaMemcpyDeviceToHost, ctx->stream)); CK(cudaStreamSynchronize(ctx->stream)); }
  return DCU_OK;
}

int dcu_run(dcu_ctx* ctx, const dcu_window* win, uint64_t nwin, const dcu_slice* sl, uint64_t nsl, dcu_result* res, uint8_t* cons, uint8_t* ops) {
  int rc = dcu_upload(ctx, win, nwin, sl, nsl);
  if (rc) return rc;
  int rl = dcu_launch(ctx, nullptr);
  if (rl && rl != DCU_ERR_OVERFLOW) return rl;
  rc = dcu_download(ctx, res, cons, ops);
  return rc ? rc : rl;
}

int dcu_last_stats(dcu_ctx* ctx, uint64_t* launches, uint64_t* hard_windows) {
  if (!ctx) return DCU_ERR_PARAM;
  if (launches) *launches = ctx->launches;
  if (hard_windows) *hard_windows = ctx->hard;
  return DCU_OK;
}
int dcu_last_stats2(dcu_ctx* ctx, uint64_t* second_pass_windows, uint64_t* lost_windows, uint32_t* smem_warps, uint32_t* smem_bytes_per_warp) {
  if (!ctx) return DCU_ERR_PARAM;
  if (second_pass_windows) *second_pass_windows = ctx->second;
  if (lost_windows) *lost_windows = ctx->lost;
  const bool smem = ctx->use_smem && ctx->warpsS >= 2;
  if (smem_warps) *smem_warps = smem ? (uint32_t)ctx->warpsS : (ctx->hybrid_ok ? (uint32_t)(WPB * BPS) : 0u);
  if (smem_bytes_per_warp) *smem_bytes_per_warp = smem ? ctx->layS.sbytes : (ctx->hybrid_ok ? ctx->layH.sbytes : 0u);
  return DCU_OK;
}

// the tables as the kernel reads them: copied back from the device buffers, not the host copy they were uploaded from
int64_t dcu_get_tables(dcu_ctx* ctx, int which, double* out, int64_t cap) {
  if (!ctx) return -1;
  const auto& H = ctx->HT;
  std::vector<double> DPn(H.DPn.size()), DPsq(H.DPsq.size());
  std::vector<unsigned long long> VSq(H.VSq.size()), klim(H.klim.size());
  std::vector<uint16_t> suplo(H.suplo.size()), suphi(H.suphi.size());
  if (cudaSetDevice(ctx->device) != cudaSuccess) return -1;
  for (auto c : {cudaMemcpy(DPn.data(), ctx->dDPn.p, DPn.size() * 8, cudaMemcpyDeviceToHost), cudaMemcpy(DPsq.data(), ctx->dDPsq.p, DPsq.size() * 8, cudaMemcpyDeviceToHost),
                 cudaMemcpy(VSq.data(), ctx->dVSq.p, VSq.size() * 8, cudaMemcpyDeviceToHost), cudaMemcpy(klim.data(), ctx->dklim.p, klim.size() * 8, cudaMemcpyDeviceToHost),
                 cudaMemcpy(suplo.data(), ctx->dsuplo.p, suplo.size() * 2, cudaMemcpyDeviceToHost), cudaMemcpy(suphi.data(), ctx->dsuphi.p, suphi.size() * 2, cudaMemcpyDeviceToHost)})
    if (c != cudaSuccess) { ctx->err = std::string("dcu_get_tables: ") + cudaGetErrorString(c); return -1; }
  std::vector<double> v;
  if (which == 0) v = DPn; else if (which == 1) v = DPsq;
  else if (which == 2) { for (int l = 0; l < H.NP; ++l) for (int q = 0; q < H.MS; ++q) v.push_back((double)VSq[(size_t)q * H.NP + l]); }
  else if (which == 3) for (int i = 0; i < H.MS; ++i) { v.push_back(suplo[i]); v.push_back(suphi[i]); }
  else if (which == 4) for (auto x : klim) v.push_back((double)x);
  else if (which == 5) { v.push_back(H.NP); v.push_back(H.MS); v.push_back(H.KLIMN); }
  if (out && (int64_t)v.size() <= cap) memcpy(out, v.data(), v.size() * sizeof(double));
  return (int64_t)v.size();
}

}  // extern "C"
