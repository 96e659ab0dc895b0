// cse_mid.cuh -- the level loop for frontiers of some thousand to half a million nodes per round.
// Included by cse.cu after its shared definitions (CseArgs, CseDeviceState, grid_barrier, cse_step) and
// cse_slots.cuh (warp_slot_store).
//
// Why.  A round of this size moves a few hundred kilobytes: what it costs is the chain of dependent trips to L2 / DRAM
// and the grid-wide synchronisations on it.  cse_wide_kernel pays ~10 us per round whatever the size (counts -> nodes
// -> rank words -> tile aggregates -> chained scan -> stores -> grid barrier); cse_slots_kernel needs three grid
// barriers per round for its distributed scans.
//
// How.  The slot layout of cse_slots.cuh (a chunk of 32 / 64 / 128 nodes writes its zero-children, its one-children and its
// emitted words into slots it owns, so no output position depends on another warp) with the scans made REDUNDANT:
// a round's directory is a byte per slot -- at most 8 K slots here -- so after the single grid barrier of a round
// every CTA reads the whole directory (one 16-byte load per thread), scans it in shared memory and knows what every
// other CTA knows: level sizes, the slot and offset of every frontier position, the place of every chunk's words in
// its stream.  Chain per round: barrier -> directory -> nodes -> rank words -> stores.  The words of round r are moved
// from their E-slots to the stream buffers during round r + 1 (their prefix is part of that round's scan).
//
// The kernel is entered from the flat layout (the first round reads a.fs / fa / fb directly) and writes the flat
// layout back when it leaves (frontier too large / small enough for the cluster kernels / batch full / done).
#pragma once

namespace bce {

constexpr int MD_THREADS = 512, MD_WARPS = MD_THREADS / 32;
// One thread scans 16 slots and 8 chunks: 512 threads cover 8192 slots (levels start at multiples of 16) and 4096
// chunk numbers (levels start at multiples of 8) in ONE block scan.
constexpr uint32_t MD_SLOTS = 16 * MD_THREADS;            // slot numbers per round
constexpr uint32_t MD_TCAP = 8 * MD_THREADS;              // chunk numbers per round
constexpr uint32_t MD_MAX_CHUNKS = MD_TCAP - 8 * 8;       // chunks a round may have (2 slots each + padding fit MD_SLOTS)
constexpr int MD_MAX_ITEMS = 4;                           // nodes per lane of the largest instance
// Instances differ in the nodes a lane holds (chunk = 32 * ITEMS nodes): a warp alone on its scheduler issues an
// instruction every few cycles, so the fewer nodes a round has, the thinner it is spread (ITEMS = 1 up to ~100 K nodes).
constexpr unsigned long long mid_max_nodes(int items) { return (unsigned long long)(MD_MAX_CHUNKS - 8) * 32u * items; }
constexpr size_t MD_PLACES = size_t(MD_SLOTS) * 32 * MD_MAX_ITEMS;   // places of one node array (sized for the largest instance)

struct MidArgs {                                          // (one base pointer each: indexing by parity is arithmetic)
  uint32_t* arena;        // [parity][position | x0 | x1][MD_PLACES]: slot number * chunk size + place
  uint8_t* cnt;           // [parity][MD_SLOTS]: nodes in every slot
  uint32_t* eslot;        // [parity][MD_TCAP * 32 * MD_MAX_ITEMS * EW]: E-slots, chunk number * chunk size * EW
  uint16_t* ecnt;         // [parity][MD_TCAP]: words in them
};

// The directory tables are written 16 (8) consecutive entries per thread and read 32 consecutive entries per warp:
// entry c lives at (c mod 16) * 513 + c / 16, which keeps both patterns (nearly) free of bank conflicts.
__device__ __forceinline__ uint32_t mid_pidx(uint32_t c) { return (c & 15u) * (MD_THREADS + 1u) + (c >> 4); }
__device__ __forceinline__ uint32_t mid_eidx(uint32_t t) { return (t & 7u) * (MD_THREADS + 1u) + (t >> 3); }

struct MidShared {
  uint32_t P[16 * (MD_THREADS + 1)];   // [mid_pidx(c)] nodes of the level before slot c (a level's slots are consecutive)
  uint32_t PE[8 * (MD_THREADS + 1)];   // [mid_eidx(t)] words of the level before the E-slot of chunk t (previous round)
  uint16_t start[MD_SLOTS];        // [doff[l] + q] = slot holding position q * chunk size of level l
  uint64_t ex[MD_THREADS + 1];     // exclusive scan over the threads: low = nodes, high = words (read through mid_ex)
  uint32_t ex_valid;               // threads (a multiple of 32) whose ex[] entry was written this round; the others' = total
  uint64_t scan[MD_WARPS];
  uint32_t n[8], nz[8];            // this round's frontier: nodes per level, of which zero-children
  uint32_t doff[9];                // first slot number of every level (parity cur); the level has 2 * sz[l] slots
  uint32_t sz[8];                  // Z-slots (= O-slots) of every level = chunks of the level before, last round
  uint32_t nch[8], tfirst[9];      // this round's chunks per level, first chunk number (multiple of 8)
  uint32_t pnch[8], ptfirst[9];    // the same for the previous round (whose words are still in E-slots)
  uint32_t ndoff[9];               // slot numbering of the next round
  unsigned long long emitted[8];   // words in every stream buffer, E-slots of the previous round included
  unsigned long long ebase[8];     // ... where the previous round's words start
  uint32_t decision;
};

__device__ __forceinline__ uint64_t mid_ex(const MidShared& sh, uint32_t i) { return sh.ex[i < max(sh.ex_valid, 32u) ? i : MD_THREADS]; }

// slot and offset of the ITEMS positions a lane holds in chunk q of level l, from the shared directory
template <int ITEMS>
__device__ __forceinline__ void mid_locate(const MidShared& sh, int l, uint32_t q, uint32_t gend, unsigned lane,
                                           const uint32_t (&g)[ITEMS], uint32_t (&at)[ITEMS]) {
  constexpr uint32_t CH = 32u * ITEMS;
  const uint32_t first = sh.doff[l], last = first + 2u * sh.sz[l];      // the level's slot numbers
  uint32_t base = sh.start[first + q];
  uint32_t c[ITEMS], pc[ITEMS];
  const uint32_t p0 = sh.P[mid_pidx(base)];
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) { c[j] = base; pc[j] = p0; }
  for (;;) {                                                            // windows of 32 following slots (one is the rule)
    const uint32_t e = base + 1u + lane;
    const uint32_t pwv = e < last ? sh.P[mid_pidx(e)] : 0xFFFFFFFFu;
    const unsigned le = __ballot_sync(0xffffffffu, pwv < gend);         // slots that start inside the chunk
    const int nle = __popc(le);                                         // P ascends: they are the first nle lanes
    for (int i = 0; i < nle; ++i) {
      const uint32_t pv = __shfl_sync(0xffffffffu, pwv, i);
#pragma unroll
      for (int j = 0; j < ITEMS; ++j)
        if (pv <= g[j]) { c[j] = base + 1u + i; pc[j] = pv; }
    }
    if (nle < 32) break;
    base += 32u;
  }
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) at[j] = c[j] * CH + (g[j] - pc[j]);
}

#ifdef BCE_GPU_EXPERIMENTS
#define MID_STAMP(i) do { if (blockIdx.x == 0 && tid == 0) { const long long now_ = clock64(); S->prof[i] += (unsigned long long)(now_ - stamp_); stamp_ = now_; } } while (0)
#else
#define MID_STAMP(i) do { } while (0)
#endif

template <int EW, int ITEMS>
__global__ void __launch_bounds__(MD_THREADS, 1) cse_mid_kernel(CseArgs a, MidArgs ma) {
  constexpr uint32_t CH = 32u * ITEMS;                // nodes per chunk = places per slot
  constexpr size_t ESLOT = size_t(32) * MD_MAX_ITEMS * EW;   // words set aside per E-slot
  extern __shared__ __align__(16) unsigned char mid_smem[];
  MidShared& sh = *reinterpret_cast<MidShared*>(mid_smem);
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned lt_mask = (1u << lane) - 1u;
  CseDeviceState* S = a.st;
  const uint32_t G = gridDim.x;
  uint32_t round = vol_load(&S->round);
  unsigned long long barrier_no = vol_load64(&S->barriers);
  if (blockIdx.x == 0 && tid == 0) S->status = kCseRunning;
  bool from_flat = true;                              // the frontier of this round is in the flat layout
  unsigned long long visits = 0, peak = 0;
#ifdef BCE_GPU_EXPERIMENTS
  long long stamp_ = clock64();
#endif

  if (tid < 8) {
    const int par = round & 1;
    const uint32_t cz = vol_load(&S->cnt[par][tid][0]), co = vol_load(&S->cnt[par][tid][1]);
    sh.n[tid] = cz + co;
    sh.nz[tid] = cz;
    sh.sz[tid] = 0;
    sh.pnch[tid] = 0;
    sh.emitted[tid] = sh.ebase[tid] = vol_load64(&S->emitted[par][tid]);
  }
  if (tid < 9) { sh.doff[tid] = 0; sh.ptfirst[tid] = 0; }
  if (tid == 0) sh.ex_valid = 0;
  __syncthreads();

  for (;;) {
    const int cur = round & 1, nxt = cur ^ 1;
    // ---- directory of this round (written by the previous one): one scan, the same in every CTA -----------------
    uint32_t cb[4] = {0, 0, 0, 0};                    // counts of this thread's 16 slots, a byte each; beyond the level's: 0
    uint32_t eb[4] = {0, 0, 0, 0};                    // word counts of its 8 chunks of the previous round, 16 bits each
    if (!from_flat) {
      // (both loads leave at once, before anything is known about what they cover: the arrays are MD_SLOTS / MD_TCAP long)
      const uint4 vc = __ldcg(reinterpret_cast<const uint4*>(ma.cnt + size_t(cur) * MD_SLOTS) + tid);
      const uint4 ve = __ldcg(reinterpret_cast<const uint4*>(ma.ecnt + size_t(nxt) * MD_TCAP) + tid);   // E-slots of round - 1: buffer (round - 1) & 1
      const uint32_t s0 = tid * 16u;                  // this thread's 16 slots ...
      int L = 0;
#pragma unroll
      for (int k = 1; k < 8; ++k) L += s0 >= sh.doff[k] ? 1 : 0;
      const uint32_t lvl_first = sh.doff[L], lvl_end = lvl_first + 2u * sh.sz[L];
      if (s0 < lvl_end) {
        cb[0] = vc.x; cb[1] = vc.y; cb[2] = vc.z; cb[3] = vc.w;
        const uint32_t valid = lvl_end - s0;
#pragma unroll
        for (int w = 0; w < 4; ++w)
          if (valid < 4u * w + 4u) cb[w] &= valid > 4u * w ? (1u << (8u * (valid - 4u * w))) - 1u : 0u;
      }
      const uint32_t csum = __dp4a(cb[0], 0x01010101u, __dp4a(cb[1], 0x01010101u, __dp4a(cb[2], 0x01010101u, __dp4a(cb[3], 0x01010101u, 0u))));
      const uint32_t t0 = tid * 8u;                   // ... and 8 chunks of the previous round
      int LE = 0;
#pragma unroll
      for (int k = 1; k < 8; ++k) LE += t0 >= sh.ptfirst[k] ? 1 : 0;
      const uint32_t e_first = sh.ptfirst[LE], e_end = e_first + sh.pnch[LE];
      if (t0 < e_end) {
        eb[0] = ve.x; eb[1] = ve.y; eb[2] = ve.z; eb[3] = ve.w;
        const uint32_t valid = e_end - t0;
#pragma unroll
        for (int w = 0; w < 4; ++w)
          if (valid < 2u * w + 2u) eb[w] &= valid > 2u * w ? 0xFFFFu : 0u;
      }
      uint32_t esum = 0;
#pragma unroll
      for (int w = 0; w < 4; ++w) esum += (eb[w] & 0xFFFFu) + (eb[w] >> 16);
      // warps whose slots and chunks all lie beyond this round's hold zeros: they skip the scan, and their threads'
      // entries of ex[] read as the total (mid_ex)
      uint64_t tot;
      const uint64_t excl = block_exclusive_scan_sparse<uint64_t, MD_THREADS>((uint64_t(esum) << 32) | csum, sh.scan, tot,
                                                                             warp == 0 || tid < sh.ex_valid);
      if (warp == 0 || tid < sh.ex_valid) sh.ex[tid] = excl;
      if (tid == 0) sh.ex[MD_THREADS] = tot;
      __syncthreads();
      // (the plan below needs only ex[]: the last warp makes it -- its slots are beyond those of all but the widest
      //  rounds -- while the others write the tables)
    }
    MID_STAMP(0);

    // ---- plan of this round: lanes 0..7 of the last warp hold a level each; every CTA derives the same plan ------
    if (warp == MD_WARPS - 1) {
      const int l = lane & 7;
      uint32_t nl = sh.n[l], nzl = sh.nz[l];
      unsigned long long em = sh.emitted[l];
      if (!from_flat) {
        nl = uint32_t(mid_ex(sh, sh.doff[l + 1] / 16u)) - uint32_t(mid_ex(sh, sh.doff[l] / 16u));
        nzl = 0;                                      // (set by the thread that scans the first O-slot, below)
        const uint32_t words = uint32_t(mid_ex(sh, sh.ptfirst[l + 1] / 8u) >> 32) - uint32_t(mid_ex(sh, sh.ptfirst[l] / 8u) >> 32);
        if (lane < 8) sh.ebase[l] = em;               // the previous round's words start here ...
        em += words;                                  // ... and this round's behind them
      }
      const uint32_t nch = (nl + CH - 1) / CH;
      const uint32_t tpad = (nch + 7u) & ~7u;                                   // chunk numbers of the level
      const uint32_t spad = (2u * __shfl_sync(0xffffffffu, nch, (lane + 7) & 7) + 15u) & ~15u;   // slots of the level, next round
      uint32_t tin = tpad, sin = spad;                                          // inclusive scans over the 8 levels
#pragma unroll
      for (int d = 1; d < 8; d <<= 1) {
        const uint32_t o1 = __shfl_up_sync(0xffffffffu, tin, d), o2 = __shfl_up_sync(0xffffffffu, sin, d);
        if (l >= d) { tin += o1; sin += o2; }
      }
      unsigned long long ecap_l = 0, esoft_l = 0;     // (selected, not indexed: the arguments stay in the constant bank)
#pragma unroll
      for (int j = 0; j < 8; ++j) if (l == j) { ecap_l = a.ecap[j]; esoft_l = a.esoft[j]; }
      const bool drain = must_drain(em, nl, max_words(a), ecap_l, esoft_l);
      const unsigned m8 = 0xFFu;
      const bool any_drain = (__ballot_sync(0xffffffffu, drain) & m8) != 0;
      const bool too_wide = (__ballot_sync(0xffffffffu, nl > a.cap) & m8) != 0;
      uint32_t widest = nl;
      unsigned long long nodes = nl;
#pragma unroll
      for (int d = 1; d < 8; d <<= 1) {
        widest = max(widest, __shfl_xor_sync(0xffffffffu, widest, d));
        nodes += __shfl_xor_sync(0xffffffffu, nodes, d);
      }
      const uint32_t T = __shfl_sync(0xffffffffu, tin, 7), D = __shfl_sync(0xffffffffu, sin, 7);
      if (lane < 8) {
        sh.n[l] = nl; sh.emitted[l] = em;
        if (from_flat || sh.sz[l] == 0) sh.nz[l] = nzl;
        sh.nch[l] = nch;
        sh.tfirst[l] = tin - tpad;
        sh.ndoff[l] = sin - spad;
        if (l == 7) { sh.tfirst[8] = T; sh.ndoff[8] = D; }
      }
      if (lane == 0) {
        sh.decision = round_status(nodes, round, a.round_limit, too_wide, a.use_narrow && widest <= a.narrow_enter,
                                   nodes > a.max_nodes || nodes < a.min_nodes || T > MD_TCAP || D > MD_SLOTS, any_drain);
        if (sh.decision == kCseRunning) { visits += nodes; peak = max(peak, nodes); }
      }
    }
    if (!from_flat) {
      // nodes before every slot inside its level; the slot in which every chunk of this round starts
      const uint32_t s0 = tid * 16u, t0 = tid * 8u;
      int L = 0, LE = 0;
#pragma unroll
      for (int k = 1; k < 8; ++k) { L += s0 >= sh.doff[k] ? 1 : 0; LE += t0 >= sh.ptfirst[k] ? 1 : 0; }
      const uint32_t lvl_first = sh.doff[L], first_o = lvl_first + sh.sz[L];
      const uint64_t excl = mid_ex(sh, tid);
      if (s0 < lvl_first + 2u * sh.sz[L]) {           // (entries beyond a level's slots are never read)
        uint32_t run = uint32_t(excl) - uint32_t(mid_ex(sh, lvl_first / 16u));
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const uint32_t ck = (cb[k >> 2] >> (8 * (k & 3))) & 255u;
          sh.P[k * (MD_THREADS + 1) + tid] = run;     // = mid_pidx(s0 + k)
          if (s0 + k == first_o) sh.nz[L] = run;      // nodes before the first O-slot
          if (ck) {                                   // the slot holds positions [run, run + ck): at most one chunk starts in it
            const uint32_t qn = (run + CH - 1) / CH;
            if (qn * CH < run + ck) sh.start[lvl_first + qn] = uint16_t(s0 + k);
          }
          run += ck;
        }
      }
      if (t0 < sh.ptfirst[LE] + sh.pnch[LE]) {
        uint32_t erun = uint32_t(excl >> 32) - uint32_t(mid_ex(sh, sh.ptfirst[LE] / 8u) >> 32);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          sh.PE[k * (MD_THREADS + 1) + tid] = erun;   // = mid_eidx(t0 + k)
          erun += (eb[k >> 1] >> (16 * (k & 1))) & 0xFFFFu;
        }
      }
    }
    __syncthreads();
    const uint32_t decision = sh.decision;
    MID_STAMP(1);

    // the words of the previous round go from their E-slots to their streams (their places are known now); the warps
    // take them in the opposite order of this round's chunks, so that in thin rounds other warps do it
    auto move_words = [&]() {
      const uint32_t pT = sh.ptfirst[8];
      for (uint32_t t = (MD_WARPS - 1u - warp) * G + blockIdx.x; t < pT; t += MD_WARPS * G) {
        int L = 0;
#pragma unroll
        for (int k = 1; k < 8; ++k) L += t >= sh.ptfirst[k] ? 1 : 0;
        if (t - sh.ptfirst[L] >= sh.pnch[L]) continue;
        const uint32_t kk = __ldcg(ma.ecnt + size_t(nxt) * MD_TCAP + t);
        const uint32_t* __restrict__ src = ma.eslot + (size_t(nxt) * MD_TCAP + t) * ESLOT;
        const unsigned long long at = sh.ebase[L] + sh.PE[mid_eidx(t)];
        if (at + kk <= a.ecap[L]) {
          uint32_t* __restrict__ dst = a.emit[L] + at;
          for (uint32_t w = lane; w < kk; w += 32u) dst[w] = __ldcg(src + w);
        }
      }
    };

    if (decision != kCseRunning) {
      // ---- leave: the frontier goes back to the flat layout (unless it never left it) -----------------------------
      if (!from_flat) move_words();
      if (!from_flat && decision != kCseOverflow) {
        const uint32_t T = sh.tfirst[8];
        for (uint32_t t = warp * G + blockIdx.x; t < T; t += MD_WARPS * G) {
          int l = 0;
#pragma unroll
          for (int k = 1; k < 8; ++k) l += t >= sh.tfirst[k] ? 1 : 0;
          const uint32_t q = t - sh.tfirst[l];
          if (q >= sh.nch[l]) continue;
          const uint32_t gbase = q * CH, gend = min(sh.n[l], gbase + CH), nz = sh.nz[l];
          uint32_t g[ITEMS], at[ITEMS];
#pragma unroll
          for (int j = 0; j < ITEMS; ++j) g[j] = gbase + 32u * j + lane;
          mid_locate<ITEMS>(sh, l, q, gend, lane, g, at);
#pragma unroll
          for (int j = 0; j < ITEMS; ++j)
            if (g[j] < gend) {
              const uint32_t to = flat_at(a.cap, nz, g[j]);
              const uint32_t* __restrict__ src = ma.arena + size_t(cur) * 3 * MD_PLACES + at[j];
              a.fs[cur][l][to] = __ldcg(src);
              a.fa[cur][l][to] = __ldcg(src + MD_PLACES);
              a.fb[cur][l][to] = __ldcg(src + 2 * MD_PLACES);
            }
        }
      }
      if (blockIdx.x == 0 && tid < 8) {
        S->cnt[cur][tid][0] = sh.nz[tid];
        S->cnt[cur][tid][1] = sh.n[tid] - sh.nz[tid];
        S->emitted[cur][tid] = sh.emitted[tid];
      }
      if (blockIdx.x == 0 && tid == 0) {
        S->status = decision;
        S->round = round;
        S->barriers = barrier_no;
      }
      if (blockIdx.x == 0 && tid == (MD_WARPS - 1) * 32) {      // the thread that made the plans counted
        S->visits += visits;
        if (peak > S->peak_frontier) S->peak_frontier = peak;
      }
      break;
    }

    // ================= the round: every warp takes chunks from load to store on its own ============================
    {
      const uint32_t T = sh.tfirst[8];
      const int eb = cur;                             // E-slot buffer of this round
      for (uint32_t t = warp * G + blockIdx.x; t < T; t += MD_WARPS * G) {
        int l = 0;
#pragma unroll
        for (int k = 1; k < 8; ++k) l += t >= sh.tfirst[k] ? 1 : 0;
        const uint32_t q = t - sh.tfirst[l];
        if (q >= sh.nch[l]) continue;                 // padding of the chunk numbering
        const int ln = (l + 1) & 7;
        const uint32_t nl = sh.n[l], nz = sh.nz[l];
        const uint32_t gbase = q * CH, gend = min(nl, gbase + CH);
        uint32_t g[ITEMS], at[ITEMS];
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) g[j] = gbase + 32u * j + lane;
        const uint32_t *ps, *pa, *pb;
        if (from_flat) {
#pragma unroll
          for (int j = 0; j < ITEMS; ++j) at[j] = flat_at(a.cap, nz, g[j]);
          ps = a.fs[cur][l]; pa = a.fa[cur][l]; pb = a.fb[cur][l];
        } else {
          mid_locate<ITEMS>(sh, l, q, gend, lane, g, at);
          ps = ma.arena + size_t(cur) * 3 * MD_PLACES; pa = ps + MD_PLACES; pb = pa + MD_PLACES;
        }
        // --- nodes and their three rank words
        uint32_t ns[ITEMS], na[ITEMS], nb[ITEMS];
        uint64_t wa[ITEMS], wb[ITEMS], wc[ITEMS];
        const uint64_t* __restrict__ R = a.ranks[l];
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
          ns[j] = na[j] = nb[j] = 0;
          if (g[j] < gend) {
            ns[j] = __ldcg(ps + at[j]);
            na[j] = __ldcg(pa + at[j]);
            nb[j] = __ldcg(pb + at[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
          wa[j] = wb[j] = wc[j] = 0;
          if (g[j] < gend) rank_words(R, ns[j], na[j], nb[j], wa[j], wb[j], wc[j]);
        }
        // --- compute; outputs straight into the chunk's slots of the next round
        uint32_t* __restrict__ gs = ma.arena + size_t(nxt) * 3 * MD_PLACES;
        uint32_t* __restrict__ ga = gs + MD_PLACES;
        uint32_t* __restrict__ gb = ga + MD_PLACES;
        const uint32_t zslot = sh.ndoff[ln] + q, oslot = sh.ndoff[ln] + sh.nch[l] + q;
        const uint32_t zbase = zslot * CH, obase = oslot * CH;
        uint32_t* __restrict__ ew = ma.eslot + (size_t(eb) * MD_TCAP + t) * ESLOT;
        const uint32_t one_base = a.C[ln];
        uint32_t cz = 0, co = 0, ce = 0;
#pragma unroll
        for (int j = 0; j < ITEMS; ++j) {
          CseStep r{false, false, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
          if (g[j] < gend) r = cse_step(a, l, one_base, ns[j], na[j], nb[j], wa[j], wb[j], wc[j]);
          warp_slot_store<EW>(r, nb[j], na[j] + nb[j], lt_mask, gs, ga, gb, zbase, obase, ew, cz, co, ce);
        }
        if (lane == 0) {
          ma.cnt[size_t(nxt) * MD_SLOTS + zslot] = uint8_t(cz);
          ma.cnt[size_t(nxt) * MD_SLOTS + oslot] = uint8_t(co);
          ma.ecnt[size_t(eb) * MD_TCAP + t] = uint16_t(ce);
        }
      }
    }
    MID_STAMP(2);
    if (!from_flat) move_words();
    MID_STAMP(3);
    // what the next round's scan needs to know about this one
    __syncthreads();
    if (tid < 8) {
      sh.sz[tid] = sh.nch[(tid + 7) & 7];
      sh.pnch[tid] = sh.nch[tid];
    }
    if (tid < 9) { sh.doff[tid] = sh.ndoff[tid]; sh.ptfirst[tid] = sh.tfirst[tid]; }
    if (tid == 0)       // threads that will hold slots (16 each) or chunks (8 each) of the next round, rounded up to warps
      sh.ex_valid = (max((sh.ndoff[8] + 15u) / 16u, (sh.tfirst[8] + 7u) / 8u) + 31u) & ~31u;
    MID_STAMP(4);
    const bool ok = grid_barrier(S, barrier_no++, round);
    MID_STAMP(5);
    ++round;
    from_flat = false;
    if (!ok) {
      if (blockIdx.x == 0 && tid == 0) { S->round = round; S->barriers = barrier_no; }
      break;
    }
  }
}

}  // namespace bce
